"""Synthetic GGJT-v1 model files (bench / test tooling; no real weights are available offline).

File layout (reference include/file_loader.hpp:94-250 reader, scripts/convert.py:903-928 writer):
  u32 magic 'ggjt', u32 version 1, 7 x i32 {n_vocab, n_embd, n_mult, n_head, n_layer, n_rot, ftype},
  n_vocab x {i32 len, bytes, f32 score}, then per tensor
  {i32 n_dims, i32 name_len, i32 type, i32 ne[n_dims] (ne0 = K first), name, pad to 32 B, data}.
Tensor names / shapes: reference lib/llama.cpp:223-245.  2-D tensors ~ N(0, std^2) quantised row by row with
quantize_row_q4_{0,1}_reference semantics; norms = 1.0 (f32).
"""
from __future__ import annotations

import struct
from typing import Callable, Iterator, Tuple

import numpy as np

GGJT_MAGIC = 0x67676A74
F32, Q4_0, Q4_1 = 0, 2, 3
FTYPE = {Q4_0: 2, Q4_1: 3}
BLOCK_BYTES = {Q4_0: 20, Q4_1: 24}

LLAMA_SIZES = {     # n_embd, n_head, n_layer (n_mult 256, n_vocab 32000); reference lib/llama.cpp:129-139
    "toy": (256, 4, 2), "7B": (4096, 32, 32), "13B": (5120, 40, 40), "30B": (6656, 52, 60), "65B": (8192, 64, 80),
}


def n_ff(n_embd: int, n_mult: int) -> int:
    return ((2 * (4 * n_embd) // 3 + n_mult - 1) // n_mult) * n_mult


def vocab_entries(n_vocab: int):
    """ids 0-2 specials, 3-258 the byte-fallback tokens (the tokenizer maps byte b to id b+3,
    reference include/tokenizer.hpp:130-133), the rest unique ASCII dummies with decreasing scores.
    Every string is ASCII so the Python stream callback can always decode it."""
    for i in range(n_vocab):
        if i == 0:
            tok = b"<unk>"
        elif i == 1:
            tok = b"<s>"
        elif i == 2:
            tok = b"</s>"
        elif i < 259:
            tok = b"<0x%02X>" % (i - 3)
        else:
            tok = b"~t%05d" % i
        yield tok, -float(i)


def tensor_plan(n_vocab, n_embd, n_mult, n_head, n_layer) -> Iterator[Tuple[str, Tuple[int, ...]]]:
    """(name, ne) with ne0 = K (input features) first."""
    ff = n_ff(n_embd, n_mult)
    yield "tok_embeddings.weight", (n_embd, n_vocab)
    yield "norm.weight", (n_embd,)
    yield "output.weight", (n_embd, n_vocab)
    for i in range(n_layer):
        yield f"layers.{i}.attention.wq.weight", (n_embd, n_embd)
        yield f"layers.{i}.attention.wk.weight", (n_embd, n_embd)
        yield f"layers.{i}.attention.wv.weight", (n_embd, n_embd)
        yield f"layers.{i}.attention.wo.weight", (n_embd, n_embd)
        yield f"layers.{i}.attention_norm.weight", (n_embd,)
        yield f"layers.{i}.feed_forward.w1.weight", (n_embd, ff)
        yield f"layers.{i}.feed_forward.w2.weight", (ff, n_embd)
        yield f"layers.{i}.feed_forward.w3.weight", (n_embd, ff)
        yield f"layers.{i}.ffn_norm.weight", (n_embd,)


def write_ggjt(path: str, wtype: int, n_vocab: int, n_embd: int, n_mult: int, n_head: int, n_layer: int,
               matrix_bytes: Callable[[str, int, int, int], bytes]) -> int:
    """matrix_bytes(name, K, M, wtype) -> the M*K/32*block_bytes quantised bytes of that tensor."""
    with open(path, "wb") as f:
        f.write(struct.pack("<II", GGJT_MAGIC, 1))
        f.write(struct.pack("<7i", n_vocab, n_embd, n_mult, n_head, n_layer, n_embd // n_head, FTYPE[wtype]))
        for tok, score in vocab_entries(n_vocab):
            f.write(struct.pack("<i", len(tok)) + tok + struct.pack("<f", score))
        for name, ne in tensor_plan(n_vocab, n_embd, n_mult, n_head, n_layer):
            nm = name.encode()
            t = F32 if len(ne) == 1 else wtype
            f.write(struct.pack("<iii", len(ne), len(nm), t))
            f.write(struct.pack(f"<{len(ne)}i", *ne))
            f.write(nm)
            f.write(b"\0" * (-f.tell() & 31))
            if len(ne) == 1:
                f.write(np.ones(ne[0], dtype=np.float32).tobytes())
            else:
                data = matrix_bytes(name, ne[0], ne[1], wtype)
                assert len(data) == ne[1] * (ne[0] // 32) * BLOCK_BYTES[wtype], name
                f.write(data)
        return f.tell()


def write_synthetic_numpy(path, wtype=Q4_0, n_vocab=512, n_embd=256, n_mult=64, n_head=4, n_layer=2, seed=0, std=0.02,
                          quantize=None) -> int:
    """CPU generator for toy models (tests).  `quantize(w_f32[M,K], wtype) -> uint8` must follow the
    reference's quantize_row_q4_*_reference; the tests pass the oracle's."""
    rng = np.random.default_rng(seed)

    def gen(name, k, m, t):
        scale = 1.0 if name.startswith("tok_embeddings") else std * (4.0 if n_embd < 1024 else 1.0)
        w = (rng.standard_normal((m, k)) * scale).astype(np.float32)
        return np.ascontiguousarray(quantize(w, t)).tobytes()

    return write_ggjt(path, wtype, n_vocab, n_embd, n_mult, n_head, n_layer, gen)


def write_synthetic_gpu(path, size="7B", wtype=Q4_0, seed=0, std=0.02, n_vocab=32000, n_mult=256, fl=None, n_layer=None) -> int:
    """GPU generator for full-size models: a counter-based Gaussian filled on the device and quantised
    by the library's bit-exact quantize_row_q4_*_reference kernel, streamed to the file per tensor."""
    import ctypes as C

    from .cuda_abi import FlCuda

    fl = fl or FlCuda()
    n_embd, n_head, layers = LLAMA_SIZES[size]
    n_layer = n_layer or layers
    ff = n_ff(n_embd, n_mult)
    max_el = max(n_vocab, ff) * max(n_embd, ff) if False else max(n_vocab * n_embd, ff * n_embd)
    d_f32 = fl.alloc(max_el * 4)
    d_q = fl.alloc(max_el // 32 * BLOCK_BYTES[wtype])
    counter = [0]

    def gen(name, k, m, t):
        n = k * m
        fl.check(fl.lib.fl_dev_fill_normal(d_f32, n, C.c_uint64(seed * 1000003 + counter[0]), C.c_float(std)))
        counter[0] += 1
        fl.check(fl.lib.fl_dev_quantize_q4(t, d_f32, d_q, k, m))
        return fl.to_host(d_q, (n // 32 * BLOCK_BYTES[t],), np.uint8).tobytes()

    try:
        return write_ggjt(path, wtype, n_vocab, n_embd, n_mult, n_head, n_layer, gen)
    finally:
        fl.free(d_f32)
        fl.free(d_q)


GGLA_MAGIC = 0x67676C61


def write_lora(path: str, factors: dict, r: int, alpha: int) -> int:
    """LoRA adapter file ('ggla' v1): u8 cached (0: factors), u32 r, u32 alpha, then per adapted weight W the f32 tensors
    "<W>.loraA" (ne = r, K; already scaled by alpha / r) and "<W>.loraB" (ne = r, M), records laid out as in write_ggjt.
    `factors` maps W's name to (A[K, r], B[M, r]) float32 arrays."""
    with open(path, "wb") as f:
        f.write(struct.pack("<IIBII", GGLA_MAGIC, 1, 0, r, alpha))
        for name, mats in factors.items():
            for tag, m in zip("AB", mats):
                m = np.ascontiguousarray(m, dtype=np.float32)
                nm = f"{name}.lora{tag}".encode()
                f.write(struct.pack("<iiiii", 2, len(nm), F32, m.shape[1], m.shape[0]))
                f.write(nm)
                f.write(b"\0" * (-f.tell() & 31))
                f.write(m.tobytes())
        return f.tell()
