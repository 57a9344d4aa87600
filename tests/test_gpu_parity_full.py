"""GPU: whole-model parity at the GRADED size -- the synthetic LLaMA-7B q4_0 file of bench.py (N(0, 0.02^2), seed 0) and a 4-layer
LLaMA-13B q4_1 file -- through the reference-facing API (Model.ingest / Model.generate on the drop-in pyfastllama.so) against what the
reference itself (its CPU library) produced on the same files: same prompt, greedy.  The reference's tokens, a SHA-256 of every step's
logit bits and a fixed sample of its logits are stored in tests/golden/model_parity_*.npz (oracle/gen_golden_model.py --full).

What is asserted (north_star: "logits match the reference CPU path on the same prompt within a stated fp tolerance, greedy token-id
sequence bit-exact"): the greedy token sequences are IDENTICAL and the logits of every step (32000 floats) carry the reference's BITS.
Tolerance zero: every fp32 operation of the path follows the reference's order (fastllama_b200/csrc/fl_exact.cuh) -- anything less
exact ends up at the per-cent level after a few layers, because every activation vector is re-quantised to q8_0 before every matmul
(DESIGN.md section 5; the round-1/early round-2 kernels, which only reordered the fp32 sums, measured 7.5e-2 of max|logit| at 32 layers
and lost the token sequence at step 10).  A third case ingests a LONG prompt (>= 16 tokens: the tcgen05 GEMM, whose block terms are added
in another order) and asserts the stated budget for that path, and bit equality again with FASTLLAMA_B200_INGEST=exact."""
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

pytestmark = pytest.mark.gpu

N_TOKENS = 24


LONG_PROMPT = ("The quick brown fox jumps over the lazy dog, then turns around and does it again while the farmer counts his sheep "
               "and the sun goes down behind the hills.")      # well over 16 tokens: a multi-token eval on the tensor-core path
# The stored reference covers a fixed sample of 2048 logits plus the top 64 of every step (all 32000 per step would exceed the 1 MB a
# fixture may take), so this tolerance is checked on that sample against the step's true max|reference logit|; bit identity is checked
# on all logits through the per-step SHA-256.
LONG_TOL = 0.15           # of max|reference logit|: what a re-ordered fp32 sum in the prompt's matmuls costs after a few layers (see above)


def _ours(path, n, prompt=None, n_batch=1):
    import bench

    be = bench.Backend(0)
    m = be.model(path, n_batch=n_batch)
    assert m.ingest(prompt or bench.PROMPT)
    toks, logits = [], []
    for _ in range(n):
        got = []
        m.generate(lambda s: got.append(s), num_tokens=1, **bench.GREEDY)
        if not got:
            break
        toks.append("".join(got))
        logits.append(m.get_logits_array())
    mode = int(be.ggml.ggml_b200_decode_mode())
    m.close()
    return toks, np.stack(logits), mode


def _golden(name):
    return np.load(os.path.join(ROOT, "tests", "golden", name))


def _compare(golden, our_tokens, our_logits):
    """Tokens compared, first divergence, per-step bit identity (SHA-256 of the logits) and max|ours - reference| / max|reference| over
    the stored sample, for the steps where both arms evaluated the same token sequence."""
    from oracle.gen_golden_model import logits_digest

    ref_tokens = list(golden["tokens"])
    n = min(len(ref_tokens), len(our_tokens))
    first = next((i for i in range(n) if ref_tokens[i] != our_tokens[i]), None)
    upto = n if first is None else first + 1
    idx = golden["index"][:upto]
    rel = np.abs(np.take_along_axis(our_logits[:upto], idx, axis=1).astype(np.float64) - golden["sample"][:upto]).max(axis=1) / golden["absmax"][:upto]
    same_bits = bool(np.array_equal(logits_digest(our_logits[:upto]), golden["digest"][:upto]))
    return {"tokens_compared": n, "greedy_ids_equal": first is None and n > 0, "first_divergence": first, "logits_bit_identical": same_bits,
            "logits_maxabs_over_range": float(rel.max()) if upto else None}


def _check(golden, our_tokens, our_logits):
    par = _compare(golden, our_tokens, our_logits)
    print("parity:", par)
    assert par["tokens_compared"] >= N_TOKENS // 2
    assert par["greedy_ids_equal"], par
    assert par["logits_bit_identical"] and par["logits_maxabs_over_range"] == 0.0, par
    return par


def model_13b_4l():
    import bench
    from fastllama_b200.ggjt import write_synthetic_gpu

    path = os.path.join(bench.bench_dir(), "fastllama_b200_synth_13B_q4_1_4layers_seed0.bin")
    if not os.path.exists(path):
        write_synthetic_gpu(path + ".tmp", size="13B", wtype=3, seed=0, std=0.02, n_layer=4)
        os.replace(path + ".tmp", path)
    return path


def test_7b_q4_0_tokens_and_logits_against_the_reference(tmp_path):
    import bench

    path = bench.ensure_model("7B", "q4_0")
    our_tokens, our_logits, mode = _ours(path, N_TOKENS)
    assert mode == 2, "decode steps did not run as the persistent token kernel"
    _check(_golden("model_parity_7b_q4_0.npz"), our_tokens, our_logits)


def test_13b_q4_1_four_layers_against_the_reference(tmp_path):
    path = model_13b_4l()
    our_tokens, our_logits, mode = _ours(path, N_TOKENS)
    assert mode == 2
    _check(_golden("model_parity_13b_q4_1_4l.npz"), our_tokens, our_logits)
    # a long prompt, ingested 128 tokens at a time
    # (the reference's own bits depend on n_batch: the value mix of a multi-token eval is a dot product over ALL its positions, masked ones included)
    long_ref = _golden("model_parity_13b_q4_1_4l_long.npz")
    os.environ["FASTLLAMA_B200_INGEST"] = "exact"               # the reference-order kernel for every eval: the reference's bits again
    try:
        our_tokens, our_logits, _ = _ours(path, N_TOKENS, LONG_PROMPT, n_batch=128)
    finally:
        del os.environ["FASTLLAMA_B200_INGEST"]
    _check(long_ref, our_tokens, our_logits)
    our_tokens, our_logits, _ = _ours(path, N_TOKENS, LONG_PROMPT, n_batch=128)     # default: tcgen05 GEMM for the prompt, reordering budget
    par = _compare(long_ref, our_tokens, our_logits)
    print("parity (tcgen05 prompt ingest):", par)
    assert par["logits_maxabs_over_range"] <= LONG_TOL, par
    os.remove(path)
