"""Model.attach_lora / detach_lora end to end: a toy q4_0 model and a rank-4 adapter on six of its matrices, with the model file
read into memory and mapped.  Greedy tokens and logits before, with and after the adapter are compared with what the reference
library produced for the same sequence (tests/golden/model_lora_toy.npz, oracle/gen_golden_model.py), on the CPU stand-in of the
device layer and on the B200."""
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
from tests.mockbuild import ensure_mock  # noqa: E402

MOCK = ensure_mock()

WORKER = r'''
import ctypes as C, os, sys, numpy as np
sys.path.insert(0, sys.argv[1])
from fastllama_b200.model import Model, QuietLogger
lib, path, lora, out = sys.argv[2], sys.argv[3], sys.argv[4], sys.argv[5]
if "mock" in lib:
    C.CDLL(os.path.join(os.path.dirname(lib), "libfl_cuda.so"), mode=C.RTLD_GLOBAL)
greedy = dict(temp=0.0, top_k=1, top_p=1.0, repeat_penalty=1.0)
res = {}
for mmap in (0, 1):
    m = Model(path, num_threads=2, n_ctx=64, n_batch=4, use_mmap=bool(mmap), logger=QuietLogger(), library_path=lib)
    for phase in ("base", "lora", "after"):
        if phase == "lora":
            assert m.attach_lora(lora)
            assert not m.attach_lora(lora)            # one adapter at a time
        if phase == "after":
            assert m.detach_lora()
            assert not m.detach_lora()
        assert m.reset()
        assert m.ingest("Adapters change the weights.")
        toks = []
        m.generate(lambda s: toks.append(s), num_tokens=6, **greedy)
        res[f"{phase}{mmap}_tokens"] = np.array(toks)
        res[f"{phase}{mmap}_logits"] = m.get_logits_array()
    m.close()
np.savez(out, **res)
'''


def lora_files(tmp_path):
    from fastllama_b200.ggjt import Q4_0, n_ff, write_lora, write_synthetic_numpy
    from oracle.pyoracle import Oracle

    orc = Oracle()
    model = str(tmp_path / "toy.bin")
    n_embd, n_mult = 256, 64
    write_synthetic_numpy(model, Q4_0, n_vocab=512, n_embd=n_embd, n_mult=n_mult, n_head=4, n_layer=3, seed=11, std=0.01,
                          quantize=lambda w, t: orc.quantize_q4(w, t))
    rng = np.random.default_rng(5)
    r, ff = 4, n_ff(n_embd, n_mult)
    shapes = {"attention.wq": (n_embd, n_embd), "attention.wv": (n_embd, n_embd), "feed_forward.w2": (ff, n_embd)}
    factors = {f"layers.{il}.{w}.weight": ((rng.standard_normal((k, r)) * 0.3).astype(np.float32), (rng.standard_normal((m, r)) * 0.3).astype(np.float32))
               for il in (0, 2) for w, (k, m) in shapes.items()}
    lora = str(tmp_path / "adapter.bin")
    write_lora(lora, factors, r=r, alpha=r)
    return model, lora


def run(tmp_path, lib, tag):
    model, lora = lora_files(tmp_path)
    script = tmp_path / "lora_worker.py"
    script.write_text(WORKER)
    out = str(tmp_path / f"{tag}.npz")
    p = subprocess.run([sys.executable, str(script), ROOT, lib, model, lora, out], capture_output=True, text=True, timeout=600,
                       env=dict(os.environ, OMP_NUM_THREADS="2"))
    assert p.returncode == 0, p.stderr[-3000:]
    return np.load(out)


def _check(tmp_path, lib):
    ref = np.load(os.path.join(ROOT, "tests", "golden", "model_lora_toy.npz"))
    assert list(ref["base0_tokens"]) != list(ref["lora0_tokens"]), "the adapter must change the toy model's output"
    ours = run(tmp_path, lib, "ours")
    for key in ref.files:
        if key.endswith("_tokens"):
            assert list(ours[key]) == list(ref[key]), key
        else:
            assert np.abs(ours[key] - ref[key]).max() <= 2e-2 * np.abs(ref[key]).max(), key


@pytest.mark.skipif(not os.path.exists(os.path.join(MOCK, "pyfastllama.so")), reason="tests/mock not built (needs the drop-in library)")
def test_lora_attach_detach_matches_reference_on_cpu_mock(tmp_path):
    _check(tmp_path, os.path.join(MOCK, "pyfastllama.so"))


@pytest.mark.gpu
def test_lora_attach_detach_matches_reference_on_gpu(tmp_path):
    from fastllama_b200.build import lib_path

    _check(tmp_path, lib_path("pyfastllama.so"))
