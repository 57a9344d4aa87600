"""Model.perplexity (n_batch > 1 evals that return the logits of every token): what the reference library computed
(tests/golden/model_perplexity_toy.npz, oracle/gen_golden_model.py) vs our stack -- on the CPU stand-in of the device layer (host logic; its matmul is
bit-identical to the reference's,
so only the non-matmul ops differ) and on the B200 (tensor-core ingest kernel + generic executor)."""
import os
import subprocess
import sys

import pytest

from tests.mockbuild import ensure_mock

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

WORKER = r'''
import ctypes as C, os, sys
sys.path.insert(0, sys.argv[1])
from fastllama_b200.model import Model, QuietLogger
lib, path = sys.argv[2], sys.argv[3]
if "mock" in lib:
    C.CDLL(os.path.join(os.path.dirname(lib), "libfl_cuda.so"), mode=C.RTLD_GLOBAL)
m = Model(path, num_threads=2, n_ctx=64, n_batch=8, logger=QuietLogger(), library_path=lib)
print("PPL", repr(m.perplexity("The quick brown fox jumps over the lazy dog. " * 4)))
m.close()
'''


def ppl(tmp_path, lib, model):
    script = tmp_path / "ppl_worker.py"
    script.write_text(WORKER)
    p = subprocess.run([sys.executable, str(script), ROOT, lib, model], capture_output=True, text=True, timeout=300, env=dict(os.environ, OMP_NUM_THREADS="2"))
    assert p.returncode == 0, p.stderr[-3000:]
    return float([ln for ln in p.stdout.splitlines() if ln.startswith("PPL ")][-1].split()[1])


def toy_model(tmp_path):
    from fastllama_b200.ggjt import Q4_0, write_synthetic_numpy
    from oracle.pyoracle import Oracle

    orc = Oracle()
    path = str(tmp_path / "toy.bin")
    write_synthetic_numpy(path, Q4_0, n_vocab=512, n_embd=256, n_mult=256, n_head=4, n_layer=3, seed=11, std=0.02, quantize=lambda w, t: orc.quantize_q4(w, t))
    return path


def reference_ppl():
    import numpy as np

    return float(np.load(os.path.join(ROOT, "tests", "golden", "model_perplexity_toy.npz"))["ppl"])


def test_perplexity_host_stack_matches_reference(tmp_path):
    ours = os.path.join(ensure_mock(), "pyfastllama.so")
    if not os.path.exists(ours):
        pytest.skip("needs tests/mock")
    model = toy_model(tmp_path)
    a, b = reference_ppl(), ppl(tmp_path, ours, model)
    # matmuls are bit-identical here; soft-max / rope / attention of the stand-in differ in the last ulps and a few fp16 table
    # flips move the mean log-likelihood by ~5e-4 (observed)
    assert a > 1.0 and abs(a - b) <= 2e-3 * a, (a, b)


@pytest.mark.gpu
def test_perplexity_on_b200_matches_reference(tmp_path):
    from fastllama_b200.build import lib_path

    model = toy_model(tmp_path)
    a, b = reference_ppl(), ppl(tmp_path, lib_path("pyfastllama.so"), model)
    assert a > 1.0 and abs(a - b) <= 1e-2 * a, (a, b)          # same policy as the logits: 5e-4 observed on the CPU stand-in
