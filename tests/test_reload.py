"""Model lifetime on one process: load model A, decode, close it, load model B -- B must never see A's weights.

External ("mmap'ed") weight tensors are mirrored on the device keyed by HOST ADDRESS, and a second mapping can land on the
addresses of the first (round-1 advisor finding).  Two defences, both exercised here on the CPU stand-in of the device layer and on
the B200: Model.close() releases every device resource (ggml_b200_release_all), and a new no_alloc context (= a model load with
mmap'ed tensors) drops all external mirrors of earlier mappings.  The check is against the reference library on model B."""
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
lib, path_a, path_b, out, use_close = sys.argv[2], sys.argv[3], sys.argv[4], sys.argv[5], sys.argv[6] == "1"
if "mock" in lib:
    C.CDLL(os.path.join(os.path.dirname(lib), "libfl_cuda.so"), mode=C.RTLD_GLOBAL)
greedy = dict(temp=0.0, top_k=1, top_p=1.0, repeat_penalty=1.0)
res = {}
for tag, path in (("a", path_a), ("b", path_b), ("a2", path_a)):
    if not path:
        continue
    m = Model(path, num_threads=2, n_ctx=64, n_batch=4, use_mmap=True, logger=QuietLogger(), library_path=lib)
    m.ingest("Two models, one process.")
    toks = []
    m.generate(lambda s: toks.append(s), num_tokens=6, **greedy)
    res[tag + "_tokens"] = np.array(toks)
    res[tag + "_logits"] = m.get_logits_array()
    if use_close:
        m.close()
    else:
        m.lib.llama_free_context(m.ctx)      # what a C user of the bridge does: no backend hook at all
        m.ctx = None
np.savez(out, **res)
'''


def _run(tmp_path, lib, a, b, tag, use_close=True):
    script = tmp_path / "worker.py"
    script.write_text(WORKER)
    out = str(tmp_path / f"{tag}.npz")
    p = subprocess.run([sys.executable, str(script), ROOT, lib, a, b, out, "1" if use_close else "0"], capture_output=True, text=True, timeout=600,
                       env=dict(os.environ, OMP_NUM_THREADS="2"))
    assert p.returncode == 0, p.stderr[-3000:]
    return np.load(out)


def _models(tmp_path):
    from fastllama_b200.ggjt import Q4_0, write_synthetic_numpy
    from oracle.pyoracle import Oracle

    orc = Oracle()
    paths = []
    for seed in (11, 12):                     # same shapes, different weights: the mappings have the same size
        p = str(tmp_path / f"toy{seed}.bin")
        write_synthetic_numpy(p, Q4_0, n_vocab=512, n_embd=256, n_mult=256, n_head=4, n_layer=3, seed=seed, std=0.01, quantize=lambda w, t: orc.quantize_q4(w, t))
        paths.append(p)
    return paths


def _check(tmp_path, lib):
    a, b = _models(tmp_path)
    ref = np.load(os.path.join(ROOT, "tests", "golden", "model_reload_toy.npz"))
    assert list(ref["a_tokens"]) != list(ref["b_tokens"]), "the two toy models must behave differently"
    for use_close in (True, False):
        ours = _run(tmp_path, lib, a, b, f"ours{int(use_close)}", use_close)
        for tag in ("a", "b", "a2"):
            assert list(ours[f"{tag}_tokens"]) == list(ref[f"{tag}_tokens"]), (tag, use_close)
            assert np.abs(ours[f"{tag}_logits"] - ref[f"{tag}_logits"]).max() <= 2e-2 * np.abs(ref[f"{tag}_logits"]).max(), (tag, use_close)


@pytest.mark.skipif(not os.path.exists(os.path.join(MOCK, "pyfastllama.so")), reason="tests/mock not built (needs the drop-in library)")
def test_second_model_does_not_see_the_first_models_weights_on_cpu_mock(tmp_path):
    _check(tmp_path, os.path.join(MOCK, "pyfastllama.so"))


@pytest.mark.gpu
def test_second_model_does_not_see_the_first_models_weights_on_gpu(tmp_path):
    from fastllama_b200.build import lib_path

    _check(tmp_path, lib_path("pyfastllama.so"))
