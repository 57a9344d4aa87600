"""GPU: end to end through the product boundary B2.  The same prompt is run through the drop-in pyfastllama.so of this repo
(llama_* C ABI over libggml_b200) via the Python Model class (fastllama_b200/model.py, mirror of the reference's fastllama.Model)
and compared with what the reference product library (reference bridge + reference ggml, CPU) produced on the same seeded model
file: tests/golden/model_e2e_toy.npz (oracle/gen_golden_model.py).

north_star bar: greedy token-id sequence identical; logits within a stated fp tolerance.  The tolerance here is ZERO: the logits after
the prompt and the decode steps carry the reference's bits (every fp32 operation in the reference's order, fl_exact.cuh; the prompt of
these tests stays below the 16 columns from which the tcgen05 GEMM -- reordering budget, not bit-identical -- takes over).
"""
import os

import numpy as np
import pytest

from fastllama_b200.build import lib_path
from fastllama_b200.ggjt import Q4_0, Q4_1, write_synthetic_numpy
from fastllama_b200.model import Model, QuietLogger
from oracle.pyoracle import Oracle

pytestmark = pytest.mark.gpu
DROPIN = os.environ.get("FASTLLAMA_TEST_DROPIN", lib_path("pyfastllama.so"))     # tests/mock/build/... for host-logic dry runs
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
PROMPT = "The quick brown fox jumps over the lazy dog. 0123456789"


def _run(lib, path, n_batch, n_gen=24):
    m = Model(path, num_threads=8, n_ctx=128, n_batch=n_batch, logger=QuietLogger(), library_path=lib)
    assert m.ingest(PROMPT)
    toks = []
    assert m.generate(lambda s: toks.append(s), num_tokens=n_gen, temp=0.0, top_k=1, top_p=1.0, repeat_penalty=1.0)
    logits = m.get_logits_array()
    m.close()
    return toks, logits


def toy_model(tmp_path, wtype):
    orc = Oracle()
    path = str(tmp_path / f"toy{wtype}.bin")
    write_synthetic_numpy(path, wtype, n_vocab=512, n_embd=256, n_mult=64, n_head=4, n_layer=3, seed=11, std=0.01,
                          quantize=lambda w, t: orc.quantize_q4(w, t))
    return path


@pytest.mark.parametrize("wtype", [Q4_0, Q4_1])
@pytest.mark.parametrize("n_batch", [1, 8])
def test_greedy_tokens_and_logits_match_reference(tmp_path, wtype, n_batch):
    path = toy_model(tmp_path, wtype)
    assert os.path.exists(DROPIN), "drop-in library not built"
    golden = np.load(os.path.join(GOLDEN, "model_e2e_toy.npz"))
    key = f"{'q4_0' if wtype == Q4_0 else 'q4_1'}_b{n_batch}"
    ref_toks, ref_logits = list(golden[key + "_tokens"]), golden[key + "_logits"]
    our_toks, our_logits = _run(DROPIN, path, n_batch)
    assert len(ref_toks) > 4
    assert our_toks == ref_toks, (our_toks, ref_toks)
    nd = int((our_logits.view(np.uint32) != ref_logits.view(np.uint32)).sum())
    assert nd == 0, (nd, our_logits.size, float(np.abs(our_logits - ref_logits).max()))      # the reference's bits, after prompt + decode steps
    assert int(our_logits.argmax()) == int(ref_logits.argmax())
