"""CPU: Model.save_state / load_state of pyfastllama.so on top of libggml_b200, with the KV cache living in "device" memory
(the CPU stand-in of the device layer, tests/mock).  The library touches kv_self.{k,v}->data on the host right after a
ggml_nbytes(k) call, which is the hook libggml_b200 uses to copy the cache back and to schedule its re-upload.  Checks: a
state saved by us resumes identically in us; it carries what the reference library writes at the same point (its state file
and tokens are stored in tests/golden/model_state_toy.npz, oracle/gen_golden_model.py); and a state saved by the reference
resumes in us with the reference's tokens."""
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
mode, lib, path, state, out = sys.argv[2], sys.argv[3], sys.argv[4], sys.argv[5], sys.argv[6]
if "mock" in lib:
    C.CDLL(os.path.join(os.path.dirname(lib), "libfl_cuda.so"), mode=C.RTLD_GLOBAL)
m = Model(path, num_threads=2, n_ctx=64, n_batch=4, logger=QuietLogger(), library_path=lib)
toks = []
gen = lambda n: m.generate(lambda s: toks.append(s), num_tokens=n, temp=0.0, top_k=1, top_p=1.0, repeat_penalty=1.0)
if mode == "save":                       # prompt, 5 tokens, save, 8 more tokens, then load and redo the 8
    m.ingest("State files must survive a round trip.")
    gen(5)
    assert m.save_state(state)
    gen(8)
    first = list(toks[5:])
    assert m.load_state(state)
    del toks[:]
    gen(8)
    np.savez(out, first=np.array(first), again=np.array(toks), logits=m.get_logits_array())
else:                                    # resume from a state file written by somebody else
    assert m.load_state(state)
    gen(8)
    np.savez(out, again=np.array(toks), logits=m.get_logits_array())
m.close()
'''


def _run(tmp_path, mode, lib, model, state, tag):
    script = tmp_path / "worker.py"
    script.write_text(WORKER)
    out = str(tmp_path / f"{tag}.npz")
    p = subprocess.run([sys.executable, str(script), ROOT, mode, lib, model, state, out], capture_output=True, text=True, timeout=300,
                       env=dict(os.environ, OMP_NUM_THREADS="2"))
    assert p.returncode == 0, p.stderr[-3000:]
    return np.load(out)


def state_model(tmp_path):
    from fastllama_b200.ggjt import Q4_0, write_synthetic_numpy
    from oracle.pyoracle import Oracle

    orc = Oracle()
    model = str(tmp_path / "toy.bin")
    write_synthetic_numpy(model, Q4_0, n_vocab=512, n_embd=256, n_mult=256, n_head=4, n_layer=3, seed=7, std=0.01, quantize=lambda w, t: orc.quantize_q4(w, t))
    return model


def parse_state(raw: bytes) -> dict:
    """The fields of a state file: i32 n_past, u64 + text of the RNG, u64 mem_per_token, u64 + i32[] pending tokens, u64 + i32[]
    last tokens, u64 + f32[] logits, u64 + i32[] system prompt, i32 KV type, then K and V (f32, equal halves)."""
    out, off = {}, 0

    def take(dtype, n):
        nonlocal off
        a = np.frombuffer(raw, dtype=dtype, count=n, offset=off)
        off += a.nbytes
        return a

    out["n_past"] = int(take(np.int32, 1)[0])
    out["rng"] = take(np.uint8, int(take(np.uint64, 1)[0])).tobytes()
    out["mem_per_token"] = int(take(np.uint64, 1)[0])
    for name, dt in (("pending", np.int32), ("last_tokens", np.int32), ("logits", np.float32), ("system_prompt", np.int32)):
        out[name] = take(dt, int(take(np.uint64, 1)[0]))
    out["kv_type"] = int(take(np.int32, 1)[0])
    kv = np.frombuffer(raw, dtype=np.float32, offset=off)
    out["k"], out["v"] = kv[: kv.size // 2], kv[kv.size // 2:]
    return out


def check_state_interop(tmp_path, ours_lib):
    model = state_model(tmp_path)
    golden = np.load(os.path.join(ROOT, "tests", "golden", "model_state_toy.npz"))
    ref_state = tmp_path / "ref.state"
    ref_state.write_bytes(golden["state"].tobytes())

    ours = _run(tmp_path, "save", ours_lib, model, str(tmp_path / "ours.state"), "ours")
    assert list(ours["first"]) == list(ours["again"])                       # our own state resumes identically in us
    assert list(golden["first"]) == list(golden["again"])
    assert list(ours["first"]) == list(golden["first"])
    assert os.path.getsize(tmp_path / "ours.state") == ref_state.stat().st_size

    # what the reference would resume from: every field of our state file is the reference's, the floats within the logits' budget
    # (mem_per_token is informational and differs: the reference's compute arena also holds its CPU work buffer)
    a, b = parse_state((tmp_path / "ours.state").read_bytes()), parse_state(ref_state.read_bytes())
    for key in ("n_past", "rng", "pending", "last_tokens", "system_prompt", "kv_type"):
        assert np.array_equal(a[key], b[key]), key
    for key in ("logits", "k", "v"):
        assert a[key].shape == b[key].shape and np.abs(a[key] - b[key]).max() <= 2e-2 * np.abs(b[key]).max(), key

    ours_from_ref = _run(tmp_path, "load", ours_lib, model, str(ref_state), "ours_from_ref")
    assert list(ours_from_ref["again"]) == list(golden["first"])            # a cache loaded on the host reaches the device
    tol = 2e-2 * np.abs(golden["logits"]).max()
    assert np.abs(ours_from_ref["logits"] - golden["logits"]).max() <= tol


@pytest.mark.skipif(not os.path.exists(os.path.join(MOCK, "pyfastllama.so")), reason="tests/mock not built (needs the drop-in library)")
def test_state_round_trip_and_interop_with_reference(tmp_path):
    check_state_interop(tmp_path, os.path.join(MOCK, "pyfastllama.so"))
