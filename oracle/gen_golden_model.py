"""Generate tests/golden/model_*.npz: what the REFERENCE product library (oracle/_ref/pyfastllama_ref.so, CPU) computes through its
C ABI on the synthetic model files of the whole-model tests, so that those tests compare against it wherever only the committed
files exist.

    python -m oracle.gen_golden_model          # toy models (CPU only): e2e, reload, state files, LoRA, perplexity
    python -m oracle.gen_golden_model --full   # also the 7B q4_0 / 13B q4_1 parity files (their model files are written on a GPU)

Every model file is rebuilt by the tests from a seed, so only the reference's outputs are stored.  Full-size logits are too large
to keep: a fixed sample of them plus a SHA-256 of every step's complete logit bits is stored instead.
"""
import hashlib
import os
import pathlib
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

OUT = os.path.join(ROOT, "tests", "golden")
N_SAMPLE = 2048          # logits kept per step of a full-size run (plus the top 64 of the step)


def logits_digest(logits: np.ndarray) -> np.ndarray:
    """[steps, n_vocab] f32 -> one SHA-256 (as 32 uint8) per step over the logit bits."""
    logits = np.ascontiguousarray(logits, dtype=np.float32)
    return np.stack([np.frombuffer(hashlib.sha256(row.tobytes()).digest(), dtype=np.uint8) for row in logits])


def logits_sample_index(ref_logits: np.ndarray, seed: int = 0) -> np.ndarray:
    """Per step: a fixed random sample of N_SAMPLE logit indices followed by the indices of the step's 64 largest reference logits."""
    fixed = np.random.default_rng(seed).choice(ref_logits.shape[1], N_SAMPLE, replace=False)
    return np.stack([np.concatenate([fixed, np.argsort(row)[-64:]]) for row in ref_logits]).astype(np.int32)


def save(name: str, **arrays):
    path = os.path.join(OUT, name)
    np.savez_compressed(path, **arrays)
    print("wrote", path, os.path.getsize(path), "bytes")


def toy(ref_so: str):
    from tests import test_gpu_e2e, test_lora_e2e, test_perplexity, test_reload, test_state_mock
    from fastllama_b200.ggjt import Q4_0, Q4_1

    with tempfile.TemporaryDirectory() as td:
        tmp = pathlib.Path(td)
        out = {}
        for wname, wtype in (("q4_0", Q4_0), ("q4_1", Q4_1)):
            path = test_gpu_e2e.toy_model(tmp, wtype)
            for n_batch in (1, 8):
                toks, logits = test_gpu_e2e._run(ref_so, path, n_batch)
                out[f"{wname}_b{n_batch}_tokens"] = np.array(toks)
                out[f"{wname}_b{n_batch}_logits"] = logits
        save("model_e2e_toy.npz", **out)

        a, b = test_reload._models(tmp)
        ref = test_reload._run(tmp, ref_so, a, b, "ref")
        save("model_reload_toy.npz", **{k: ref[k] for k in ref.files})

        model = test_state_mock.state_model(tmp)
        ref = test_state_mock._run(tmp, "save", ref_so, model, str(tmp / "ref.state"), "ref")
        save("model_state_toy.npz", first=ref["first"], again=ref["again"], logits=ref["logits"],
             state=np.frombuffer((tmp / "ref.state").read_bytes(), dtype=np.uint8))

        ref = test_lora_e2e.run(tmp, ref_so, "ref")
        save("model_lora_toy.npz", **{k: ref[k] for k in ref.files})

        save("model_perplexity_toy.npz", ppl=np.float64(test_perplexity.ppl(tmp, ref_so, test_perplexity.toy_model(tmp))))


def full():
    import bench
    from tests import test_gpu_parity_full as P

    with tempfile.TemporaryDirectory() as td:
        tmp = pathlib.Path(td)
        runs = [("model_parity_7b_q4_0.npz", bench.ensure_model("7B", "q4_0"), None, 1),
                ("model_parity_13b_q4_1_4l.npz", P.model_13b_4l(), None, 1),
                ("model_parity_13b_q4_1_4l_long.npz", P.model_13b_4l(), P.LONG_PROMPT, 128)]
        for name, path, prompt, n_batch in runs:
            lp = str(tmp / "ref_logits.npy")
            r = bench.run_ref_worker({"path": path, "threads": min(32, os.cpu_count() or 1), "prompt": prompt or bench.PROMPT,
                                      "n_parity": P.N_TOKENS, "logits_out": lp, "n_batch": n_batch})
            logits = np.load(lp)
            idx = logits_sample_index(logits)
            save(name, tokens=np.array(r["parity_tokens"]), digest=logits_digest(logits), index=idx,
                 sample=np.take_along_axis(logits, idx, axis=1), absmax=np.abs(logits).max(axis=1))


def main():
    from oracle.pyoracle import REF_PYFASTLLAMA_SO, build_oracle

    build_oracle()
    if not os.path.exists(REF_PYFASTLLAMA_SO):
        raise SystemExit("oracle/_ref/pyfastllama_ref.so is missing: build() compiles it where the reference's sources are present")
    os.makedirs(OUT, exist_ok=True)
    toy(REF_PYFASTLLAMA_SO)
    if "--full" in sys.argv:
        full()


if __name__ == "__main__":
    main()
