#!/usr/bin/env python
"""bench.py -- tokens/sec of LLaMA-7B q4_0 greedy decode (n_batch = 1) on B200, BASELINE.json's metric.

    python bench.py --gpus N --steps K --warmup W            # our arm
    python bench.py --impl reference --gpus N --steps K ...   # the reference's CPU path (rank 0 only)
    python bench.py --mode ingest                             # BASELINE configs[2]: prompt ingest, n_batch = 128 (tensor-core GEMM)
    python bench.py --size 13B --wtype q4_1                   # BASELINE configs[3]

A "step" is one decoded token = one pass of the hot path (7*32+1 quantised matvecs, 4 129 423 360 algorithmic weight bytes) over a
synthetic random-weight 7B q4_0 model (N(0, 0.02^2), seed 0, GGJT file written once to $FASTLLAMA_BENCH_DIR or /tmp by a child
process).  Keys of the JSON line:
  value      tokens/s with everything resident in HBM: K / (CUDA-event time around the K timed evals' kernels on the library stream),
             whole job over all ranks (max over ranks of the time)
  e2e        tokens/s through the reference-facing API -- fastllama_b200.Model.generate() on the drop-in pyfastllama.so (the
             llama_* C ABI over libggml_b200): wall clock around the call, which per step copies the token id + position host->device
             (pinned) and the logits + embeddings row device->host (pinned staging)
  roofline   dominant kernel = k_decode_token, the persistent kernel that runs the whole decode step (one launch per token, reads every
             quantised weight once): algorithmic bytes per launch / mean launch duration (CUDA events on the launching stream),
             against MEASURED_PEAKS.json's hbm_gbs
  cpu_baseline  the reference itself (oracle/_ref/pyfastllama_ref.so, built from the reference's sources in place) on the host cores:
             thread sweep, best setting reported, bounded sample; runs in child processes that never load this repository's libraries
  parity     same prompt, greedy: the reference's token sequence and per-step logits against ours (7B q4_0, N = 1); under torchrun the
             ranks' logits are compared with each other and the tokens with the N = 1 run's (written next to the model file)
  extra      further BASELINE configs measured in the same invocation (N = 1 only): 13B q4_1 decode, 7B prompt ingest n_batch = 128,
             7B decode at n_past ~ 256 and ~ 480, each with its own roofline object
"""
from __future__ import annotations

import argparse
import ctypes as C
import hashlib
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

PROMPT = "The quick brown fox jumps over the lazy dog."
# weights-only bytes of the 7*n_layer+1 quantised matmuls (SURVEY.md 8d)
ALGO_BYTES_PER_TOKEN = {("7B", "q4_0"): 4129423360, ("7B", "q4_1"): 4955308032, ("13B", "q4_1"): 9638707200, ("13B", "q4_0"): 8032256000,
                        ("65B", "q4_0"): 40638873600}
MATMUL_PARAMS = {"7B": 6607077376, "13B": 12851609600, "65B": 65022197760}     # elements of the 7*n_layer+1 quantised matrices


def log(*a):
    print(*a, file=sys.stderr, flush=True)


# The reference's C++ layers print a banner and progress on the process's stdout (fd 1).  The driver wants exactly one JSON
# line there, so fd 1 is pointed at stderr for the whole run and the line is written to a private duplicate of the real stdout.
_REAL_STDOUT = None


def _claim_stdout():
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.fdopen(os.dup(1), "w")
        os.dup2(2, 1)


def emit(line: dict):
    out = _REAL_STDOUT or sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


class _Stats(C.Structure):
    _fields_ = [("n_evals", C.c_uint64), ("last_eval_device_us", C.c_double), ("total_device_us", C.c_double),
                ("launches", C.c_uint64), ("graph_replays", C.c_uint64)]


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        super().__init__(daemon=True)
        self.gpu = gpu_index
        self.samples = []
        self.stop_flag = threading.Event()

    def run(self):
        while not self.stop_flag.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i", str(self.gpu)],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.samples.append([x.strip() for x in out.split(",")])
            except Exception:
                pass
            self.stop_flag.wait(0.1)

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unsampled"]}
        sm = sorted(float(s[0]) for s in self.samples if s[0].replace(".", "").isdigit())
        reasons = set()
        for s in self.samples:
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), s[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": float(self.samples[0][1]), "reasons": sorted(reasons),
                "samples": len(self.samples)}


# ---------------------------------------------------------------------------------------------------------------------
# model files and child processes
# ---------------------------------------------------------------------------------------------------------------------
def bench_dir() -> str:
    return os.environ.get("FASTLLAMA_BENCH_DIR", "/tmp")


def model_path(size: str, wtype_name: str) -> str:
    return os.path.join(bench_dir(), f"fastllama_b200_synth_{size}_{wtype_name}_seed0.bin")


def _child(args_list, timeout):
    """Run this script in a child process with a private stdout (the native layers are chatty) and return its rc."""
    return subprocess.run([sys.executable, os.path.abspath(__file__)] + args_list, stdout=sys.stderr, stderr=sys.stderr, timeout=timeout).returncode


def ensure_model(size: str, wtype_name: str) -> str:
    """The synthetic model file; generated on the GPU by a CHILD process, so the process that times the reference never maps
    this repository's CUDA library."""
    path = model_path(size, wtype_name)
    if not os.path.exists(path):
        t0 = time.time()
        rc = _child(["--_gen", size, wtype_name], timeout=1800)
        if rc != 0 or not os.path.exists(path):
            raise RuntimeError(f"synthetic model generation failed (rc {rc})")
        log(f"[bench] wrote synthetic {size} {wtype_name} model in {time.time() - t0:.1f}s -> {path}")
    return path


def _gen_main(size: str, wtype_name: str):
    from fastllama_b200.ggjt import write_synthetic_gpu

    path = model_path(size, wtype_name)
    tmp = path + f".tmp{os.getpid()}"
    n = write_synthetic_gpu(tmp, size=size, wtype={"q4_0": 2, "q4_1": 3}[wtype_name], seed=0, std=0.02)
    os.replace(tmp, path)
    log(f"[bench] {n / 1e9:.2f} GB")


def _long_prompt(n_chars: int, salt: int = 0) -> str:
    """Deterministic ASCII text; with the synthetic vocabulary every character is one token (byte fallback), plus BOS and
    the space the bridge prepends (reference lib/bridge.cpp:193-195): n_chars + 2 tokens."""
    words = PROMPT.split()
    out, i = [], salt
    while sum(len(w) + 1 for w in out) < n_chars + 1:
        out.append(words[i % len(words)])
        i += 1
    return " ".join(out)[:n_chars]


def _ref_worker_main(spec_path: str):
    """Child process: the reference's own CPU implementation through its own C ABI (oracle/_ref/pyfastllama_ref.so, the
    reference's sources compiled in place).  Loads nothing else native."""
    import numpy as np

    from fastllama_b200.model import Model, QuietLogger
    from oracle.pyoracle import REF_PYFASTLLAMA_SO

    spec = json.load(open(spec_path))
    if not os.path.exists(REF_PYFASTLLAMA_SO):
        raise RuntimeError("oracle/_ref/pyfastllama_ref.so is missing (build() must run where /root/reference exists)")
    t0 = time.time()
    m = Model(spec["path"], num_threads=spec["threads"], n_ctx=512, n_batch=spec.get("n_batch", 1), last_n_size=64, logger=QuietLogger(),
              use_mmap=True, library_path=REF_PYFASTLLAMA_SO)
    load_s = time.time() - t0
    res = {"load_s": load_s, "threads": spec["threads"]}
    greedy = dict(temp=0.0, top_k=1, top_p=1.0, repeat_penalty=1.0)
    if spec.get("ingest_chars"):
        # one n_batch-token eval of the prompt-ingest path: the prompt is n_batch + 1 tokens, ingest() evaluates the first chunk
        t1 = time.perf_counter()
        assert m.ingest(_long_prompt(spec["ingest_chars"]))
        res["ingest_s"] = time.perf_counter() - t1
    else:
        assert m.ingest(spec["prompt"])
    toks, logits = [], []
    for _ in range(spec.get("n_parity", 0)):
        got = []
        m.generate(lambda s: got.append(s), num_tokens=1, **greedy)
        if not got:
            break
        toks.append("".join(got))
        logits.append(m.get_logits_array())
    res["parity_tokens"] = toks
    if logits and spec.get("logits_out"):
        np.save(spec["logits_out"], np.stack(logits))
    n_timed = spec.get("n_timed", 0)
    if n_timed:
        # one generate(1) call per token so that a hopeless thread setting can be abandoned after `budget_s` (the bridge evaluates the
        # pending token and samples the next one per call, exactly as inside one long generate())
        budget = float(spec.get("budget_s", 60.0))
        for _ in range(spec.get("n_warm", 2)):
            m.generate(lambda s: None, num_tokens=1, **greedy)
        t_begin = time.perf_counter()
        n = 0
        while n < n_timed:
            m.generate(lambda s: None, num_tokens=1, **greedy)
            n += 1
            if time.perf_counter() - t_begin > budget:
                break
        dt = time.perf_counter() - t_begin
        res["timed_tokens"] = n
        res["tps"] = n / dt if dt > 0 else 0.0
    m.close()
    json.dump(res, open(spec["out"], "w"))


def run_ref_worker(spec: dict, timeout=900) -> dict:
    with tempfile.TemporaryDirectory() as td:
        spec = dict(spec, out=os.path.join(td, "out.json"))
        sp = os.path.join(td, "spec.json")
        json.dump(spec, open(sp, "w"))
        rc = _child(["--_ref-worker", sp], timeout=timeout)
        if rc != 0 or not os.path.exists(spec["out"]):
            raise RuntimeError(f"reference worker failed (rc {rc})")
        return json.load(open(spec["out"]))


def cpu_reference(path: str, size: str, wtype_name: str, steps: int, n_parity: int = 0, logits_out: str | None = None) -> dict:
    """Thread sweep of the reference's CPU path on the same file (BASELINE.md section 3: nproc, nproc/2, 32 -- the spin-barrier
    thread pool often peaks below nproc), then the sample proper at the best setting."""
    ncpu = os.cpu_count() or 1
    env = os.environ.get("FASTLLAMA_BENCH_CPU_THREADS")
    cands = [int(x) for x in env.split(",")] if env else sorted({t for t in (8, 16, 32, max(1, ncpu // 2), ncpu) if t <= ncpu})
    sweep = {}
    if len(cands) > 1:
        for t in cands:                                   # ascending; every setting is bounded to ~10 s
            r = run_ref_worker({"path": path, "threads": t, "prompt": PROMPT, "n_timed": 6, "n_warm": 1, "budget_s": 8.0})
            sweep[t] = r["tps"]
            log(f"[bench] reference CPU path, {t} threads: {r['tps']:.2f} tokens/s")
            if r["tps"] < 0.5 * max(sweep.values()):
                break                                     # past the knee of the spin-barrier thread pool: more threads only get slower
        best = max(sweep, key=sweep.get)
    else:
        best = cands[0]
    r = run_ref_worker({"path": path, "threads": best, "prompt": PROMPT, "n_parity": n_parity, "logits_out": logits_out, "n_timed": steps, "n_warm": 2, "budget_s": 60.0})
    sweep[best] = max(sweep.get(best, 0.0), r["tps"])
    cb = {"value": r["tps"], "unit": "tokens/s", "cores": best, "kind": "reference",
          "sample": f"{r['timed_tokens']} greedy decode tokens of the same synthetic {size} {wtype_name} file after 2 warm-up tokens, reference pyfastllama "
                    f"(oracle/_ref, AVX2 build) with num_threads={best}, the best of the sweep {{{', '.join(f'{k}: {v:.2f}' for k, v in sorted(sweep.items()))}}} tokens/s (threads: rate; ascending, stopped past the knee) "
                    f"on {ncpu} host cpus; child process, mmap load {r['load_s']:.1f}s not counted",
          "thread_sweep": {str(k): v for k, v in sorted(sweep.items())}, "host_cpus": ncpu}
    return {"cpu_baseline": cb, "parity_tokens": r.get("parity_tokens", [])}


# ---------------------------------------------------------------------------------------------------------------------
# our arm
# ---------------------------------------------------------------------------------------------------------------------
class Backend:
    """Handles to the three in-tree libraries; fails loudly without the CUDA library / a B200."""

    def __init__(self, local_rank: int):
        os.environ.setdefault("FASTLLAMA_DEVICE", str(local_rank))
        from fastllama_b200.build import lib_path
        from fastllama_b200.cuda_abi import FlCuda

        self.fl = FlCuda()
        self.props = self.fl.device_props()
        self.lib_path = lib_path
        g = C.CDLL(lib_path("libggml_b200.so"))
        g.ggml_b200_get_stats.argtypes = [C.POINTER(_Stats)]
        g.ggml_b200_get_host_profile.argtypes = [C.POINTER(C.c_double), C.c_int]
        self.ggml = g

    def stats(self) -> _Stats:
        s = _Stats()
        self.ggml.ggml_b200_get_stats(C.byref(s))
        return s

    def host_profile(self, reset=True):
        a = (C.c_double * 8)()
        self.ggml.ggml_b200_get_host_profile(a, 1 if reset else 0)
        return list(a)

    def model(self, path, n_batch=1):
        from fastllama_b200.model import Model, QuietLogger

        return Model(path, num_threads=1, n_ctx=512, n_batch=n_batch, last_n_size=64, logger=QuietLogger(), library_path=self.lib_path("pyfastllama.so"))


GREEDY = dict(temp=0.0, top_k=1, top_p=1.0, repeat_penalty=1.0)


def _synth_vocab():
    from fastllama_b200.ggjt import vocab_entries

    return {tok.decode(): i for i, (tok, _) in enumerate(vocab_entries(32000))}


SYNTH_VOCAB = _synth_vocab()          # text -> id of the synthetic model's vocabulary: every token streams as its own text


def dump_outputs(out_dir, **arrays):
    """--dump-outputs: what the timed path computed, as DIR/<name>.npy (logits float32, token ids float64)."""
    if not out_dir:
        return
    import numpy as np

    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), np.asarray(a, dtype=np.float32 if name == "logits" else np.float64))


def timed_decode(be: Backend, m, steps: int, dist=None, local_rank=0, sample_clocks=True):
    """K decode steps through Model.generate: device time (CUDA events around each eval's launches, summed by the library), wall
    clock, launches.  The streaming callback only counts: nothing but the reference-facing call sits in the timed region."""
    count, streamed = [0], []

    def on_token(s):
        count[0] += 1
        streamed.append(s)

    if dist:
        dist.barrier()
    be.fl.check(be.fl.lib.fl_sync())
    sampler = ClockSampler(local_rank) if sample_clocks else None
    if sampler:
        sampler.start()
    be.host_profile(reset=True)
    s0 = be.stats()
    launches0 = be.fl.lib.fl_launch_count()
    t0 = time.perf_counter()
    m.generate(on_token, num_tokens=steps, **GREEDY)
    be.fl.check(be.fl.lib.fl_sync())
    t1 = time.perf_counter()
    s1 = be.stats()
    launches = be.fl.lib.fl_launch_count() - launches0
    if sampler:
        sampler.stop_flag.set()
        sampler.join(timeout=2)
    hp = be.host_profile(reset=True)
    n_evals = int(s1.n_evals - s0.n_evals)
    return {"tokens": count[0], "token_ids": [SYNTH_VOCAB.get(t, -1) for t in streamed], "evals": n_evals, "device_s": (s1.total_device_us - s0.total_device_us) * 1e-6, "wall_s": t1 - t0, "launches": int(launches),
            "clocks": sampler.summary() if sampler else None,
            "host_us_per_step": ({"graph_match": hp[1] / hp[0], "match_scalars_launch_issue": hp[2] / hp[0], "device_wait_and_result_copies": hp[3] / hp[0],
                                  "caller_between_steps(sampling, graph build, callback)": hp[4] / hp[0]} if hp[0] else None)}


def roofline_hbm(algo_bytes, device_s, launches_timed, peak, peak_src, kernel, traffic=None, traffic_src=None):
    per_launch_s = device_s / launches_timed if launches_timed else 0.0
    achieved = algo_bytes / per_launch_s / 1e9 if per_launch_s else 0.0
    return {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak if peak else None, "traffic": traffic,
            "traffic_source": traffic_src, "kernel": kernel, "peak_source": peak_src, "launches_timed": launches_timed, "us_per_launch": per_launch_s * 1e6,
            "algorithmic_bytes_per_launch": algo_bytes}


TOKEN_KERNEL = "k_decode_token (persistent per-token kernel: every quantised matvec + attention of the decode step, 1 launch per token)"


def load_peaks():
    try:
        p = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        return p, "MEASURED_PEAKS.json (of measured)"
    except Exception:
        return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "B200_PROFILING.md fallback (of fallback)"


def committed_traffic():
    """DRAM bytes per k_decode_token launch from the newest committed ncu --set full capture (NOT measured in this run)."""
    best = None
    pdir = os.path.join(ROOT, "profiles")
    for name in sorted(os.listdir(pdir)) if os.path.isdir(pdir) else []:
        if name.endswith("_ncu_token_kernel.json"):
            best = name
    if not best:
        return None, None
    try:
        cap = json.load(open(os.path.join(pdir, best)))
        return int(cap["dram_bytes_read"]) + int(cap["dram_bytes_write"]), f"from_committed_profile: profiles/{best} (ncu --set full, one launch; not re-measured in this run)"
    except Exception:
        return None, None


def ingest_run(be: Backend, path: str, size: str, wtype_name: str, peaks, peak_src, steps: int = 2):
    """Prompt ingest with n_batch = 128: `steps` timed evals of 128 prompt tokens.  The 512-token context holds three of them, so they
    run in groups of at most three, each group one prompt of group*128 + 1 tokens on a reset model (ingest() evaluates the full
    128-token chunks; the last chunk, one token, is left to the first generate(); reference lib/bridge.cpp:213-232)."""
    m = be.model(path, n_batch=128)
    warm = _long_prompt(128 + 1 - 2)
    assert m.ingest(warm)                                  # uploads the weights, builds the N = 128 path once (untimed)
    m.generate(lambda s: None, num_tokens=1, **GREEDY)
    be.fl.check(be.fl.lib.fl_sync())
    s0 = be.stats()
    l0 = be.fl.lib.fl_launch_count()
    wall = 0.0
    left = steps
    while left > 0:
        batches = min(3, left)
        assert m.reset()
        t0 = time.perf_counter()
        assert m.ingest(_long_prompt(batches * 128 + 1 - 2, salt=3))
        be.fl.check(be.fl.lib.fl_sync())
        wall += time.perf_counter() - t0
        left -= batches
    last_logits = m.get_logits_array()                     # the last timed eval's logits (its last token)
    s1 = be.stats()
    evals = int(s1.n_evals - s0.n_evals)
    dev_s = (s1.total_device_us - s0.total_device_us) * 1e-6
    launches = int(be.fl.lib.fl_launch_count() - l0)
    n_tok = evals * 128
    flops = 2.0 * 128 * MATMUL_PARAMS[size]
    per_eval = dev_s / evals if evals else 0.0
    tf = flops / per_eval / 1e12 if per_eval else 0.0
    peak_t = float(peaks.get("bf16_tflops_sustained", 1400.0))
    algo = ALGO_BYTES_PER_TOKEN.get((size, wtype_name))
    res = {"metric": f"prompt tokens/sec LLaMA-{size} {wtype_name} ingest (n_batch=128)", "value": n_tok / dev_s if dev_s else 0.0, "unit": "tokens/s", "steps": evals,
           "ms_per_step": per_eval * 1e3, "config": {"workload": f"LLaMA-{size} {wtype_name} prompt ingest, n_batch=128, {evals} evals of 128 tokens at n_past 0..{n_tok - 128}, n_ctx=512"},
           "e2e": {"value": n_tok / wall, "unit": "tokens/s", "h2d_bytes_per_step": 128 * 4, "d2h_bytes_per_step": 32000 * 4 + 4 * {"7B": 4096, "13B": 5120, "65B": 8192}[size]},
           "gpu_launches": launches,
           "roofline": {"bound": "tensor", "achieved": tf, "peak": peak_t, "unit": "TFLOP/s", "frac": tf / peak_t, "traffic": None,
                        "kernel": "k_mul_mat_q_umma (tcgen05.mma kind::i8, one MMA per quant block into TMEM; exact fp32 block scaling on the CUDA cores) -- the whole eval "
                                  "(all 7*n_layer+1 GEMMs + attention + element-wise ops) is in the timed bracket",
                        "algorithmic_flops_per_step": flops, "peak_source": peak_src + " bf16_tflops_sustained (the MMAs are 8-bit integer; nominal i8 peak is 2x bf16)",
                        "hbm_line": {"achieved_gbs": (algo / per_eval / 1e9) if (algo and per_eval) else None, "peak_gbs": float(peaks.get("hbm_gbs", 6650.0)),
                                     "note": "weights read once per 128-token eval"}}}
    # continue into decode at n_past ~ 256: the KV cache now adds 2 * n_layer * n_past * n_embd * 4 bytes of reads per token
    extra_decode = []
    for target in (256, 480):
        cur = None
        if target == 480:
            # n_past is batches*128 + 16 now (+1 pending token).  A second prompt brings it to ~464; its last chunk is evaluated by an untimed
            # generate(1) so that the timed steps are all N = 1
            assert m.ingest(_long_prompt(464 - (batches * 128 + 16 + 1) - 2, salt=5))
            m.generate(lambda s: None, num_tokens=1, **GREEDY)
        r = timed_decode(be, m, 16, sample_clocks=False)       # 16 steps: what the 512-token context holds after these prompts
        if r["evals"]:
            cur = r
        if cur and algo:
            n_embd = {"7B": 4096, "13B": 5120, "65B": 8192}[size]
            n_layer = {"7B": 32, "13B": 40, "65B": 80}[size]
            n_past_mid = (batches * 128 + 8) if target == 256 else 464 + 8
            kv = 2 * n_layer * n_past_mid * n_embd * 4
            # the first eval of the 16 is the pending prompt chunk; all are N = 1 here
            rl = roofline_hbm(algo, cur["device_s"], cur["evals"], float(peaks.get("hbm_gbs", 6650.0)), peak_src + " hbm_gbs", TOKEN_KERNEL)
            rl["kv_cache_bytes_per_token_not_in_achieved"] = kv
            rl["achieved_incl_kv_gbs"] = (algo + kv) / (cur["device_s"] / cur["evals"]) / 1e9
            extra_decode.append({"metric": f"tokens/sec LLaMA-{size} {wtype_name} decode (n_batch=1, greedy) at n_past ~{n_past_mid}", "value": cur["evals"] / cur["device_s"], "unit": "tokens/s",
                                 "steps": cur["evals"], "ms_per_step": 1e3 * cur["device_s"] / cur["evals"], "e2e": {"value": cur["tokens"] / cur["wall_s"], "unit": "tokens/s"},
                                 "config": {"workload": f"LLaMA-{size} {wtype_name} greedy decode at n_past ~{n_past_mid} of n_ctx 512"}, "roofline": rl})
    m.close()
    res["last_logits"] = last_logits
    return res, extra_decode


def decode_run(be: Backend, path, size, wtype_name, steps, warmup, peaks, peak_src, dist=None, local_rank=0, parity_n=0):
    t0 = time.time()
    m = be.model(path, n_batch=1)
    log(f"[bench] model loaded in {time.time() - t0:.1f}s on {be.props['name']}")
    assert m.ingest(PROMPT)
    import numpy as np

    toks, logits = [], []
    for _ in range(parity_n):                                    # same procedure as the reference worker
        got = []
        m.generate(lambda s: got.append(s), num_tokens=1, **GREEDY)
        if not got:
            break
        toks.append("".join(got))
        logits.append(m.get_logits_array())
    m.generate(lambda s: None, num_tokens=max(warmup - len(toks), 3), **GREEDY)       # >= 3 untimed warm-up steps on the graph-replay path
    r = timed_decode(be, m, steps, dist=dist, local_rank=local_rank)
    r["last_logits"] = m.get_logits_array()                      # what the caller holds after the last timed step
    mode = int(be.ggml.ggml_b200_decode_mode())
    m.close()
    return r, mode, toks, (np.stack(logits) if logits else None)


def compare_parity(ref_tokens, ref_logits, our_tokens, our_logits):
    import numpy as np

    n = min(len(ref_tokens), len(our_tokens))
    first = next((i for i in range(n) if ref_tokens[i] != our_tokens[i]), None)
    out = {"prompt": PROMPT, "tokens_compared": n, "greedy_ids_equal": first is None and n > 0, "first_divergence": first}
    if ref_logits is not None and our_logits is not None and n:
        # logits are comparable while both arms have evaluated the same token sequence: steps 0 .. first_divergence inclusive
        upto = n if first is None else first + 1
        rel = []
        for i in range(upto):
            rel.append(float(np.abs(our_logits[i].astype(np.float64) - ref_logits[i]).max() / np.abs(ref_logits[i]).max()))
        out["logits_maxabs_over_range"] = max(rel)
        out["logits_maxabs_over_range_median_step"] = float(np.median(rel))
        out["logits_steps_compared"] = upto
        out["logits_unit"] = "max|ours - reference| / max|reference| per step (fp32 logits of 32000 tokens)"
        gaps = []
        for i in range(upto):
            srt = np.sort(ref_logits[i])
            gaps.append(float((srt[-1] - srt[-2]) / np.abs(ref_logits[i]).max()))
        out["reference_top1_top2_gap_min"] = min(gaps)
        out["reference_top1_top2_gap_median"] = float(np.median(gaps))
        if first is not None:
            out["reference_top1_top2_gap_at_divergence"] = gaps[first]
            out["logits_maxabs_at_divergence"] = rel[first]
        out["logits_bit_identical"] = bool(all(np.array_equal(our_logits[i].view(np.uint32), np.asarray(ref_logits[i], dtype=np.float32).view(np.uint32)) for i in range(upto)))
        if out["logits_bit_identical"]:
            out["note"] = ("every fp32 operation of the path follows the reference's order (the eight accumulators of its AVX2 row kernels, ggml_vec_dot_f32's "
                           "lanes and leftovers; fastllama_b200/csrc/fl_exact.cuh), so the logits carry the reference's bits; DESIGN.md section 5")
        else:
            out["note"] = ("every activation is re-quantised to q8_0 before every matmul (reference lib/ggml.c:8105-8119): a dense relative perturbation d becomes "
                           "sqrt(d * step) after one quantised matmul (step = 1/127 of a block's amax), so one differing ulp anywhere settles at a few per cent of "
                           "max|logit| within a layer or two on this random-weight model; DESIGN.md section 5.  A prompt of 16 tokens or more goes through the "
                           "tcgen05 GEMM, whose block terms are added in another fp32 order (FASTLLAMA_B200_INGEST=exact keeps the reference's order)")
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=128)
    ap.add_argument("--warmup", type=int, default=8)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--mode", default="decode", choices=["decode", "ingest"])
    ap.add_argument("--size", default="7B")
    ap.add_argument("--wtype", default="q4_0", choices=["q4_0", "q4_1"])
    ap.add_argument("--cpu-steps", type=int, default=12, help="decode tokens of the CPU baseline sample")
    ap.add_argument("--parity-tokens", type=int, default=32)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true")
    ap.add_argument("--dump-outputs", default=None, metavar="DIR",
                    help="write what the timed path computed to DIR: logits.npy (float32, the last timed eval's logits) and, for decode, "
                         "tokens.npy (float64, the token ids the timed steps produced), to compare two builds output for output")
    ap.add_argument("--_gen", nargs=2, default=None, help=argparse.SUPPRESS)
    ap.add_argument("--_ref-worker", default=None, help=argparse.SUPPRESS)
    args = ap.parse_args()
    if args._gen:
        return _gen_main(*args._gen)
    if args._ref_worker:
        return _ref_worker_main(args._ref_worker)
    args.warmup = max(args.warmup, 3)
    _claim_stdout()

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    workload = (f"LLaMA-{args.size} {args.wtype} greedy decode, n_batch=1, n_ctx=512, synthetic random weights N(0,0.02^2) seed 0" if args.mode == "decode" else
                f"LLaMA-{args.size} {args.wtype} prompt ingest, n_batch=128, n_ctx=512, synthetic random weights N(0,0.02^2) seed 0")
    metric = (f"tokens/sec LLaMA-{args.size} {args.wtype} decode (n_batch=1, greedy)" if args.mode == "decode" else
              f"prompt tokens/sec LLaMA-{args.size} {args.wtype} ingest (n_batch=128)")
    algo = ALGO_BYTES_PER_TOKEN.get((args.size, args.wtype))
    # identical in both arms (the driver compares it): what is measured, not how
    config = {"workload": workload, "prompt": PROMPT, "algorithmic_bytes_per_token": algo,
              "parallelism": "1 GPU" if args.gpus == 1 else f"tp{args.gpus} (one decode stream, tensor parallel)",
              "l2": f"inputs ({(algo or 0) / 1e9:.2f} GB of weights per step) are {(algo or 0) / 126e6:.0f}x larger than L2; no flush needed"}

    # ---------------------------------------------------------------- reference arm (CPU, rank 0 only; no library of this repository in the timing process)
    if args.impl == "reference":
        if rank != 0:
            return
        t0 = time.perf_counter()
        path = ensure_model(args.size, args.wtype)
        steps = min(args.steps, int(os.environ.get("FASTLLAMA_BENCH_REF_MAX_STEPS", "24")))
        if args.mode == "ingest":
            ncpu = os.cpu_count() or 1
            r = run_ref_worker({"path": path, "threads": min(32, ncpu), "n_batch": 128, "ingest_chars": 128 + 1 - 2}, timeout=1800)
            value = 128 / r["ingest_s"]
            cb = {"value": value, "unit": "tokens/s", "cores": r["threads"], "kind": "reference",
                  "sample": f"ONE 128-token eval of the prompt-ingest path (prompt of 129 tokens, the reference evaluates the first chunk inside ingest()), num_threads={r['threads']} of {ncpu}"}
            steps = 1
        else:
            cb = cpu_reference(path, args.size, args.wtype, steps)["cpu_baseline"]
            value = cb["value"]
        line = {"impl": "reference", "metric": metric, "value": value, "unit": "tokens/s", "n_gpus": args.gpus, "steps": steps, "warmup": 2,
                "ms_per_step": 1000.0 / value if value else None, "higher_is_better": True, "scaling": "strong" if args.gpus > 1 else "weak", "vs_baseline": None, "dtype": "u8",
                "data": "synthetic", "config": config, "cpu_baseline": cb,
                "e2e": {"value": value, "unit": "tokens/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "arm": "reference CPU path: oracle/_ref/pyfastllama_ref.so = the reference's lib/ggml.c, lib/llama.cpp, lib/bridge.cpp, interfaces/c/main.cpp compiled in place "
                       "(oracle/Makefile), driven through its C ABI by the ctypes mirror of its own interfaces/python/fastllama.py (that file cannot travel to the GPU box)",
                "wall_s": time.perf_counter() - t0}
        emit(line)
        return

    # ---------------------------------------------------------------- our arm
    dist = None
    if world > 1:
        import torch
        import torch.distributed as dist_mod

        torch.cuda.set_device(local_rank)
        dist_mod.init_process_group("nccl")
        dist = dist_mod
    be = Backend(local_rank)
    fl = be.fl
    tp = world > 1 and not os.environ.get("FASTLLAMA_BENCH_REPLICAS")
    if tp:
        # tensor parallelism (SURVEY.md 8e): one NCCL communicator over all ranks; rank 0's unique id travels by torch.distributed
        import torch

        idbuf = torch.zeros(128, dtype=torch.uint8, device="cuda")
        if rank == 0:
            raw = C.create_string_buffer(128)
            fl.check(fl.lib.fl_comm_unique_id(raw))
            idbuf = torch.tensor(list(raw.raw), dtype=torch.uint8, device="cuda")
        dist.broadcast(idbuf, 0)
        fl.check(fl.lib.fl_comm_init(rank, world, bytes(idbuf.cpu().numpy().tobytes())))
    if rank == 0:
        ensure_model(args.size, args.wtype)
    if dist:
        dist.barrier()
    path = model_path(args.size, args.wtype)
    peaks, peak_src = load_peaks()
    peak = float(peaks.get("hbm_gbs", 6650.0))

    if args.mode == "ingest":
        assert world == 1, "--mode ingest is a single-GPU measurement"
        res, extra_decode = ingest_run(be, path, args.size, args.wtype, peaks, peak_src, steps=args.steps)
        res.update({"n_gpus": 1, "warmup": 1, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic"})
        res["config"] = config
        res["device"] = be.props["name"]
        res["extra"] = extra_decode
        dump_outputs(args.dump_outputs, logits=res.pop("last_logits"))
        emit(res)
        return

    headline = args.size == "7B" and args.wtype == "q4_0"
    # CPU baseline + parity reference first (rank 0, N = 1), in child processes
    cpu_baseline, parity = None, None
    ref_tokens, ref_logits = [], None
    parity_n = args.parity_tokens if headline else 0
    from oracle.pyoracle import REF_PYFASTLLAMA_SO

    if rank == 0 and world == 1 and not args.no_cpu_baseline and not os.path.exists(REF_PYFASTLLAMA_SO):
        log("[bench] cpu_baseline and parity skipped: the reference's CPU library (oracle/_ref) is not built here")
    elif rank == 0 and world == 1 and not args.no_cpu_baseline:
        import numpy as np

        with tempfile.TemporaryDirectory() as td:
            lp = os.path.join(td, "ref_logits.npy")
            cr = cpu_reference(path, args.size, args.wtype, args.cpu_steps, n_parity=parity_n, logits_out=lp)
            cpu_baseline, ref_tokens = cr["cpu_baseline"], cr["parity_tokens"]
            if os.path.exists(lp):
                ref_logits = np.load(lp)
        log(f"[bench] cpu_baseline: {cpu_baseline['value']:.2f} tokens/s on {cpu_baseline['cores']} threads")

    r, decode_mode, our_tokens, our_logits = decode_run(be, path, args.size, args.wtype, args.steps, args.warmup, peaks, peak_src, dist=dist, local_rank=local_rank,
                                                         parity_n=parity_n if (world == 1 or tp) else 0)
    n_tok = r["tokens"]
    if n_tok < args.steps:
        log(f"[bench] rank {rank}: generation stopped after {n_tok} of {args.steps} tokens (EOS); rates use the tokens produced")
    wall, device_s = r["wall_s"], r["device_s"]
    if rank == 0:
        dump_outputs(args.dump_outputs, logits=r["last_logits"], tokens=r["token_ids"])
    tok_file = os.path.join(bench_dir(), f"fastllama_b200_parity_{args.size}_{args.wtype}_n1.json")
    if world == 1 and our_tokens:
        if ref_tokens:
            parity = compare_parity(ref_tokens, ref_logits, our_tokens, our_logits)
        try:
            json.dump({"tokens": our_tokens, "logits_sha256": hashlib.sha256(our_logits.tobytes()).hexdigest()}, open(tok_file, "w"))
        except Exception:
            pass
    if dist:
        import numpy as np
        import torch

        t = torch.tensor([wall, device_s, float(n_tok)], dtype=torch.float64, device="cuda")
        mx = t.clone()
        dist.all_reduce(mx, op=dist.ReduceOp.MAX)
        sm = t.clone()
        dist.all_reduce(sm, op=dist.ReduceOp.SUM)
        wall, device_s = float(mx[0]), float(mx[1])
        total_tokens = float(n_tok) if tp else float(sm[2])        # tensor parallel: every rank decodes the SAME stream
        if tp and our_logits is not None:
            # every rank must hold bit-identical logits (the reductions add the ranks' partial sums in rank order everywhere)
            h = np.frombuffer(hashlib.sha256(our_logits.tobytes()).digest()[:8], dtype=np.int64).copy()
            hs = [torch.zeros(1, dtype=torch.int64, device="cuda") for _ in range(world)]
            dist.all_gather(hs, torch.tensor(h, device="cuda"))
            same = all(int(x) == int(hs[0]) for x in hs)
            parity = {"prompt": PROMPT, "ranks_logits_bit_identical": same, "tokens_compared": len(our_tokens), "logits_sha256": hashlib.sha256(our_logits.tobytes()).hexdigest()}
            try:
                n1 = json.load(open(tok_file))
                k = min(len(n1["tokens"]), len(our_tokens))
                first = next((i for i in range(k) if n1["tokens"][i] != our_tokens[i]), None)
                parity.update({"vs_n1_run": {"tokens_compared": k, "greedy_ids_equal": first is None, "first_divergence": first,
                                             "logits_bit_identical": n1.get("logits_sha256") == parity["logits_sha256"] and k == len(our_tokens),
                                             "note": "every matrix is row-split and the activation vectors are gathered, so each row is summed on one GPU in the reference's order: N GPUs give the bits of one"}})
            except Exception:
                parity["vs_n1_run"] = "no 1-GPU token file on this box"
    else:
        total_tokens = float(n_tok)
    if rank != 0:
        return

    value = total_tokens / device_s if device_s > 0 else 0.0
    e2e = total_tokens / wall if wall > 0 else 0.0
    from fastllama_b200.ggjt import LLAMA_SIZES

    n_embd_model = LLAMA_SIZES[args.size][0]
    traffic, traffic_src = committed_traffic() if (headline and world == 1 and decode_mode == 2) else (None, None)
    if decode_mode == 2 and algo and r["evals"]:
        # per-GPU algorithmic bytes: the weights are sharded N ways under tensor parallelism (the LM head and all layers split evenly)
        rl = roofline_hbm(algo / (world if tp else 1), device_s, r["evals"], peak, peak_src + " hbm_gbs", TOKEN_KERNEL, traffic, traffic_src)
        if tp:
            rl["per_gpu"] = True
    else:
        rl = {"bound": "hbm", "achieved": (algo * value / 1e9) if algo else None, "peak": peak, "unit": "GB/s", "frac": (algo * value / 1e9 / peak) if algo else None, "traffic": None,
              "kernel": "k_mv_fused (one launch per matrix group; the persistent token kernel was not used)", "peak_source": peak_src}
    par_detail = "1 GPU" if world == 1 else (
        (f"tp{world}: every matrix row-split (wq/wk/wv by heads; wo, w1/w3, w2, output by rows); the 4 activation vectors per layer are gathered inside the persistent "
         "token kernel as dataflow vectors ({value, epoch} words pushed into every rank's peer-mapped buffer over NVLink, no barrier), 1 NCCL all-gather of the logits, all in the CUDA graph") if tp else f"{world} independent replicas")
    line = {
        "metric": metric, "value": value, "unit": "tokens/s", "n_gpus": world, "steps": n_tok, "warmup": args.warmup,
        "ms_per_step": 1000.0 * device_s / n_tok if n_tok else None, "higher_is_better": True,
        # one decode stream: the total work is fixed as N grows (tensor parallel = strong scaling); N = 1 carries the same label
        "scaling": "weak" if (world > 1 and not tp) else "strong",
        "vs_baseline": None, "dtype": "u8", "data": "synthetic", "config": config,
        "e2e": {"value": e2e, "unit": "tokens/s", "h2d_bytes_per_step": 8, "d2h_bytes_per_step": 32000 * 4 + n_embd_model * 4,
                "api": "fastllama_b200.Model.generate -> pyfastllama.so (llama_* C ABI) -> libggml_b200 -> libfl_cuda",
                "host_us_per_step": r["host_us_per_step"]},
        "gpu_launches": r["launches"], "roofline": rl, "clocks": r["clocks"], "parallelism_detail": par_detail, "device": be.props["name"],
    }
    if cpu_baseline:
        line["cpu_baseline"] = cpu_baseline
        line["speedup_like_for_like"] = {"e2e_over_cpu_wall": e2e / cpu_baseline["value"] if cpu_baseline["value"] else None,
                                         "note": "both wall-clock through Model.generate; `value` is device-timed and is not comparable with cpu_baseline"}
    if parity:
        line["parity"] = parity

    # ---------------------------------------------------------------- further BASELINE configs, same invocation (N = 1 headline run only)
    if headline and world == 1 and not args.no_extras and not os.environ.get("FASTLLAMA_BENCH_NO_EXTRAS"):
        extra = []
        try:
            res, extra_decode = ingest_run(be, path, "7B", "q4_0", peaks, peak_src, steps=2)
            res.pop("last_logits")
            extra.append(res)
            extra.extend(extra_decode)
        except Exception as e:                                     # an extra never takes the headline line down
            extra.append({"metric": "prompt ingest n_batch=128", "error": repr(e)})
        try:
            p13 = ensure_model("13B", "q4_1")
            r13, mode13, _, _ = decode_run(be, p13, "13B", "q4_1", 32, 5, peaks, peak_src)
            a13 = ALGO_BYTES_PER_TOKEN[("13B", "q4_1")]
            extra.append({"metric": "tokens/sec LLaMA-13B q4_1 decode (n_batch=1, greedy)", "value": r13["evals"] / r13["device_s"], "unit": "tokens/s", "steps": r13["evals"],
                          "ms_per_step": 1e3 * r13["device_s"] / r13["evals"], "e2e": {"value": r13["tokens"] / r13["wall_s"], "unit": "tokens/s"},
                          "config": {"workload": "LLaMA-13B q4_1 greedy decode, n_batch=1, n_ctx=512, synthetic random weights"},
                          "roofline": roofline_hbm(a13, r13["device_s"], r13["evals"], peak, peak_src + " hbm_gbs", TOKEN_KERNEL if mode13 == 2 else "k_mv_fused")})
            try:
                os.remove(p13)                                     # 9.6 GB; the headline model stays for the reference arm / scaling runs
            except OSError:
                pass
        except Exception as e:
            extra.append({"metric": "LLaMA-13B q4_1 decode", "error": repr(e)})
        line["extra"] = extra
    emit(line)


if __name__ == "__main__":
    main()
