#!/usr/bin/env python
"""bench.py -- the north-star measurement: RWKV-6-World-7B-shape Q5_1, single-token decode and 128-token
prefill through the rwkv.h C ABI of rwkv.cpp_b200/librwkv.so, on N B200s of one node.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload rwkv6-7b:Q5_1] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

One "step" = one single-token evaluation (with logits) of the whole model. Prints ONE JSON line:
  value        decode tokens/s, state resident in HBM, CUDA-event timed on the library's own stream
  e2e          the same metric through rwkv_eval() with HOST state/logits buffers (H2D + D2H inside the timed region)
  prefill      128-token rwkv_eval_sequence chunk: device-timed and e2e tokens/s
  roofline     dominant kernel (fused dequant-GEMV): algorithmic weight bytes / its share of the graph-replayed step (critical-path
               attribution of the in-kernel %globaltimer timeline x the CUDA-event step time) vs MEASURED_PEAKS.json
  cpu_baseline the UNMODIFIED reference (oracle/_ref) timed on this box's host cores on a bounded sample
Weights are synthetic (random-init, exact shapes/dtypes; tools/synthetic_model.py); no checkpoints exist offline.
The 6 GB of weights streamed per token exceed the 126 MB L2 48x, so no explicit L2 flush is needed between steps.
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
sys.path.insert(0, os.path.join(ROOT, "oracle"))

PF = ctypes.POINTER(ctypes.c_float)
PU = ctypes.POINTER(ctypes.c_uint32)
CACHE_DIR = os.environ.get("RWKV_B200_BENCH_DIR", "/tmp/rwkv_b200_bench")
PREFILL_TOKENS = 128


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=128)
    ap.add_argument("--warmup", type=int, default=8)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="rwkv6-7b:Q5_1", help="<preset>:<format>, presets in tools/synthetic_model.py")
    ap.add_argument("--prefill-steps", type=int, default=8)
    ap.add_argument("--skip-cpu-baseline", action="store_true")
    ap.add_argument("--quick", action="store_true", help="A/B aid, not a bench line: resident decode timing + kernel timeline only")
    ap.add_argument("--cpu-budget-s", type=float, default=20.0, help="CPU seconds the bounded reference sample may take per leg")
    ap.add_argument("--mode", default="decode", choices=["decode", "prefill"],
                    help="headline metric: single-token decode tokens/s (default) or 128-token-chunk prefill tokens/s (one step = one chunk)")
    ap.add_argument("--dump-outputs", default=None, metavar="DIR",
                    help="after the timed steps of the headline metric, write the logits and recurrent state of its last step as DIR/<name>.npy (float32)")
    # internal: the reference library only ever runs in child processes (hard timeouts), see cpu_reference_leg
    ap.add_argument("--ref-child", default=None, choices=["probe", "full"], help=argparse.SUPPRESS)
    ap.add_argument("--ref-threads", default="8", help=argparse.SUPPRESS)
    ap.add_argument("--workload-path", default=None, help=argparse.SUPPRESS)
    ap.add_argument("--no-prefill", action="store_true", help=argparse.SUPPRESS)
    return ap.parse_args()


# ------------------------------------------------------------------------------------------------
def workload_file(spec, rank=0, world=1, barrier=None):
    import synthetic_model as sm
    preset, fmt = spec.split(":")
    os.makedirs(CACHE_DIR, exist_ok=True)
    path = os.path.join(CACHE_DIR, f"{preset}-{fmt}-seed1.bin")
    if rank == 0 and not os.path.isfile(path):
        tmp = path + ".tmp"
        sm.write_direct(tmp, preset, fmt, seed=1)
        os.replace(tmp, path)
    if barrier:
        barrier()
    return path, sm.PRESETS[preset]


class ClockSampler:
    """nvidia-smi clocks/throttle reasons DURING the timed regions (B200_PROFILING.md recipe)."""

    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, gpu_index=0):
        self.rows, self.proc, self.gpu = [], None, gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [c.strip() for c in line.split(",")]))

    def stop(self):
        if self.proc:
            self.proc.terminate()

    def summary(self, windows):
        rows = [r for ts, r in self.rows if any(a <= ts <= b for a, b in windows)] or [r for _, r in self.rows]
        sm, reasons, mx = [], set(), None
        for r in rows:
            try:
                sm.append(float(r[0])); mx = float(r[1])
            except (ValueError, IndexError):
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


def host_buffers(n_state, n_logits, kind="pinned"):
    """Host state / logits buffers for the e2e legs: pinned (what a serving process would hold) or pageable numpy arrays (what the
    reference's Python binding passes, rwkv_cpp_model.py:330-351)."""
    if kind == "pinned":
        try:
            import torch
            if torch.cuda.is_available():
                s = torch.zeros(n_state, dtype=torch.float32).pin_memory()
                l = torch.zeros(n_logits, dtype=torch.float32).pin_memory()
                return s, l, s.data_ptr(), l.data_ptr(), "pinned"
        except Exception:
            pass
    s, l = np.zeros(n_state, np.float32), np.zeros(n_logits, np.float32)
    return s, l, s.ctypes.data, l.ctypes.data, "pageable"


DUMP_BYTES = 64 << 20


def dump_outputs(L, ctx, n_state, n_vocab, out_dir):
    """Writes what the last resident step left on the device, the arrays a caller of rwkv_b200_eval_resident reads back: the logits
    of its last token and the recurrent state. The inputs are seeded, so two builds run with the same arguments can be compared
    array by array. A state too large for the 64 MB budget is written as a fixed sample (seed 0, ascending indices)."""
    logits, state = np.zeros(n_vocab, np.float32), np.zeros(n_state, np.float32)
    ok = L.rwkv_b200_stage_logits(ctx.ptr, logits.ctypes.data_as(PF), None) and L.rwkv_b200_state_store(ctx.ptr, state.ctypes.data_as(PF))
    assert ok, "reading the outputs of the last step back failed"
    room = (DUMP_BYTES - logits.nbytes - 2 * 4096) // state.itemsize       # 4 KB per .npy header is ample
    if state.size > room:
        state = state[np.sort(np.random.default_rng(0).choice(state.size, room, replace=False))]
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "logits.npy"), logits)
    np.save(os.path.join(out_dir, "state.npy"), state)
    log("outputs of the last timed step written to %s (logits %d, state %d of %d values)" % (out_dir, logits.size, state.size, n_state))


def prefill_matmul_flops(preset, n_tokens):
    """FLOPs of the weight contractions of one chunk: 2 * (elements of every per-layer matrix) * tokens (+ the head, one token)."""
    major, minor = preset["arch"]
    C, F, Lr, V = preset["C"], preset["F"], preset["L"], preset["V"]
    if major == 4:
        per_layer = 4 * C * C + 2 * C * F + C * C
    elif major == 5:
        per_layer = (5 if minor >= 2 else 4) * C * C + 2 * C * F + C * C
    elif major == 6:
        mix, dec = preset["mix"], preset["decay"]
        per_layer = 5 * C * C + C * 5 * mix + 5 * mix * C + 2 * C * dec + 2 * C * F + C * C
    else:
        per_layer = 4 * C * C + 2 * C * (preset["lora_w"] + preset["lora_a"] + preset["lora_v"] + preset["lora_g"]) + 2 * C * F
    return 2.0 * per_layer * Lr * n_tokens + 2.0 * C * V


def measured_tensor_peak():
    try:
        p = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        return float(p["bf16_tflops_sustained"]), "measured (MEASURED_PEAKS.json bf16_tflops_sustained)"
    except Exception:
        return 1500.0, "fallback (B200_PROFILING.md)"


def ncu_traffic(preset):
    """DRAM bytes of the dominant kernel's largest per-layer launch from the committed ncu capture (tools/ncu_summary.py --traffic),
    next to that launch's algorithmic bytes (ffn key + receptance batch: (F + C) rows of C/32 Q5_1 blocks)."""
    try:
        import glob
        f = sorted(glob.glob(os.path.join(ROOT, "profiles", "*_ncu_traffic.json")))[-1]
        t = json.load(open(f))
        algo = (preset["F"] + preset["C"]) * (preset["C"] // 32) * 24
        return t["dram_bytes"], {"source": os.path.relpath(f, ROOT), "kernel": t["kernel"], "launch": "ffn key + receptance (one launch, 296 CTAs)",
                                 "algorithmic_bytes": algo, "dram_over_algorithmic": t["dram_bytes"] / algo}
    except Exception:
        return None, None


def measured_peaks():
    try:
        p = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        return float(p["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs, STREAM-style copy)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


def kernel_timeline(L, ctx, tok_arr, T=1, passes=6, skip=3):
    """One decode step as the kernels see it: every kernel folds %globaltimer of its CTAs into a [start, end] record (works inside
    CUDA-graph replays). Returns the traced span and the critical-path attribution per kernel family: a kernel is charged the time by
    which it pushed the end of the timeline out, so the shares add up to the span exactly."""
    N = 1024
    st, en = (ctypes.c_double * N)(), (ctypes.c_double * N)()
    names = ctypes.create_string_buffer(32 * N)
    L.rwkv_b200_state_load(ctx.ptr, None)
    if not L.rwkv_b200_trace_enable(ctx.ptr):
        return {"span_us": 0.0, "attributed_us": {}, "busy_us": {}, "launches": {}}
    best = None
    for i in range(passes):                    # eager, eager, capture, replay ... : keep the shortest replayed step
        L.rwkv_b200_eval_resident(ctx.ptr, ctypes.cast(ctypes.byref(tok_arr, 4 * i * T), PU), T, True, None)
        n = L.rwkv_b200_trace_read(ctx.ptr, st, en, ctypes.cast(names, ctypes.c_void_p), N)
        if i < skip or n <= 0:
            continue
        rows = [(names.raw[32 * j:32 * j + 32].split(b"\0")[0].decode(), st[j], en[j]) for j in range(n)]
        t_begin, t_end = min(r[1] for r in rows), max(r[2] for r in rows)
        att, busy, cnt, pe = {}, {}, {}, t_begin
        for nm, s_, e_ in rows:
            fam = "gemv" if nm.startswith("gemv") else ("gemm_tc" if nm.startswith("gemm_tc") else nm)
            cnt[fam] = cnt.get(fam, 0) + 1
            busy[fam] = busy.get(fam, 0.0) + (e_ - s_)
            if e_ > pe:
                att[fam] = att.get(fam, 0.0) + (e_ - pe)
                pe = e_
        cur = {"span_us": t_end - t_begin, "attributed_us": att, "busy_us": busy, "launches": cnt}
        if best is None or cur["span_us"] < best["span_us"]:
            best = cur
    L.rwkv_b200_trace_disable(ctx.ptr)
    return best or {"span_us": 0.0, "attributed_us": {}, "busy_us": {}, "launches": {}}


# ------------------------------------------------------------------------------------------------
def physical_cores():
    """Distinct (socket, core) pairs among the CPUs this process may run on (hyper-threads counted once)."""
    allowed = os.sched_getaffinity(0) if hasattr(os, "sched_getaffinity") else set(range(os.cpu_count() or 1))
    seen, cpu, phys = set(), None, "0"
    try:
        for line in open("/proc/cpuinfo"):
            k, _, v = line.partition(":")
            k = k.strip()
            if k == "processor":
                cpu = int(v)
            elif k == "physical id":
                phys = v.strip()
            elif k == "core id" and cpu in allowed:
                seen.add((phys, v.strip()))
    except (OSError, ValueError):
        pass
    return len(seen) or len(allowed)


def reference_thread_candidates():
    """ggml's spin barriers collapse when oversubscribed (round 1: 128 threads on the 8-GPU node never returned), so the
    reference is never given more threads than min(32, cgroup quota / affinity, physical cores)."""
    if "RWKV_REF_THREADS" in os.environ:
        return [int(os.environ["RWKV_REF_THREADS"])]
    cap = max(1, min(32, available_cpus(), physical_cores()))
    return sorted({max(1, min(cap, c)) for c in (8, 16, 32)})


def _ref_bind(path, threads):
    import ref_lib
    ref = ref_lib.load_reference_library()
    ref.rwkv_set_print_errors(None, False)
    t0 = time.time()
    ctx = ref.rwkv_init_from_file(path.encode(), threads, 0)
    if not ctx:
        raise RuntimeError("reference failed to load " + path)
    return ref, ctx, time.time() - t0, os.path.basename(ref_lib.reference_library_path())


def ref_child_probe(path, candidates):
    """Child process: loads the model ONCE, then one clone per candidate thread count (rwkv_clone_context takes n_threads,
    rwkv.h:80), 1 warm + 2 timed tokens each; one JSON line per candidate as soon as it is known, so a candidate that
    hangs costs the parent only its own timeout."""
    ref, ctx, load_s, _ = _ref_bind(path, candidates[0])
    n_state, n_vocab = ref.rwkv_get_state_len(ctx), ref.rwkv_get_logits_len(ctx)
    st, lg = np.zeros(n_state, np.float32), np.zeros(n_vocab, np.float32)
    sp, lp = st.ctypes.data_as(PF), lg.ctypes.data_as(PF)
    emit({"loaded": True, "load_s": load_s})
    for th in candidates:
        c = ref.rwkv_clone_context(ctx, th)
        ref.rwkv_init_state(c, sp)
        ref.rwkv_eval(c, 1, sp, sp, lp)
        t0 = time.perf_counter()
        for t in (2, 3):
            ref.rwkv_eval(c, t, sp, sp, lp)
        emit({"threads": th, "ms": (time.perf_counter() - t0) / 2 * 1e3})
        ref.rwkv_free(c)
    ref.rwkv_free(ctx)


def ref_child_full(path, threads, steps, warmup, budget_s, want_prefill):
    """Child process: `warmup` untimed + up to `steps` timed rwkv_eval calls (bounded by budget_s of CPU time), then one
    128-token chunk after one warm-up chunk when that fits the budget."""
    import synthetic_model as sm
    ref, ctx, load_s, libname = _ref_bind(path, threads)
    n_state, n_vocab = ref.rwkv_get_state_len(ctx), ref.rwkv_get_logits_len(ctx)
    state, logits = np.zeros(n_state, np.float32), np.zeros(n_vocab, np.float32)
    ref.rwkv_init_state(ctx, state.ctypes.data_as(PF))
    toks = sm.synthetic_tokens(4096, n_vocab)
    sp, lp = state.ctypes.data_as(PF), logits.ctypes.data_as(PF)
    warmup = max(2, warmup)                      # the first call builds the scheduler
    t0 = time.time()
    for t in toks[:warmup]:
        ref.rwkv_eval(ctx, t, sp, sp, lp)
    probe = (time.time() - t0) / warmup
    n = int(max(4, min(steps, budget_s / max(probe, 1e-6))))
    times = []
    for t in toks[warmup:warmup + n]:
        t0 = time.perf_counter()
        ref.rwkv_eval(ctx, t, sp, sp, lp)
        times.append(time.perf_counter() - t0)
    med, mean = float(np.median(times)), float(np.mean(times))
    out = {"decode_tokens_per_s": 1.0 / mean, "decode_ms_per_token": mean * 1e3, "decode_ms_median": med * 1e3, "decode_sample_tokens": n, "warmup": warmup,
           "threads": threads, "load_s": load_s, "library": libname}
    if want_prefill and mean * PREFILL_TOKENS < 4 * budget_s:
        arr = (ctypes.c_uint32 * PREFILL_TOKENS)(*toks[:PREFILL_TOKENS])
        ref.rwkv_eval_sequence_in_chunks(ctx, arr, PREFILL_TOKENS, PREFILL_TOKENS, None, sp, lp)   # builds + caches the sequence graph
        reps = []
        for _ in range(2):
            t0 = time.perf_counter()
            ref.rwkv_eval_sequence_in_chunks(ctx, arr, PREFILL_TOKENS, PREFILL_TOKENS, None, sp, lp)
            reps.append(time.perf_counter() - t0)
            if reps[-1] > budget_s / 2:
                break
        out["prefill_tokens_per_s"] = PREFILL_TOKENS / float(np.mean(reps))
        out["prefill_ms_per_chunk"] = float(np.mean(reps)) * 1e3
        out["prefill_sample"] = "%d chunk(s) of 128 tokens after one warm-up chunk" % len(reps)
    ref.rwkv_free(ctx)
    emit(out)


def _run_child(argv, timeout_s, on_line=None):
    """Runs `bench.py <argv>` as a child; returns its JSON stdout lines. The child is killed when `timeout_s` passes without
    it finishing (lines printed before that are kept) -- a hung ggml thread pool can never take the bench with it."""
    proc = subprocess.Popen([sys.executable, os.path.abspath(__file__)] + argv, stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
    lines, deadline = [], time.time() + timeout_s

    def reader():
        for ln in proc.stdout:
            if ln.startswith("{"):
                lines.append(json.loads(ln))
                if on_line:
                    on_line(lines[-1])
    th = threading.Thread(target=reader, daemon=True)
    th.start()
    while proc.poll() is None and time.time() < deadline:
        time.sleep(0.2)
    timed_out = proc.poll() is None
    if timed_out:
        proc.kill()
        proc.wait()
    th.join(timeout=5)
    return lines, timed_out


def cpu_reference_leg(path, preset, n_decode, budget_s, want_prefill=True, warmup=2):
    """Times the unmodified reference (oracle/_ref) on the host cores: a bounded sample of the same workload. Everything that
    touches the reference library runs in child processes under hard timeouts; the whole leg is bounded by ~2 x budget_s +
    two model loads."""
    cores = available_cpus()
    candidates = reference_thread_candidates()
    size_gb = os.path.getsize(path) / 1e9
    load_allow = 20.0 + 12.0 * size_gb                      # page-cache read + ggml allocation of the file
    probes = []
    if len(candidates) > 1:
        last = {"t": time.time()}
        lines, timed_out = _run_child(["--impl", "reference", "--ref-child", "probe", "--ref-threads", ",".join(map(str, candidates)), "--workload-path", path],
                                      load_allow + 30.0 * len(candidates), on_line=lambda _l: last.update(t=time.time()))
        probes = [l for l in lines if "threads" in l]
        for pr in probes:
            log("reference probe: %d threads -> %.1f ms/token" % (pr["threads"], pr["ms"]))
        if timed_out:
            log("reference probe: child killed after its timeout; candidates seen: %s" % [p["threads"] for p in probes])
    threads = min(probes, key=lambda p: p["ms"])["threads"] if probes else candidates[0]
    lines, timed_out = _run_child(["--impl", "reference", "--ref-child", "full", "--ref-threads", str(threads), "--workload-path", path, "--steps", str(n_decode),
                                   "--warmup", str(warmup), "--cpu-budget-s", str(budget_s)] + ([] if want_prefill else ["--no-prefill"]),
                                  load_allow + 5.0 * budget_s + 60.0)
    full = [l for l in lines if "decode_tokens_per_s" in l]
    if not full:
        raise RuntimeError("reference child produced no result (timed out: %s)" % timed_out)
    out = full[-1]
    out.update({"cores": cores, "physical_cores": physical_cores(), "candidates": candidates, "probes": probes})
    return out


def available_cpus():
    """CPUs this process may actually run on: affinity mask, capped by the cgroup quota (a container often sees every
    core of the host in os.cpu_count() while being limited to a few)."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()
        if quota != "max":
            n = max(1, min(n, int(float(quota) / float(period))))
    except (OSError, ValueError):
        pass
    return n


def log(msg):
    print("[bench %6.1fs] %s" % (time.time() - _T0, msg), file=sys.stderr, flush=True)


_T0 = time.time()


def cpu_model_name():
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name"):
                return line.split(":", 1)[1].strip()
    except OSError:
        pass
    return "unknown"


# ------------------------------------------------------------------------------------------------
def dtype_label(workload):
    fmt = workload.split(":")[1]
    return {"Q4_0": "q4_0 weights x q8_0 activations (int8 dot, fp32 accumulate); fp16 head", "Q4_1": "q4_1 weights x q8_1 activations (int8 dot, fp32 accumulate); fp16 head",
            "Q5_0": "q5_0 weights x q8_0 activations (int8 dot, fp32 accumulate); fp16 head", "Q5_1": "q5_1 weights x q8_1 activations (int8 dot, fp32 accumulate); fp16 head",
            "Q8_0": "q8_0 weights x q8_0 activations (int8 dot, fp32 accumulate); fp16 head", "FP16": "f16 weights x f16-rounded activations, fp32 accumulate",
            "FP32": "f32"}.get(fmt, fmt)


def workload_label(args, preset):
    what = "single-token rwkv_eval with logits" if args.mode == "decode" else "%d-token rwkv_eval_sequence_in_chunks chunk with logits" % PREFILL_TOKENS
    return f"{args.workload} {what} ({preset['L']} layers, n_embed {preset['C']}, ffn {preset['F']}, vocab {preset['V']})"


def run_reference(args, rank, world):
    if args.ref_child:                          # child process of cpu_reference_leg
        ths = [int(t) for t in args.ref_threads.split(",")]
        if args.ref_child == "probe":
            ref_child_probe(args.workload_path, ths)
        else:
            ref_child_full(args.workload_path, ths[0], args.steps, args.warmup, args.cpu_budget_s, not args.no_prefill)
        return
    if rank != 0:
        return
    path, preset = workload_file(args.workload)
    r = cpu_reference_leg(path, preset, n_decode=args.steps, budget_s=max(args.cpu_budget_s, 5.0), warmup=args.warmup)
    prefill = args.mode == "prefill"
    if prefill and "prefill_tokens_per_s" not in r:
        emit({"impl": "reference", "unavailable": "the 128-token chunk did not fit the CPU budget"})
        return
    value = r["prefill_tokens_per_s"] if prefill else r["decode_tokens_per_s"]
    sample = (r["prefill_sample"] if prefill else f"{r['decode_sample_tokens']} rwkv_eval calls (mean) after {r['warmup']} warm-up calls")
    line = {
        "impl": "reference", "metric": "prefill_tokens_per_sec" if prefill else "decode_tokens_per_sec", "value": value, "unit": "tokens/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "steps_timed": 1 if prefill else r["decode_sample_tokens"],
        "ms_per_step": r["prefill_ms_per_chunk"] if prefill else r["decode_ms_per_token"], "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": dtype_label(args.workload), "data": "synthetic",
        "config": {"workload": workload_label(args, preset), "parallelism": "reference CPU path (oracle/_ref), %d threads" % r["threads"], "cpu": cpu_model_name()},
        "cpu_baseline": {"value": value, "unit": "tokens/s", "cores": r["threads"], "kind": "reference",
                         "sample": f"{sample}, {r['library']}, {r['threads']} threads (candidates {r['candidates']}; {r['cores']} usable logical CPUs, {r['physical_cores']} physical cores)"},
        "e2e": {"value": value, "unit": "tokens/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "prefill": {"tokens_per_s": r.get("prefill_tokens_per_s"), "chunk": PREFILL_TOKENS},
        "decode": {"tokens_per_s": r["decode_tokens_per_s"], "ms_median": r["decode_ms_median"]},
        "gpu_launches": 0,
    }
    emit(line)


def run_ours(args, rank, world, dist):
    import __graft_entry__
    import synthetic_model as sm
    pkg = __graft_entry__.load_package()
    lib = pkg.load_rwkv_shared_library()
    L = lib.library
    barrier = (lambda: dist.barrier()) if dist else None
    path, preset = workload_file(args.workload, rank, world, barrier)
    log("workload file ready: %s" % path)
    local = int(os.environ.get("LOCAL_RANK", rank))
    t0 = time.time()
    ctx = lib.rwkv_b200_init_from_file_ex(path, local, 0, -1)   # N > 1 replicas: one full model per GPU
    load_s = time.time() - t0
    log("loaded %s in %.1fs" % (path, load_s))
    n_state, n_vocab = lib.rwkv_get_state_len(ctx), lib.rwkv_get_logits_len(ctx)
    prefill_mode = args.mode == "prefill"
    K, W = args.steps, max(args.warmup, 3)
    P = K if prefill_mode else args.prefill_steps
    toks = sm.synthetic_tokens(max(K + W + 8, (P + W + 3) * PREFILL_TOKENS), n_vocab)
    tok_arr = (ctypes.c_uint32 * len(toks))(*toks)
    sampler = ClockSampler(local)
    sampler.start()
    windows = []

    def sync_all():
        L.rwkv_b200_synchronize(ctx.ptr)
        if dist:
            dist.barrier()

    def max_over_ranks(*vals):
        if not dist:
            return vals if len(vals) > 1 else vals[0]
        import torch
        t = torch.tensor(list(vals), device=f"cuda:{local}", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        out = [float(v) for v in t]
        return out if len(out) > 1 else out[0]

    # ---- decode, state resident in HBM, CUDA events on the library's stream -------------------------------
    KD = K if not prefill_mode else 32
    L.rwkv_b200_state_load(ctx.ptr, None)
    L.rwkv_b200_eval_resident(ctx.ptr, tok_arr, 1, True, None)   # lazy allocations; graph capture happens in warm-up
    sync_all()
    launches0 = L.rwkv_b200_kernel_launch_count()
    w0 = time.time()
    ms = L.rwkv_b200_time_resident(ctx.ptr, tok_arr, 1, KD, W, True)
    windows.append((w0, time.time()))
    decode_launches = (L.rwkv_b200_kernel_launch_count() - launches0) * KD // (KD + W)
    assert ms > 0, "device timing failed"
    if args.dump_outputs and not prefill_mode:
        dump_outputs(L, ctx, n_state, n_vocab, args.dump_outputs)
    ms_max = max_over_ranks(ms)
    decode_tps = world * KD / (ms_max / 1e3)
    step_ms = ms_max / KD
    overlap_groups = int(L.rwkv_b200_overlap_groups(ctx.ptr))
    log("decode resident: %.3f ms/token (CUDA graph of per-launch kernels)" % step_ms)
    if args.quick:
        tl = kernel_timeline(L, ctx, tok_arr, 1)
        bytes_tok = int(L.rwkv_b200_bytes_per_token(ctx.ptr, True))
        sampler.stop()
        if rank == 0:
            emit({"quick": True, "workload": args.workload, "ms_per_token": step_ms, "tokens_per_s": decode_tps, "gpu_launches": int(decode_launches),
                  "whole_step_frac": bytes_tok / (step_ms * 1e-3) / 1e9 / measured_peaks()[0], "traced_us": tl["span_us"],
                  "attributed_us": {k: round(v, 1) for k, v in tl["attributed_us"].items()}, "launches": tl["launches"],
                  "env": {k: v for k, v in os.environ.items() if k.startswith("RWKV_B200_") and k != "RWKV_B200_BENCH_DIR"}})
        lib.rwkv_free(ctx)
        return

    # ---- decode end to end through rwkv_eval with HOST buffers: pinned (a serving process) and pageable (what the reference's
    # ---- Python binding hands over, rwkv_cpp_model.py:330-351) ----------------------------------------------------
    e2e = {}
    for kind in ("pinned", "pageable"):
        sbuf, lbuf, sp, lp, got = host_buffers(n_state, n_vocab, kind)
        lib.rwkv_init_state(ctx, sp)
        for t in toks[:W]:
            lib.rwkv_eval(ctx, t, sp, sp, lp)
        sync_all()
        w0 = time.time()
        t0 = time.perf_counter()
        for t in toks[W:W + KD]:
            lib.rwkv_eval(ctx, t, sp, sp, lp)
        dt = time.perf_counter() - t0
        windows.append((w0, time.time()))
        dt = max_over_ranks(dt)
        e2e[kind] = {"tokens_per_s": world * KD / dt, "ms_per_step": dt / KD * 1e3, "buffers": got}
        log("decode e2e (%s host buffers): %.3f ms/token" % (got, dt / KD * 1e3))
    sbuf, lbuf, sp, lp, kind = host_buffers(n_state, n_vocab, "pinned")

    # ---- prefill: 128-token chunk ----------------------------------------------------------------------------------
    L.rwkv_b200_state_load(ctx.ptr, None)
    launches0 = L.rwkv_b200_kernel_launch_count()
    w0 = time.time()
    pms = L.rwkv_b200_time_resident(ctx.ptr, tok_arr, PREFILL_TOKENS, P, W if prefill_mode else 2, True)
    windows.append((w0, time.time()))
    if args.dump_outputs and prefill_mode:
        dump_outputs(L, ctx, n_state, n_vocab, args.dump_outputs)
    prefill_launches = (L.rwkv_b200_kernel_launch_count() - launches0) * P // (P + (W if prefill_mode else 2))
    arr128 = (ctypes.c_uint32 * PREFILL_TOKENS)(*toks[:PREFILL_TOKENS])
    reps = P if prefill_mode else max(2, P // 2)
    for _ in range(W if prefill_mode else 1):
        L.rwkv_eval_sequence_in_chunks(ctx.ptr, arr128, PREFILL_TOKENS, PREFILL_TOKENS, None, ctypes.cast(sp, PF), ctypes.cast(lp, PF))
    w0 = time.time()
    t0 = time.perf_counter()
    for _ in range(reps):
        L.rwkv_eval_sequence_in_chunks(ctx.ptr, arr128, PREFILL_TOKENS, PREFILL_TOKENS, None, ctypes.cast(sp, PF), ctypes.cast(lp, PF))
    pe2e_s = (time.perf_counter() - t0) / reps
    windows.append((w0, time.time()))
    pms, pe2e_s = max_over_ranks(pms, pe2e_s)
    chunk_ms = pms / P
    log("prefill: %.3f ms/chunk resident, %.3f ms/chunk e2e" % (chunk_ms, pe2e_s * 1e3))

    # ---- roofline legs: the dominant kernel's share of a step from the in-kernel %globaltimer timeline (works inside CUDA-graph
    # ---- replays; per-launch CUDA events would serialise what programmatic dependent launch overlaps) ------------------
    tl = kernel_timeline(L, ctx, tok_arr, 1)
    gemv_share = tl["attributed_us"].get("gemv", 0.0) / tl["span_us"] if tl["span_us"] else 0.0
    tlp = kernel_timeline(L, ctx, tok_arr, PREFILL_TOKENS, passes=3, skip=1)
    gemm_share = tlp["attributed_us"].get("gemm_tc", 0.0) / tlp["span_us"] if tlp["span_us"] else 0.0
    gemv_bytes = int(L.rwkv_b200_gemv_bytes_per_token(ctx.ptr, True))
    bytes_tok = int(L.rwkv_b200_bytes_per_token(ctx.ptr, True))
    peak, peak_src = measured_peaks()
    tpeak, tpeak_src = measured_tensor_peak()
    gemv_ms = gemv_share * step_ms
    flops = prefill_matmul_flops(preset, PREFILL_TOKENS)
    sampler.stop()
    clocks = sampler.summary(windows)
    log("roofline legs done: decode traced %.1f us (gemv share %.3f), chunk traced %.1f us (gemm_tc share %.3f)" % (tl["span_us"], gemv_share, tlp["span_us"], gemm_share))

    line = None
    if rank == 0:
        decode_roofline = {
            "bound": "hbm", "kernel": "gemv_tma_kernel (fused dequantize-GEMV, all launches of one decode step)",
            "achieved": gemv_bytes / (gemv_ms * 1e-3) / 1e9 if gemv_ms else None, "peak": peak, "unit": "GB/s",
            "frac": gemv_bytes / (gemv_ms * 1e-3) / 1e9 / peak if gemv_ms else None, "peak_source": peak_src,
            "traffic": ncu_traffic(preset)[0] if "rwkv6-7b:Q5_1" == args.workload else None,
            "traffic_launch": ncu_traffic(preset)[1] if "rwkv6-7b:Q5_1" == args.workload else None,
            "bytes_per_step": gemv_bytes, "ms_per_step": gemv_ms, "share_of_step": gemv_share,
            "method": "critical-path attribution of the %globaltimer timeline of a graph-replayed step x the CUDA-event step time",
            "launches_per_step": tl["launches"], "attributed_us": {k: round(v, 2) for k, v in tl["attributed_us"].items()},
            "whole_step": {"bytes": bytes_tok, "ms": step_ms, "gbs": bytes_tok / (step_ms * 1e-3) / 1e9, "frac": bytes_tok / (step_ms * 1e-3) / 1e9 / peak}}
        gemm_ms = gemm_share * chunk_ms
        prefill_roofline = {
            "bound": "tensor", "kernel": "gemm_tc_kernel (tcgen05 + TMEM, all launches of one 128-token chunk)",
            "achieved": flops / (gemm_ms * 1e-3) / 1e12 if gemm_ms else None, "peak": tpeak, "unit": "TFLOP/s",
            "frac": flops / (gemm_ms * 1e-3) / 1e12 / tpeak if gemm_ms else None, "peak_source": tpeak_src, "traffic": None,
            "flops_per_step": flops, "ms_per_step": gemm_ms, "share_of_step": gemm_share,
            "launches_per_step": tlp["launches"], "attributed_us": {k: round(v, 2) for k, v in tlp["attributed_us"].items()},
            "whole_step": {"flops": flops, "ms": chunk_ms, "tflops": flops / (chunk_ms * 1e-3) / 1e12, "frac": flops / (chunk_ms * 1e-3) / 1e12 / tpeak}}
        prefill_obj = {"tokens_per_s": world * PREFILL_TOKENS / (chunk_ms / 1e3), "ms_per_chunk": chunk_ms, "chunk": PREFILL_TOKENS, "steps": P,
                       "e2e_tokens_per_s": world * PREFILL_TOKENS / pe2e_s, "gpu_launches": int(prefill_launches)}
        decode_obj = {"tokens_per_s": decode_tps, "ms_per_token": step_ms, "steps": KD, "e2e_tokens_per_s": e2e["pinned"]["tokens_per_s"],
                      "e2e_pageable_tokens_per_s": e2e["pageable"]["tokens_per_s"], "gpu_launches": int(decode_launches)}
        state_copies = ("pipelined against %d layer groups on copy streams" % overlap_groups) if overlap_groups else "one upload before, one download after the pass"
        common = {"n_gpus": world, "steps": K, "warmup": W, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": dtype_label(args.workload), "data": "synthetic",
                  "config": {"workload": workload_label(args, preset),
                             "parallelism": "1 GPU" if world == 1 else f"{world} independent replicas (single-stream decode does not shard; DESIGN.md)",
                             "l2": "%.2f GB of weights per step >> 126 MB L2, no flush needed" % (bytes_tok / 1e9) if bytes_tok > 4 * 126e6 else
                                   "%.0f MB of weights per step: fits L2, steps run back to back WITHOUT a flush (stated, launch-bound config)" % (bytes_tok / 1e6),
                             "bytes_per_token": bytes_tok, "load_s": round(load_s, 2), "cuda_graph": True},
                  "clocks": clocks, "prefill": prefill_obj, "decode": decode_obj}
        if prefill_mode:
            line = dict(common, metric="prefill_tokens_per_sec", value=prefill_obj["tokens_per_s"], unit="tokens/s", ms_per_step=chunk_ms,
                        e2e={"value": prefill_obj["e2e_tokens_per_s"], "unit": "tokens/s", "h2d_bytes_per_step": 4 * PREFILL_TOKENS, "d2h_bytes_per_step": n_state * 4 + n_vocab * 4,
                             "host_buffers": "pinned", "ms_per_step": pe2e_s * 1e3, "state_copies": state_copies},
                        gpu_launches=int(prefill_launches), roofline=dict(prefill_roofline, decode=decode_roofline))
        else:
            line = dict(common, metric="decode_tokens_per_sec", value=decode_tps, unit="tokens/s", ms_per_step=step_ms,
                        e2e={"value": e2e["pinned"]["tokens_per_s"], "unit": "tokens/s", "h2d_bytes_per_step": n_state * 4 + 4, "d2h_bytes_per_step": n_state * 4 + n_vocab * 4,
                             "host_buffers": "pinned", "ms_per_step": e2e["pinned"]["ms_per_step"], "state_copies": state_copies,
                             "pageable": {"value": e2e["pageable"]["tokens_per_s"], "ms_per_step": e2e["pageable"]["ms_per_step"], "buffers": e2e["pageable"]["buffers"]},
                             "prefill_tokens_per_s": prefill_obj["e2e_tokens_per_s"]},
                        gpu_launches=int(decode_launches), roofline=dict(decode_roofline, prefill=prefill_roofline))
    lib.rwkv_free(ctx)
    if rank == 0:
        if world == 1 and not args.skip_cpu_baseline:
            log("cpu baseline (reference library in child processes)")
            try:
                r = cpu_reference_leg(path, preset, n_decode=32, budget_s=args.cpu_budget_s, want_prefill=True, warmup=2)
                v = r.get("prefill_tokens_per_s") if prefill_mode else r["decode_tokens_per_s"]
                line["cpu_baseline"] = {"value": v, "unit": "tokens/s", "cores": r["threads"], "kind": "reference",
                                        "sample": f"{r['decode_sample_tokens']} rwkv_eval calls (mean) + {r.get('prefill_sample', 'no prefill chunk')}, {r['library']}, "
                                                  f"{r['threads']} threads (candidates {r['candidates']}; {r['cores']} usable logical CPUs, {r['physical_cores']} physical cores)",
                                        "decode_tokens_per_s": r["decode_tokens_per_s"], "prefill_tokens_per_s": r.get("prefill_tokens_per_s"), "cpu": cpu_model_name()}
            except Exception as e:   # the baseline is reported, never required for the GPU number
                line["cpu_baseline"] = {"value": None, "unit": "tokens/s", "cores": 0, "kind": "reference", "sample": "failed: %r" % (e,)}
        emit(line)


def run_pipeline(args, rank, world, dist):
    """N > 1: layer pipeline (SURVEY.md 8e). Rank g holds a contiguous block of layers (balanced by BYTES: the last stage also
    streams the head) and their slice of the recurrent state; `world` sequences are in flight, one per stage. The hand-off is
    inside the library (csrc/kernels/pipe.cu): x f32[C x T] goes into the next GPU's mailbox with NVLink peer stores from the last
    kernel of the stage's pass, flags + device-side item counters order it -- NCCL only carries the 64-byte IPC handles at set-up
    and the barriers / reductions of the measurement. One step = one token of every in-flight sequence (`world` tokens)."""
    import torch
    import __graft_entry__
    import synthetic_model as sm
    pkg = __graft_entry__.load_package()
    pipeline = pkg.pipeline
    lib = pkg.load_rwkv_shared_library()
    L = lib.library
    path, preset = workload_file(args.workload, rank, world, lambda: dist.barrier())
    local = int(os.environ.get("LOCAL_RANK", rank))
    info = lib.rwkv_b200_inspect_file(path)
    head_bytes = preset["C"] * preset["V"] * (4 if args.workload.endswith("FP32") else 2)
    layer_bytes = (info.bytes_per_token - head_bytes - 8 * info.state_len) / preset["L"]
    begin, end = pipeline.stage_layers_balanced(preset["L"], world, rank, head_layers=head_bytes / layer_bytes)
    t0 = time.time()
    ctxs = [lib.rwkv_b200_init_from_file_ex(path, local, begin, end)]
    for _ in range(world - 1):
        ctxs.append(lib.rwkv_clone_context(ctxs[0], 1))          # one context = one in-flight sequence's state slice
    load_s = time.time() - t0
    log("rank %d: layers [%d, %d) loaded in %.1fs" % (rank, begin, end, load_s))
    n_vocab = lib.rwkv_get_logits_len(ctxs[0])
    first, last = rank == 0, rank == world - 1
    # ---- connect the stages: 64-byte CUDA IPC handles of the mailboxes, all_gathered once. Should a box refuse CUDA IPC / peer
    # access between its GPUs (or RWKV_B200_PIPE_TRANSPORT=nccl ask for it), every rank falls back to the round-1 transport: the
    # stage API (rwkv_b200_stage_eval) with x handed on by NCCL send / recv on the stage's stream. The line says which one ran.
    transport = os.environ.get("RWKV_B200_PIPE_TRANSPORT", "peer")
    if transport == "peer":
        ok = 1
        try:
            hsz = int(L.rwkv_b200_pipe_handle_size())
            hbuf = ctypes.create_string_buffer(hsz)
            ok = 1 if L.rwkv_b200_pipe_export(ctxs[0].ptr, hbuf) else 0
            mine = torch.frombuffer(bytearray(hbuf.raw), dtype=torch.uint8).to(f"cuda:{local}")
            gathered = [torch.empty_like(mine) for _ in range(world)]
            dist.all_gather(gathered, mine)
            handles = [bytes(g.cpu().numpy().tobytes()) for g in gathered]
            if ok and not L.rwkv_b200_pipe_connect(ctxs[0].ptr, None if first else handles[rank - 1], None if last else handles[rank + 1]):
                ok = 0
        except Exception as exc:      # noqa: BLE001 -- any failure of the set-up means "use the fallback", on every rank
            log("rank %d: peer-memory set-up failed: %r" % (rank, exc))
            ok = 0
        flag = torch.tensor([ok], device=f"cuda:{local}", dtype=torch.int32)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        if int(flag.item()) == 0:
            log("rank %d: peer-memory mailboxes unavailable on this box -> NCCL send/recv transport" % rank)
            transport = "nccl"
    dist.barrier()
    for c in ctxs:
        L.rwkv_b200_state_load(c.ptr, None)
        L.rwkv_b200_synchronize(c.ptr)
    K, W, P = args.steps, max(args.warmup, 3), args.prefill_steps
    # one stream per stage: a link's hand-offs are enqueued in item order (the legacy default stream has handle 0, which
    # rwkv_b200_pipe_eval reads as "use the context's own stream")
    stream = torch.cuda.Stream(device=local)
    torch.cuda.set_stream(stream)
    sp = ctypes.c_void_p(stream.cuda_stream)
    assert stream.cuda_stream != 0
    sampler = ClockSampler(local)
    sampler.start()
    windows = []
    logits_host = torch.zeros(n_vocab, dtype=torch.float32).pin_memory()
    bytes_tok = int(L.rwkv_b200_bytes_per_token(ctxs[0].ptr, True))   # this stage's share of the byte model
    kept = {}

    def leg(T, steps, warm, read_logits, n_seq=world, keep=None):
        """`steps` timed steps of `n_seq` work items each (one per in-flight sequence), after `warm` untimed ones. Every rank simply
        enqueues its stage for every item in order; the flags in the mailboxes make a stage wait for its neighbour ON THE DEVICE."""
        n_items = (steps + warm) * n_seq
        toks = sm.synthetic_tokens(n_items * T + T, n_vocab)
        arr = (ctypes.c_uint32 * len(toks))(*toks)

        n_hidden = int(L.rwkv_b200_stage_hidden_len(ctxs[0].ptr, T))
        hin = torch.empty(n_hidden, dtype=torch.float32, device=f"cuda:{local}") if transport == "nccl" and not first else None
        hout = torch.empty(n_hidden, dtype=torch.float32, device=f"cuda:{local}") if transport == "nccl" and not last else None

        def run(u0, u1):
            for u in range(u0, u1):
                seq = u % n_seq
                tok_p = ctypes.cast(ctypes.byref(arr, 4 * u * T), PU) if first else None
                if transport == "peer":
                    ok = L.rwkv_b200_pipe_eval(ctxs[seq].ptr, tok_p, T, True, sp)
                else:       # every rank walks the items in the same order, so sends and receives pair up; all of it is stream-ordered
                    if hin is not None:
                        dist.recv(hin, src=rank - 1)
                    ok = L.rwkv_b200_stage_eval(ctxs[seq].ptr, tok_p, T, ctypes.c_void_p(hin.data_ptr()) if hin is not None else None,
                                                ctypes.c_void_p(hout.data_ptr()) if hout is not None else None, True, sp)
                    if hout is not None:
                        dist.send(hout, dst=rank + 1)
                assert ok, "pipeline stage evaluation failed"
                if read_logits and last:
                    assert L.rwkv_b200_stage_logits(ctxs[seq].ptr, ctypes.cast(logits_host.data_ptr(), PF), sp)
                    if keep is not None and seq == 0 and len(keep) < 4:
                        keep.append((list(toks[u * T:(u + 1) * T]), logits_host.numpy().copy()))

        run(0, warm * n_seq)
        torch.cuda.synchronize(); dist.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        launches0 = L.rwkv_b200_kernel_launch_count()
        w0 = time.time(); t0 = time.perf_counter()
        e0.record(stream)
        run(warm * n_seq, n_items)
        e1.record(stream)
        torch.cuda.synchronize()
        wall = time.perf_counter() - t0
        dist.barrier()
        windows.append((w0, time.time()))
        t = torch.tensor([e0.elapsed_time(e1), wall * 1e3, float(L.rwkv_b200_kernel_launch_count() - launches0)], device=f"cuda:{local}")
        mx = t.clone(); dist.all_reduce(mx, op=dist.ReduceOp.MAX)
        sm_ = t.clone(); dist.all_reduce(sm_, op=dist.ReduceOp.SUM)
        return float(mx[0]), float(mx[1]), float(sm_[2])

    def reset_states():
        for c in ctxs:
            L.rwkv_b200_state_load(c.ptr, None)
            L.rwkv_b200_synchronize(c.ptr)
        dist.barrier()

    # ---- correctness inside the bench: the pipeline's logits of sequence 0 vs the same tokens on ONE GPU (last rank loads the whole model)
    check = []
    leg(1, 4, 0, True, keep=check)
    check_out = None
    if last:
        whole = lib.rwkv_b200_init_from_file_ex(path, local, 0, -1)
        lg = np.zeros(n_vocab, np.float32)
        L.rwkv_b200_state_load(whole.ptr, None)
        worst, same = 0.0, True
        for toks_u, got in check:
            arr1 = (ctypes.c_uint32 * 1)(*toks_u)
            assert L.rwkv_b200_eval_resident(whole.ptr, arr1, 1, True, lg.ctypes.data_as(PF))
            worst = max(worst, float(np.abs(lg - got).max()))
            same = same and lg.tobytes() == got.tobytes()
        lib.rwkv_free(whole)
        check_out = {"tokens": len(check), "max_abs_diff_vs_single_gpu": worst, "bitwise_equal": same}
        log("pipeline check: %s" % check_out)
    reset_states()
    dev_ms, _, launches = leg(1, K, W, False)                         # decode, logits stay on the last stage's GPU
    log("pipeline decode: %.3f ms per step of %d tokens" % (dev_ms / K, world))
    _, e2e_ms, _ = leg(1, K, W, True)                                 # + token H2D on stage 0, logits D2H on the last stage, per token
    lat_ms, _, _ = leg(1, max(8, K // 2), 2, False, n_seq=1)          # ONE sequence through all stages: the single-stream latency
    lat_steps = max(8, K // 2)
    pdev_ms, _, _ = leg(PREFILL_TOKENS, P, 2, False)
    _, pe2e_ms, _ = leg(PREFILL_TOKENS, P, 1, True)
    sampler.stop()
    clocks = sampler.summary(windows)
    stage_bytes = torch.tensor([float(bytes_tok)], device=f"cuda:{local}")
    dist.all_reduce(stage_bytes, op=dist.ReduceOp.MAX)
    chk = [check_out]
    dist.broadcast_object_list(chk, src=world - 1)
    for c in ctxs[1:]:
        lib.rwkv_free(c)
    lib.rwkv_free(ctxs[0])
    if rank == 0:
        peak, peak_src = measured_peaks()
        tick_ms = dev_ms / (K * world)                                      # one token leaves the pipeline per tick
        gbs = float(stage_bytes.item()) / (tick_ms * 1e-3) / 1e9
        blocks = [pipeline.stage_layers_balanced(preset["L"], world, r, head_layers=head_bytes / layer_bytes) for r in range(world)]
        line = {
            "metric": "decode_tokens_per_sec", "value": world * K / (dev_ms / 1e3), "unit": "tokens/s", "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": dev_ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": dtype_label(args.workload), "data": "synthetic",
            "config": {"workload": workload_label(args, preset),
                       "parallelism": f"pp{world}: layer blocks {blocks} balanced by bytes (head = {head_bytes / layer_bytes:.1f} layers) + their state slice per GPU, "
                                      f"{world} sequences in flight (one per stage), x f32[{preset['C']}] per token by "
                                      + ("NVLink peer stores + flags inside the library (csrc/kernels/pipe.cu)" if transport == "peer" else "NCCL send/recv on the stage's stream (fallback transport)")
                                      + f"; one step = {world} tokens",
                       "transport": transport,
                       "l2": "each stage streams its share of the weights per token >> 126 MB L2, no flush needed", "load_s": round(load_s, 2), "cuda_graph": True},
            "clocks": clocks,
            "e2e": {"value": world * K / (e2e_ms / 1e3), "unit": "tokens/s", "h2d_bytes_per_step": 4 * world, "d2h_bytes_per_step": 4 * n_vocab * world,
                    "host_buffers": "pinned", "ms_per_step": e2e_ms / K,
                    "note": "token ids enter on stage 0, logits leave from the last stage; the recurrent state stays resident on its stage"},
            "gpu_launches": int(launches),
            "single_stream": {"ms_per_token": dev_ms / K, "tokens_per_s": K / (dev_ms / 1e3),
                              "note": "latency of ONE sampled stream (the next token comes out of the logits): a token crosses all `world` stages, i.e. "
                                      "`world` ticks = one step of the loaded pipeline (layer i+1 needs layer i: a pipeline cannot speed a single stream up)",
                              "teacher_forced_ms_per_token": lat_ms / lat_steps,
                              "teacher_forced_note": "ONE sequence whose tokens are known in advance (prompt ingestion token by token): stage 0 already works on "
                                                     "token u+1 while the last stage finishes token u"},
            "pipeline_check": chk[0],
            "prefill": {"tokens_per_s": world * P * PREFILL_TOKENS / (pdev_ms / 1e3), "ms_per_chunk": pdev_ms / (P * world), "chunk": PREFILL_TOKENS, "steps": P,
                        "e2e_tokens_per_s": world * P * PREFILL_TOKENS / (pe2e_ms / 1e3)},
            "roofline": {"bound": "hbm", "kernel": "whole pipeline tick of the slowest stage (fused dequant-GEMV launches + glue)",
                         "achieved": gbs, "peak": peak, "unit": "GB/s", "frac": gbs / peak, "peak_source": peak_src, "traffic": None,
                         "bytes_per_step": float(stage_bytes.item()), "ms_per_step": tick_ms,
                         "note": "per GPU: the largest stage's bytes per token / time per pipeline tick; per-launch figures are in the N=1 line"},
            "cpu_baseline": {"value": None, "unit": "tokens/s", "cores": 0, "kind": "reference", "sample": "reported by the N=1 run and by --impl reference"},
        }
        emit(line)


_REAL_STDOUT = None


def emit(line):
    """The ONE JSON line goes to the process's real stdout; everything libraries print (NCCL's version banner ...) goes to stderr."""
    out = _REAL_STDOUT if _REAL_STDOUT is not None else sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


def main():
    global _REAL_STDOUT
    _REAL_STDOUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    args = parse_args()
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    dist = None
    if args.dump_outputs and (args.impl != "ours" or world > 1):
        raise SystemExit("--dump-outputs writes the outputs of this library's one-process run (--impl ours, one GPU)")
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if world > 1:
        import torch
        import torch.distributed as dist_mod
        torch.cuda.set_device(int(os.environ.get("LOCAL_RANK", rank)))
        dist_mod.init_process_group("nccl")
        dist = dist_mod
    if world > 1:
        run_pipeline(args, rank, world, dist)
    else:
        run_ours(args, rank, world, dist)
    if dist:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
