#!/usr/bin/env python
"""bench.py -- decode tokens/s of the layer-sliced LLaMA forward on B200 (BASELINE.json's metric).

A "step" is one pass of the hot path over one batch of synthetic input: ONE token (batch 1)
propagated through every layer of the model's slice(s) with the KV cache at position p, p cycling
through [256, 512) (seq_len 512) after a 256-token prefill.  Workload = BASELINE.json configs[1]
(LLaMA-7B Q4_0, 1 slice on 1xB200) at N=1; at N>1 the same 32 layers are cut into N contiguous
slices, one rank per GPU, and the activation is handed from rank r to r+1 by one NCCL send/recv
(configs[2] at N=4).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--dump-outputs DIR]     # this framework
    python bench.py --impl reference [...]                          # the reference's CPU path

Prints ONE JSON line (rank 0).  `value` = tokens/s with the activation resident in HBM;
`e2e` = the same metric through the reference-facing C ABI call b200_slice_forward() with HOST
buffers (H2D + D2H inside the timed region); `roofline` = achieved HBM GB/s of the weight-matmul
kernel vs the measured peak; `cpu_baseline` = the reference CPU path timed on this box's cores.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

from distributedllm_b200 import ggjt  # noqa: E402
from distributedllm_b200.pipeline import layer_ranges  # noqa: E402

METRIC = "decode tokens/sec LLaMA-7B Q4_0 seq512 bs1"
UNIT = "tokens/s"
N_CTX = 512
PREFILL = 256
SEED = 0
FALLBACK_HBM_GBS = 6650.0
NCU_CAPTURE = os.path.join(ROOT, "profiles", "r02_decode_kernels_ncu_full.md")


def ncu_traffic_per_launch():
    """dram__bytes_read.sum + dram__bytes_write.sum per k_gemv launch, averaged over the launches of the committed
    `ncu --set full` capture of a decode step (profiles/r02_decode_kernels_ncu_full.md, produced by scripts/summarize_ncu.py
    from the .ncu-rep): parsed here, not a constant.  Returns (read + write bytes, read bytes, launches) or (None, None, 0)."""
    try:
        rd = wr = n = 0
        cols = None
        for line in open(NCU_CAPTURE):
            f = [x.strip() for x in line.strip().strip("|").split("|")]
            if "dram_rd_MB" in f:
                cols = {name: i for i, name in enumerate(f)}
            elif cols and f and f[0].startswith("void k_gemv<"):
                rd += float(f[cols["dram_rd_MB"]]) * 1e6
                wr += float(f[cols["dram_wr_MB"]]) * 1e6
                n += 1
        return ((rd + wr) / n, rd / n, n) if n else (None, None, 0)
    except Exception:
        return None, None, 0


def model_dir() -> str:
    d = os.environ.get("B200_BENCH_DIR") or os.path.join(tempfile.gettempdir(), "b200_bench_models")
    os.makedirs(d, exist_ok=True)
    return d


def slice_file(shape_name: str, a: int, b: int) -> str:
    """Synthetic Q4_0 slice file for layers [a, b] (written once per box, deterministic)."""
    p = os.path.join(model_dir(), "%s_q4_0_s%d_layers_%d_%d.bin" % (shape_name, SEED, a, b))
    sh = ggjt.SHAPES[shape_name]
    per_layer = 4 * (sh.n_embd * sh.n_embd // 32 * 18) + 3 * (sh.n_embd * sh.n_ff // 32 * 18)
    if not (os.path.isfile(p) and os.path.getsize(p) > per_layer * (b - a + 1)):
        tmp = p + ".tmp%d" % os.getpid()
        ggjt.write_fast_q4_slice(tmp, sh, a, b, SEED)
        os.replace(tmp, p)
    return p


def synth_inputs(n: int, n_embd: int, seed: int) -> np.ndarray:
    return np.random.default_rng([SEED, seed]).standard_normal((n, n_embd), dtype=np.float32)


def dump_outputs(d: str, **arrays) -> None:
    """--dump-outputs: one DIR/<name>.npy per array, float32, so that two builds run with the same arguments (hence the
    same seeded weights and inputs) can be compared output for output."""
    os.makedirs(d, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(d, name + ".npy"), np.ascontiguousarray(a, np.float32))


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return FALLBACK_HBM_GBS, "fallback (B200_PROFILING.md)"


class ClockSampler:
    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, device: int):
        self.device = device
        self.proc = None
        self.path = None

    def start(self):
        try:
            fd, self.path = tempfile.mkstemp(suffix=".csv")
            os.close(fd)
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.device), "--query-gpu=" + self.FIELDS, "--format=csv,noheader,nounits",
                 "-lms", "100"], stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self) -> dict:
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if not self.proc:
            return out
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        try:
            for line in open(self.path):
                f = [x.strip() for x in line.split(",")]
                if len(f) < 7:
                    continue
                try:
                    sm.append(float(f[0])); mx.append(float(f[1]))
                except ValueError:
                    continue
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            os.remove(self.path)
        except Exception:
            pass
        if sm:
            out.update(sm_mhz=statistics.median(sm), sm_max_mhz=max(mx), reasons=sorted(reasons), samples=len(sm))
        return out


# ------------------------------------------------------------------------------------------- reference arm
def cpu_reference_run(path: str, n_embd: int, steps: int, warmup: int, prompt: int = 16, want_outputs: bool = False):
    """Time the reference's own CPU implementation (oracle/_ref, built from /root/reference in the build
    container) on this box's host cores; falls back to the C port when oracle/_ref is absent."""
    from oracle import oracle
    try:
        avail = len(os.sched_getaffinity(0))
    except AttributeError:
        avail = os.cpu_count() or 1
    kind = "reference" if oracle.have_ref() else "port"
    cores = avail
    if kind == "reference":
        # ggml's thread pool spin-waits (ggml.c:15979-16090): past the physical core count more threads
        # make it SLOWER, so give the reference its best thread count: time 2 decode steps per candidate.
        best = None
        for nt in sorted({t for t in (3, 8, 16, 32, 64, avail) if t <= avail}):
            probe = oracle.RefSlice(path, n_threads=nt, n_ctx=N_CTX)
            xprobe = synth_inputs(3, n_embd, 9)
            probe.forward(xprobe[0:1])
            t0 = time.perf_counter()
            probe.forward(xprobe[1:2]); probe.forward(xprobe[2:3])
            dt = (time.perf_counter() - t0) / 2
            probe.close()
            if best is None or dt < best[0]:
                best = (dt, nt)
            if dt > 1.25 * best[0]:
                break               # past the optimum it only gets worse (128 threads: 20 s per token); keep the run short
        cores = best[1]
        sl = oracle.RefSlice(path, n_threads=cores, n_ctx=N_CTX)
    else:
        os.environ.setdefault("OMP_NUM_THREADS", str(cores))
        sl = oracle.PortSlice(path, N_CTX)
    steps = max(1, min(steps, N_CTX - prompt - warmup))
    x0 = synth_inputs(prompt, n_embd, 1)
    xs = synth_inputs(steps + warmup, n_embd, 2)
    outs = []
    sl.forward(x0)
    for i in range(warmup):
        outs.append(sl.forward(xs[i:i + 1]))
    t0 = time.perf_counter()
    for i in range(warmup, warmup + steps):
        outs.append(sl.forward(xs[i:i + 1]))
    dt = time.perf_counter() - t0
    sl.close()
    res = {"value": steps / dt, "unit": UNIT, "cores": cores, "kind": kind,
           "sample": "%d decode steps at positions %d..%d after a %d-token prompt, same slice file; %d threads "
                     "(fastest of 3..%d on this host; the reference ships with 3)"
                     % (steps, prompt + warmup, prompt + warmup + steps - 1, prompt, cores, avail),
           "ms_per_step": 1e3 * dt / steps, "steps": steps}
    return (res, x0, xs, outs) if want_outputs else res


def cpu_reference_chain(paths, n_embd: int, x0: np.ndarray, xq: np.ndarray):
    """The reference's own multi-node data flow on the host: the activation goes through the slice files in order
    (one reference slice loaded at a time, as one `llm` module holds one slice: tensor_processor.cpp:1992).  Returns
    (timing dict, [prompt output, step outputs...]) -- the checker for the N-GPU pipeline and its cpu_baseline."""
    from oracle import oracle
    try:
        avail = len(os.sched_getaffinity(0))
    except AttributeError:
        avail = os.cpu_count() or 1
    kind = "reference" if oracle.have_ref() else "port"
    cores = min(16, avail) if kind == "reference" else avail
    acts = [x0] + [xq[i:i + 1] for i in range(xq.shape[0])]
    dt = 0.0
    for p in paths:
        sl = oracle.RefSlice(p, n_threads=cores, n_ctx=N_CTX) if kind == "reference" else oracle.PortSlice(p, N_CTX)
        outs = [sl.forward(acts[0])]
        for a in acts[1:]:
            t0 = time.perf_counter()
            outs.append(sl.forward(a))
            dt += time.perf_counter() - t0
        sl.close()
        acts = outs
    steps = xq.shape[0]
    res = {"value": steps / dt, "unit": UNIT, "cores": cores, "kind": kind, "ms_per_step": 1e3 * dt / steps, "steps": steps,
           "sample": "%d decode steps at positions %d..%d after a %d-token prompt through the %d slice files in sequence; "
                     "%d threads" % (steps, x0.shape[0], x0.shape[0] + steps - 1, x0.shape[0], len(paths), cores)}
    return res, acts


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    sh = ggjt.SHAPES["7b"]
    path = slice_file("7b", 0, sh.n_layer - 1)
    r, _, _, outs = cpu_reference_run(path, sh.n_embd, args.steps, args.warmup, want_outputs=True)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, hidden_state=outs[-1])
    line = {"impl": "reference", "metric": METRIC, "value": r["value"], "unit": UNIT, "n_gpus": args.gpus,
            "steps": r["steps"], "warmup": args.warmup, "ms_per_step": r["ms_per_step"], "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "q4_0*q8_0->f32", "data": "synthetic",
            "config": {"workload": "LLaMA-7B Q4_0, 1 slice x 32 layers, reference CPU path (llama.cpp/ggml via "
                                   "tensor_processor.cpp), n_ctx=512, batch=1", "threads": r["cores"]},
            "cpu_baseline": {k: r[k] for k in ("value", "unit", "cores", "kind", "sample")},
            "e2e": {"value": r["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)
    return 0


# ------------------------------------------------------------------------------------------- B200 arm
def run_b200(args):
    from distributedllm_b200 import capi

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus and world > 1:
        raise SystemExit("--gpus %d but WORLD_SIZE=%d" % (args.gpus, world))
    dist = None
    if world > 1:
        import torch
        import torch.distributed as dist_
        dist = dist_
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    sh = ggjt.SHAPES["7b"]
    E = sh.n_embd
    a, b = layer_ranges(sh.n_layer, world)[rank]
    path = slice_file("7b", a, b)
    t_init = time.perf_counter()
    capi.check(capi.lib().b200_device_init(local))          # CUDA context creation (seconds on an 8-GPU box), not slice load
    cuda_init_seconds = time.perf_counter() - t_init
    t_load = time.perf_counter()
    sl = capi.Slice(path, local, N_CTX)
    load_seconds = time.perf_counter() - t_load
    K, W = args.steps, args.warmup
    cycle = N_CTX - PREFILL

    transport = None
    if world > 1:
        import torch
        from distributedllm_b200.pipeline import join_pipeline, torch_collectives
        bcast, gather = torch_collectives(dist, torch.device("cuda", local))
        transport = join_pipeline(sl, rank, world, bcast, gather, peer=os.environ.get("B200_PP_PEER", "1") != "0")

    def barrier():
        sl.sync()
        if dist is not None:
            dist.barrier()
            sl.sync()

    # ---- prefill 256 tokens (untimed), in chunks
    xp = synth_inputs(PREFILL, E, 1)
    chunk = 64
    for i in range(0, PREFILL, chunk):
        if world == 1:
            sl.forward(xp[i:i + chunk])
        else:
            import ctypes as C
            n = min(chunk, PREFILL - i)
            if rank == 0:
                _h2d(sl, xp[i:i + n])
            capi.check(capi.lib().b200_pipeline_step(sl.handle, C.c_void_p(sl.dev_in), n, 0))
    barrier()
    assert sl.n_past == PREFILL or world > 1

    xs = synth_inputs(cycle, E, 2)

    def step_device(i: int):
        p = PREFILL + (i % cycle)
        if p == PREFILL and sl.n_past != PREFILL:
            sl.rewind(PREFILL)
        if world == 1:
            sl.forward_device(sl.dev_in, 1, sl.dev_out)
        else:
            import ctypes as C
            capi.check(capi.lib().b200_pipeline_step(sl.handle, C.c_void_p(sl.dev_in), 1, 1))

    _h2d(sl, xs[0:1])
    clocks = ClockSampler(local)
    # ---- value: K device-resident steps, CUDA events on the launching stream, max over ranks
    for i in range(W):
        step_device(i)
    barrier()
    launches0 = sl.launch_count()
    if rank == 0:
        clocks.start()
    t0 = time.perf_counter()
    sl.mark(0)
    for i in range(W, W + K):
        step_device(i)
    sl.mark(1)
    barrier()
    wall_ms = 1e3 * (time.perf_counter() - t0)
    dev_ms = sl.mark_elapsed_ms()
    launches = sl.launch_count() - launches0
    if dist is not None:
        import torch
        t = torch.tensor([dev_ms, wall_ms], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dev_ms, wall_ms = float(t[0]), float(t[1])
        lt = torch.tensor([launches], dtype=torch.int64, device="cuda")
        dist.all_reduce(lt)
        launches = int(lt[0])
    value = K / (dev_ms / 1e3)
    if args.dump_outputs and rank == 0:
        # what the last timed step returned to its caller: the model's hidden state for that token (the last slice's
        # output, which the ring hands back to rank 0 at N > 1); read before the legs below reuse the buffers
        last = np.empty((1, E), np.float32)
        _d2h(sl, last)
        dump_outputs(args.dump_outputs, hidden_state=last)
    pos_timed = [PREFILL + (i % cycle) for i in range(W, W + K)]
    timed_positions = ("%d..%d" % (pos_timed[0], pos_timed[-1]) if K <= cycle - (W % cycle) else
                       "%d..%d cyclically (%d steps)" % (PREFILL, N_CTX - 1, K))

    # ---- e2e: the C ABI call with HOST buffers, one token per call (H2D + graph + D2H + sync)
    e2e = None
    if world == 1:
        sl.rewind(PREFILL)
        for i in range(W):
            sl.forward(xs[i % cycle:i % cycle + 1])
        sl.sync()
        t0 = time.perf_counter()
        for i in range(W, W + K):
            if PREFILL + (i % cycle) == PREFILL and sl.n_past != PREFILL:
                sl.rewind(PREFILL)
            sl.forward(xs[i % cycle:i % cycle + 1])
        sl.sync()
        e2e_s = time.perf_counter() - t0
        e2e = {"value": K / e2e_s, "unit": UNIT, "h2d_bytes_per_step": E * 4, "d2h_bytes_per_step": E * 4,
               "api": "b200_slice_forward(host in, 1, host out)"}
    else:
        # pipeline e2e: rank 0 uploads the token, the ring returns the last rank's output to rank 0, rank 0 reads it back
        import ctypes as C
        sl.rewind(PREFILL) if sl.n_past > PREFILL else None
        barrier()
        host_out = np.empty((1, E), np.float32)
        t0 = time.perf_counter()
        for i in range(K):
            if PREFILL + (i % cycle) == PREFILL and sl.n_past != PREFILL:
                sl.rewind(PREFILL)
            if rank == 0:
                _h2d(sl, xs[i % cycle:i % cycle + 1])
            capi.check(capi.lib().b200_pipeline_step(sl.handle, C.c_void_p(sl.dev_in), 1, 1))
            if rank == 0:
                _d2h(sl, host_out)
        barrier()
        e2e_s = time.perf_counter() - t0
        import torch
        t = torch.tensor([e2e_s], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e = {"value": K / float(t[0]), "unit": UNIT, "h2d_bytes_per_step": E * 4, "d2h_bytes_per_step": E * 4,
               "api": "b200_pipeline_step over %d ranks, rank 0 host in/out" % world}
    clk = clocks.stop() if rank == 0 else {}

    # ---- roofline of the dominant kernel (the Q4_0 weight matmul): per-launch CUDA events, live
    roof = None
    info = sl.info
    if True:
        sl.rewind(PREFILL) if sl.n_past > PREFILL else None
        sl.profile(True)
        nprof = min(32, cycle)
        for i in range(nprof):
            if world == 1:
                sl.forward_device(sl.dev_in, 1, sl.dev_out)
            else:
                sl.forward_device(sl.dev_in, 1, sl.dev_out)      # local layers only: kernel timing, no hand-off
        ms, cnt = sl.profile_read()
        sl.profile(False)
        gemv_ms = float(ms[0] + ms[3] + ms[4] + ms[5])
        gemv_launches = int(cnt[0] + cnt[3] + cnt[4] + cnt[5])
        peak, peak_src = measured_peak()
        wbytes = float(info.weight_bytes)                       # this rank's slice, bytes as stored in the file
        ev_achieved = wbytes * nprof / (gemv_ms / 1e3) / 1e9    # per-launch event brackets (adds ~4 us per launch)
        # dominant kernel alone: the step's 4 x n_layer matmul launches replayed back to back as a graph (attention
        # skipped), two CUDA events around `reps` replays on the launching stream
        sl.rewind(PREFILL) if sl.n_past > PREFILL else None
        sl.skip_attention(True)
        reps = 32
        for i in range(3):
            sl.forward_device(sl.dev_in, 1, sl.dev_out)
        sl.sync()
        sl.mark(0)
        for i in range(reps):
            sl.forward_device(sl.dev_in, 1, sl.dev_out)
        sl.mark(1)
        sl.sync()
        only_ms = sl.mark_elapsed_ms() / reps
        sl.skip_attention(False)
        sl.rewind(PREFILL)
        n_gemv = 4 * info.n_layer
        achieved = wbytes / (only_ms / 1e3) / 1e9
        # the same kernels INSIDE the replayed graph (PDL overlap and all), from in-kernel %globaltimer stamps:
        # duration of a launch = last CTA exit - first CTA entry
        in_graph = None
        try:
            sl.trace_enable(True)
            nlayer = info.n_layer
            for i in range(3):
                sl.forward_device(sl.dev_in, 1, sl.dev_out)
            stamps, cls, ctas = sl.trace_read()
            sl.trace_enable(False)
            per = 5 * nlayer
            dur = {}
            for j in range(len(cls) - per, len(cls)):
                d = stamps[j, :ctas[j]].astype(np.int64)
                dur.setdefault(int(cls[j]), []).append((d[:, 3].max() - d[:, 0].min()) / 1e3)
            g_us = sum(sum(dur.get(c, [])) for c in (0, 3, 4, 5))
            first = stamps[len(cls) - per, :ctas[len(cls) - per]].astype(np.int64)[:, 0].min()
            last = stamps[len(cls) - 1, :ctas[len(cls) - 1]].astype(np.int64)[:, 3].max()
            in_graph = {"gemv_us_per_token": g_us, "achieved": wbytes / (g_us * 1e-6) / 1e9, "frac": wbytes / (g_us * 1e-6) / 1e9 / peak,
                        "step_us_first_entry_to_last_exit": (last - first) / 1e3,
                        "per_class_us_per_token": {nm: float(sum(dur.get(c, []))) for c, nm in
                                                   ((0, "qkv"), (2, "attention"), (3, "wo"), (4, "w13"), (5, "w2"))},
                        "note": "launches overlap under programmatic dependent launch, so per-class times can sum to more than the step"}
        except Exception as ex:
            in_graph = {"error": repr(ex)}
        traffic, traffic_rd, traffic_n = ncu_traffic_per_launch()
        replay = {"achieved": achieved, "frac": achieved / peak, "avg_launch_us": 1e3 * only_ms / n_gemv,
                  "timing": "two CUDA events on the slice's stream around %d graph replays of the step's %d k_gemv launches with the "
                            "attention launch skipped (b200_debug_skip_attention): the matmul kernels back to back" % (reps, n_gemv)}
        in_step = in_graph if isinstance(in_graph, dict) and "achieved" in in_graph else None
        roof = {"bound": "hbm", "kernel": "k_gemv (Q4_0xQ8_0 exact-mode weight matmul; qkv, wo, w1|w3, w2 = 4 launches/layer)",
                # the dominant kernel AS IT RUNS INSIDE THE STEP (the replayed decode graph, programmatic dependent launch and
                # all): launch duration = last CTA exit - first CTA entry from in-kernel %globaltimer stamps
                "achieved": in_step["achieved"] if in_step else achieved, "peak": peak, "unit": "GB/s",
                "frac": (in_step["achieved"] if in_step else achieved) / peak, "peak_source": peak_src,
                "traffic": traffic, "traffic_read_only": traffic_rd,
                "traffic_source": "profiles/r02_decode_kernels_ncu_full.md: dram__bytes_read.sum + dram__bytes_write.sum averaged over its "
                                  "%d k_gemv launches (ncu --set full, one decode step, cold caches)" % traffic_n,
                "timing": ("in-step: %globaltimer stamps of every k_gemv launch inside the replayed decode graph, last of 3 steps"
                           if in_step else "matmul-only graph replay (in-step stamps unavailable)"),
                "algorithmic_bytes_per_launch": wbytes / n_gemv,
                "avg_launch_us": (in_step["gemv_us_per_token"] / n_gemv) if in_step else 1e3 * only_ms / n_gemv,
                "matmul_only_replay": replay,
                "event_bracketed": {"achieved": ev_achieved, "frac": ev_achieved / peak,
                                    "note": "one CUDA-event pair per launch, un-graphed: includes ~4 us of event overhead per launch"},
                "share_of_step": gemv_ms / float(ms.sum()),
                "per_class_us_per_token": {n: 1e3 * float(m) / nprof for n, m in
                                           zip(("qkv", "rope_append", "attention", "wo", "w13", "w2", "advance"), ms)},
                "in_graph": in_graph}
    # whole-step roofline: B(p) = W + KV read + KV write, mean over the positions of the timed steps
    W_all = 32 * (4 * (E * E // 32 * 18) + 3 * (E * sh.n_ff // 32 * 18)) + 32 * 2 * E * 4
    kv_pos = 32 * 2 * E * 2
    mean_p = float(np.mean([PREFILL + (i % cycle) for i in range(W, W + K)]))
    b_step = W_all + kv_pos * (mean_p + 1)
    peak, peak_src = measured_peak()
    step_roof = {"algorithmic_bytes_per_step": b_step, "roofline_tokens_per_s_one_gpu": peak * 1e9 / b_step,
                 "frac_of_one_gpu": value / (peak * 1e9 / b_step), "frac_of_n_gpus": value / (world * peak * 1e9 / b_step)}

    # ---- tokens/s at the last position of the sequence (p = 511, T = 512: the longest KV read; SURVEY 8d)
    def step_any():
        if world == 1:
            sl.forward_device(sl.dev_in, 1, sl.dev_out)
        else:
            import ctypes as C
            capi.check(capi.lib().b200_pipeline_step(sl.handle, C.c_void_p(sl.dev_in), 1, 1))

    if sl.n_past > N_CTX - 1:
        sl.rewind(N_CTX - 1)
    while sl.n_past < N_CTX - 1:
        step_any()                       # fill the cache up to position 510 (values do not matter for timing)
    barrier()
    p511 = []
    for i in range(3 + 16):
        sl.mark(0)
        step_any()
        sl.mark(1)
        barrier()
        if i >= 3:
            p511.append(sl.mark_elapsed_ms())
        sl.rewind(N_CTX - 1)
    p511_ms = float(statistics.median(p511))
    if dist is not None:
        import torch
        t = torch.tensor([p511_ms], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        p511_ms = float(t[0])
    b511 = W_all + kv_pos * N_CTX
    at_p511 = {"tokens_per_s": 1e3 / p511_ms, "ms_per_step": p511_ms, "algorithmic_bytes": b511,
               "frac_of_one_gpu": (1e3 / p511_ms) / (peak * 1e9 / b511),
               "how": "median of 16 single steps at position 511, one CUDA-event pair each on the slice's stream, max over ranks"}

    # ---- CPU baseline + parity against the compiled reference, EVERY N: rank 0 runs the reference over the N slice
    # files in sequence (the reference's own multi-node data flow, cli_api/common.py:148-154) on a 16-token prompt +
    # 16 decode steps; the GPU pipeline then runs the same tokens and the ring result is compared bit for bit.
    cpu = None
    parity = None
    if not args.no_cpu:
        NPAR, PROMPT = 16, 16
        x0 = synth_inputs(PROMPT, E, 1)
        xq = synth_inputs(NPAR + 1, E, 2)
        want = None
        if rank == 0:
            try:
                if world == 1:
                    r, x0, xq, outs = cpu_reference_run(path, E, NPAR, 1, prompt=PROMPT, want_outputs=True)
                    want = [None] + outs                       # the prompt's output is not compared at N=1 (as round 1)
                else:
                    r, want = cpu_reference_chain([slice_file("7b", x, y) for x, y in layer_ranges(sh.n_layer, world)],
                                                  E, x0, xq)
                cpu = {k: r[k] for k in ("value", "unit", "cores", "kind", "sample")}
            except Exception as ex:  # the bench line must still print
                cpu = {"value": None, "unit": UNIT, "cores": os.cpu_count(), "kind": "unavailable", "sample": repr(ex)}
        barrier()
        try:
            sl.clear_context()
            barrier()
            bad = tot = 0
            got_all = []
            for j, x in enumerate([x0] + [xq[i:i + 1] for i in range(xq.shape[0])]):
                if world == 1:
                    g = sl.forward(x)
                else:
                    import ctypes as C
                    if rank == 0:
                        _h2d(sl, x)
                    capi.check(capi.lib().b200_pipeline_step(sl.handle, C.c_void_p(sl.dev_in), x.shape[0], 1))
                    g = np.empty_like(x)
                    if rank == 0:
                        _d2h(sl, g)
                if rank == 0 and want is not None and want[j] is not None:
                    bad += int((g.view(np.uint32) != np.ascontiguousarray(want[j]).view(np.uint32)).sum())
                    tot += g.size
            if rank == 0 and want is not None:
                parity = {"checked_floats": tot, "mismatching_floats": bad, "against": cpu.get("kind"),
                          "what": "hidden states of the full 32-layer model through %d slice(s): %s%d decode steps, "
                                  "bit patterns compared" % (world, "a %d-token prompt call + " % PROMPT if world > 1 else "", NPAR + 1)}
        except Exception as ex:
            parity = {"error": repr(ex)}
        barrier()

    # ---- prompt throughput of the same model (not the headline metric): one 512-token call, device-resident, exact mode and the
    # opt-in tcgen05 fast mode (K2: dequant fused into a TMA-fed tcgen05 / TMEM tile kernel; tolerance-level parity)
    prefill = None
    if world == 1:
        try:
            x512 = synth_inputs(N_CTX, E, 3)
            _h2d(sl, x512)
            prefill, outs = {}, {}
            for name, fast in (("exact", False), ("tcgen05_fast", True)):
                sl.set_fast_prefill(fast, 32)
                for rep in range(2):
                    sl.clear_context()
                    sl.mark(0)
                    sl.forward_device(sl.dev_in, N_CTX, sl.dev_out)
                    sl.mark(1)
                    sl.sync()
                prefill[name + "_tokens_per_s"] = N_CTX / (sl.mark_elapsed_ms() / 1e3)
                o = np.empty((N_CTX, E), np.float32)
                _d2h(sl, o)
                outs[name] = o
            sl.set_fast_prefill(False, 32)
            sl.clear_context()
            d = outs["tcgen05_fast"] - outs["exact"]
            prefill["fast_vs_exact_rel_rms"] = float(np.sqrt(np.mean(d * d)) / np.sqrt(np.mean(outs["exact"] ** 2)))
            prefill["what"] = ("one %d-token prompt call through all 32 layers, activations resident in HBM; fast mode = fp16 tensor-core "
                               "matmuls (fastgemm2.cuh), off by default, decode is always exact" % N_CTX)
        except Exception as ex:
            prefill = {"error": repr(ex)}

    if rank == 0:
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
                "ms_per_step": dev_ms / K, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
                "dtype": "q4_0*q8_0->f32", "data": "synthetic",
                "config": {"workload": "LLaMA-7B Q4_0 (BASELINE.json configs[%d]): %d slice(s) x %s layers on %dxB200, "
                                       "n_ctx=512 batch=1, one decoded token per step after a 256-token prefill; timed steps at "
                                       "positions %s" % (1 if world == 1 else 2, world,
                                                          "/".join(str(y - x + 1) for x, y in layer_ranges(32, world)), world,
                                                          timed_positions),
                           "weights": "synthetic Q4_0 blocks (seed %d), reference slice-file format" % SEED,
                           "mode": "exact (bit-identical to the reference CPU path)",
                           "slice_load_seconds": round(load_seconds, 3), "cuda_init_seconds": round(cuda_init_seconds, 3),
                           "parallelism": ("pp%d (layer slices; hand-off = %s)" % (world, "peer-memory store + flag over NVLink inside the step graph"
                                                                    if transport == "peer" else "one ncclSend/ncclRecv per hop")) if world > 1 else "pp1",
                           "handoff_transport": transport,
                           "l2": "no flush: each step streams %.2f GB of weights, 29x the 126 MB L2" % (W_all / 1e9),
                           "timing": "CUDA events on the slice's stream around %d steps; wall %.1f ms" % (K, wall_ms)},
                "clocks": clk, "e2e": e2e, "gpu_launches": launches, "roofline": roof, "step_roofline": step_roof,
                "tokens_per_s_at_p511": at_p511["tokens_per_s"], "at_p511": at_p511, "prefill": prefill,
                "cpu_baseline": cpu, "parity": parity}
        print(json.dumps(line), flush=True)
    if world > 1:
        if capi.lib().b200_pipeline_error(sl.handle):
            sys.stderr.write("rank %d: a mailbox poll timed out\n" % rank)
        capi.check(capi.lib().b200_pipeline_destroy(sl.handle))
        dist.barrier()
        dist.destroy_process_group()
    sl.close()
    return 0


def _cudart():
    import ctypes as C
    for name in ("libcudart.so.12", "libcudart.so"):
        try:
            return C.CDLL(name)
        except OSError:
            continue
    import glob
    for p in glob.glob("/usr/local/cuda/lib64/libcudart.so*"):
        return C.CDLL(p)
    raise OSError("libcudart not found")


def _h2d(sl, x: np.ndarray):
    """Upload x into the slice's device input buffer (bench plumbing, outside the timed kernels)."""
    import ctypes as C
    x = np.ascontiguousarray(x, np.float32)
    rc = _cudart().cudaMemcpy(C.c_void_p(sl.dev_in), C.c_void_p(x.ctypes.data), C.c_size_t(x.nbytes), 1)
    assert rc == 0, rc
    # a cudaMemcpy from PAGEABLE memory returns once the source is staged; the DMA of the tail (> 1 MiB) may still be in
    # flight, and the slice's stream is non-blocking, i.e. not ordered behind the legacy stream: wait for the device
    assert _cudart().cudaDeviceSynchronize() == 0


def _d2h(sl, out: np.ndarray):
    """Read the step's result back to the host: the slice's own output on one GPU, and on rank 0 of a ring pipeline the
    LAST slice's output that the ring returned (b200_pipeline_result), i.e. the model's hidden state, not rank 0's."""
    import ctypes as C
    sl.sync()
    rc = _cudart().cudaMemcpy(C.c_void_p(out.ctypes.data), C.c_void_p(sl.pipeline_result), C.c_size_t(out.nbytes), 2)
    assert rc == 0, rc


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=256)
    ap.add_argument("--warmup", type=int, default=8)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the hidden state the last one computed to DIR/hidden_state.npy")
    args = ap.parse_args()
    if args.warmup < 3:
        args.warmup = 3
    if args.impl == "reference":
        return run_reference(args)
    return run_b200(args)


if __name__ == "__main__":
    sys.exit(main())
