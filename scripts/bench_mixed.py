"""Admission of a new session into a running batch: today's two passes against one mixed step (b200_mixed_forward).

Workload: BASELINE config 5's per-GPU slice (LLaMA-13B shape, 5 layers, Q4_0), n_ctx 512, 64 sessions.  Sessions 0..62 are
decoding at p ~ 256; session 63 arrives with a prompt of P tokens (P = 16, 64, 128).
  A  session_forward(63, prompt), then batch_forward(0..62): the decoding sessions wait for the whole prompt pass (the stall)
  B  one mixed step: the prompt chunk and the 63 decode tokens share one weight pass
A and B alternate in one process, each from the same state (positions rewound between steps), timed with CUDA events on the
slice's stream after warm-up; one step per timed window, median over --reps.  A and B must give identical bits.
Output: one JSON object on stdout (and --out FILE).  The slice's weights (~1.1 GB) are far larger than the 126 MB L2."""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

import bench
from distributedllm_b200 import capi

N_CTX, B, P0 = 512, 64, 256


def gpu_identity():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, clock = [f.strip() for f in q.split(",")]
        return {"gpu": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as ex:                                       # the identity is reported, not required
        return {"gpu": torch.cuda.get_device_name(0), "power_limit": "unknown (%r)" % ex}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--prompts", default="16,64,128")
    ap.add_argument("--reps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    lib = capi.lib()
    sl = capi.Slice(bench.slice_file("13b", 0, 4), 0, N_CTX, n_sessions=B)
    E = sl.n_embd
    dec = list(range(B - 1))
    # decoding sessions at p = 256: the tensor-core prefill gets them there fast; the timed steps below are all exact
    sl.set_fast_prefill(True, 32)
    x = bench.synth_inputs(P0, E, 7)
    for k in dec:
        sl.session_forward(k, x)
    sl.set_fast_prefill(False, 32)
    res = {"workload": "LLaMA-13B Q4_0, 5-layer slice (1 of 8), n_ctx %d, %d sessions decoding at p=%d, session %d admits a prompt of P"
                       % (N_CTX, B - 1, P0, B - 1), **gpu_identity(), "reps": args.reps, "timing": "CUDA events, median of reps", "by_prompt": {}}
    for P in [int(p) for p in args.prompts.split(",")]:
        rows = P + B - 1
        xin = torch.from_numpy(bench.synth_inputs(rows, E, 100 + P)).cuda()     # [prompt rows][decode rows]
        out_a, out_b = torch.empty_like(xin), torch.empty_like(xin)
        torch.cuda.synchronize()
        ids_b, lens_b = [B - 1] + dec, [P] + [1] * (B - 1)

        def reset():
            for k in dec:
                sl.session_rewind(k, P0)
            sl.session_clear(B - 1)

        def run_prompt():
            capi.check(lib.b200_session_forward_device(sl.handle, B - 1, C.c_void_p(xin.data_ptr()), P, C.c_void_p(out_a.data_ptr()), 0))

        def run_a():
            run_prompt()
            sl.batch_forward_device(dec, xin.data_ptr() + 4 * P * E, out_a.data_ptr() + 4 * P * E)

        def run_b():
            sl.mixed_forward_device(ids_b, lens_b, xin.data_ptr(), out_b.data_ptr())

        def timed(fn):
            reset()
            sl.sync()
            sl.mark(0)
            fn()
            sl.mark(1)
            sl.sync()
            return sl.mark_elapsed_ms()

        for _ in range(args.warmup):
            timed(run_a)
            timed(run_b)
        ta, tb, stalls = [], [], []
        for _ in range(args.reps):
            stalls.append(timed(run_prompt))                      # the prompt pass alone: what sessions 0..62 wait in A
            ta.append(timed(run_a))
            tb.append(timed(run_b))
        torch.cuda.synchronize()
        same = bool(torch.equal(out_a.view(torch.int32), out_b.view(torch.int32)))
        a, b = float(np.median(ta)), float(np.median(tb))
        res["by_prompt"][str(P)] = {
            "A_two_passes_ms": a, "B_mixed_step_ms": b, "B_over_A": b / a,
            "A_tokens_per_s": rows * 1e3 / a, "B_tokens_per_s": rows * 1e3 / b,
            "A_decode_stall_ms": float(np.median(stalls)),
            "A_ms_min_max": [min(ta), max(ta)], "B_ms_min_max": [min(tb), max(tb)],
            "bit_identical": same}
        assert same, "mixed step differs from session_forward + batch_forward at P=%d" % P
    sl.close()
    line = json.dumps(res, indent=1)
    print(line, flush=True)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
