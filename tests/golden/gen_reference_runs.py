"""Record the compiled reference's outputs for the tests that compare with it bit for bit (reference_runs.json).

Each entry replays one test's inputs -- the same seeded slice files and input rows the test builds -- through
oracle/_ref (distllm/tensor_processor.cpp compiled unmodified, see oracle/Makefile) and keeps one record per
reference call (oracle/goldens.py: shape, SHA-256 of the float32 bytes, a few sampled values).  The tests then check
the C restatement or the GPU against these records, so they need neither the reference nor its build.

    python tests/golden/gen_reference_runs.py          # needs a built oracle/_ref
"""
import hashlib
import json
import os
import subprocess
import sys
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
from distributedllm_b200 import ggjt  # noqa: E402
from oracle import goldens, oracle  # noqa: E402
from oracle.goldens import record  # noqa: E402

THREADS = min(16, os.cpu_count() or 4)       # the reference's results do not depend on its thread count


def calls(path, n_embd, seed, schedule):
    """Records of one reference slice fed seeded rows, len(schedule) calls of schedule[i] rows each."""
    ref = oracle.RefSlice(path, THREADS, 512)
    rng = np.random.default_rng(seed)
    out = [record(ref.forward(rng.standard_normal((n, n_embd), dtype=np.float32))) for n in schedule]
    ref.close()
    return out


def port_live(tmp):
    """tests/test_oracle.py::test_port_matches_live_reference"""
    out = {}
    for shape, wtype in (("tiny", ggjt.T_F32), ("tiny128", ggjt.T_F16), ("tiny3b", ggjt.T_Q8_0), ("tiny3b", ggjt.T_Q4_1)):
        sh = ggjt.SHAPES[shape]
        path = os.path.join(tmp, "m.bin")
        ggjt.write_synth_slice(path, sh, 0, 1, wtype, seed=3)
        out["%s/%s" % (shape, ggjt.TYPE_NAME[wtype])] = calls(path, sh.n_embd, 5, (34, 1, 2, 1))
    return out


def fast_q4_1_writer(tmp):
    """tests/test_oracle.py::test_fast_q4_1_writer_files_are_valid_for_the_reference"""
    sh = ggjt.SHAPES["tiny128"]
    path = os.path.join(tmp, "fast_q4_1.bin")
    ggjt.write_fast_q4_slice(path, sh, 0, 1, 0, wtype=ggjt.T_Q4_1)
    return calls(path, sh.n_embd, 11, (20, 1, 1))


def quantize_q4_1(tmp):
    """tests/test_ggjt_and_abi.py::test_q4_1_quantizer_is_the_reference_quantize_tool: SHA-256 of every Q4_1 tensor
    the reference's `quantize ... q4_1` writes."""
    sh = ggjt.SHAPES["tiny3b"]
    full, fq = os.path.join(tmp, "f32.bin"), os.path.join(tmp, "q41.bin")
    ggjt.write_synth_full(full, sh, ggjt.T_F32, seed=0)
    subprocess.run([os.path.join(oracle.REF_DIR, "quantize"), full, fq, "q4_1"], check=True, capture_output=True)
    b = ggjt.read_file(fq)
    return {name: hashlib.sha256(b.read_raw(name)).hexdigest() for name, t in b.tensors.items() if t.ttype == ggjt.T_Q4_1}


def gpu_live(tmp):
    """tests/test_gpu_llm_api.py::test_gpu_matches_live_reference"""
    sh = ggjt.SHAPES["tiny128"]
    path = os.path.join(tmp, "tiny128.bin")
    ggjt.write_synth_slice(path, sh, 0, 2, ggjt.T_Q4_0, seed=5)
    return calls(path, sh.n_embd, 8, (45, 1, 1, 1))


def config1(tmp):
    """tests/test_gpu_full_size.py::test_config1_3b_two_nodes_greedy_decode: the reference's embedding lookup, two
    slices and argmax, 16-token prompt + 32 generated tokens."""
    sh = ggjt.SHAPES["3b"]
    pa, pb, extra = (os.path.join(tmp, n) for n in ("a.bin", "b.bin", "extra.bin"))
    ggjt.write_fast_q4_slice(pa, sh, 0, 16, seed=3)
    ggjt.write_fast_q4_slice(pb, sh, 17, 25, seed=3)
    ggjt.write_fast_q4_extra(extra, sh, seed=3)
    ref = [oracle.RefSlice(pa, THREADS, 512), oracle.RefSlice(pb, THREADS, 512)]
    tr = [1 + (i * 7919) % 31999 for i in range(16)]
    hidden, ids = [], []
    for step in range(33):
        y = oracle.ref_embed(extra, tr, sh.n_embd)
        for s in ref:
            y = s.forward(y)
        hidden.append(record(y))
        ids.append(oracle.ref_lib().ref_next_token(extra.encode(), y.ctypes.data, y.size))
        tr = [ids[-1]]
    for s in ref:
        s.close()
    return {"hidden": hidden, "ids": ids}


def config4(tmp):
    """tests/test_gpu_full_size.py::test_config4_7b_f16_layer_at_n_ctx_2048"""
    sh = ggjt.SHAPES["7b"]
    path = os.path.join(tmp, "f16.bin")
    ggjt.write_fast_f16_slice(path, sh, 0, 0, seed=4)
    return calls(path, sh.n_embd, 9, (24, 1, 1, 9, 1))


def config5(tmp):
    """tests/test_gpu_full_size.py::test_config5_13b_batch_of_8_sessions: each session run alone on the reference."""
    sh = ggjt.SHAPES["13b"]
    path = os.path.join(tmp, "q4.bin")
    ggjt.write_fast_q4_slice(path, sh, 0, 0, seed=5)
    B = 8
    refs = [oracle.RefSlice(path, THREADS, 512) for _ in range(B)]
    rng = np.random.default_rng(10)
    prompts = [record(refs[b].forward(rng.standard_normal((3 + 2 * b, sh.n_embd), dtype=np.float32))) for b in range(B)]
    steps = []
    for step in range(3):
        x = rng.standard_normal((B, sh.n_embd), dtype=np.float32)
        steps.append([record(refs[b].forward(x[b:b + 1])[0]) for b in range(B)])
    for r in refs:
        r.close()
    return {"prompts": prompts, "steps": steps}


def config2(tmp):
    """tests/test_gpu_full_size.py::test_config2_7b_q4_decode_at_the_end_of_the_sequence: prompt chunks up to p = 500,
    then single tokens at p = 500..511."""
    sh = ggjt.SHAPES["7b"]
    path = os.path.join(tmp, "q4_7b_2l.bin")
    ggjt.write_fast_q4_slice(path, sh, 0, 1, seed=6)
    chunks = [min(oracle.RefSlice.MAX_CHUNK, 500 - pos) for pos in range(0, 500, oracle.RefSlice.MAX_CHUNK)]
    return calls(path, sh.n_embd, 11, chunks + [1] * 12)


def main():
    if not oracle.have_ref():
        raise SystemExit("oracle/_ref is not built (oracle/Makefile)")
    runs = {}
    for gen in (port_live, fast_q4_1_writer, quantize_q4_1, gpu_live, config1, config4, config5, config2):
        with tempfile.TemporaryDirectory() as tmp:
            runs[gen.__name__] = gen(tmp)
        print(gen.__name__, "done", flush=True)
    with open(goldens.RUNS, "w") as f:
        json.dump(runs, f, indent=0)
        f.write("\n")
    print("written", goldens.RUNS)


if __name__ == "__main__":
    main()
