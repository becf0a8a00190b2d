"""Mixed steps (b200_mixed_forward*, b200_pipeline_step_mixed): prompt chunks and decode tokens of several sessions in one
pass.  Every segment must be bit-identical to a forward of its session alone -- against the oracle, against a twin handle,
through the `llm` module and through a two-slice pipeline -- and a rejected step must change nothing."""
import os
import subprocess
import sys

import numpy as np
import pytest

from distributedllm_b200 import ggjt

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bits(a):
    return np.ascontiguousarray(a, dtype=np.float32).view(np.uint32)


def _split(rows, n_tokens):
    return np.split(rows, np.cumsum(n_tokens)[:-1])


@pytest.mark.gpu
@pytest.mark.parametrize("shape,wtype", [("tiny128", ggjt.T_Q4_0), ("tiny3b", ggjt.T_Q4_0), ("tiny128", ggjt.T_Q8_0),
                                         ("tiny", ggjt.T_F16), ("tiny128", ggjt.T_Q4_1)])
def test_mixed_steps_equal_private_contexts(tmp_models, shape, wtype):
    from distributedllm_b200 import capi
    from oracle import oracle
    sh = ggjt.SHAPES[shape]
    path = tmp_models(shape, wtype, 0, 1, seed=41)
    n_ctx = 128
    gpu = capi.Slice(path, 0, n_ctx, n_sessions=8)
    rng = np.random.default_rng(11)
    prompt = {0: 3, 1: 0, 2: 20, 3: 9, 4: 0, 5: 40, 6: 1, 7: 31}      # every session at its own position (1, 4: empty)
    cpu = {}
    for k, n in prompt.items():
        cpu[k] = oracle.PortSlice(path, n_ctx)
        if n:
            x = rng.standard_normal((n, sh.n_embd), dtype=np.float32)
            assert (_bits(gpu.session_forward(k, x)) == _bits(cpu[k].forward(x))).all(), k
    # single tokens next to chunks of 15, 16, 17 and 33: chunks straddle the 16-query blocks and the 32-slot tail
    steps = [([6, 0, 3, 7], [15, 1, 33, 1]),
             ([2, 6, 5, 0, 3, 4], [16, 1, 17, 1, 1, 15]),
             ([1, 7, 2, 6, 4], [33, 17, 1, 16, 1])]
    for i, (ids, lens) in enumerate(steps):
        x = rng.standard_normal((sum(lens), sh.n_embd), dtype=np.float32)
        got = gpu.mixed_forward(ids, lens, x)
        for k, g, xs in zip(ids, _split(got, lens), _split(x, lens)):
            assert (_bits(g) == _bits(cpu[k].forward(xs))).all(), (i, k)
    # single-token steps read every KV row the mixed steps appended
    for k in range(8):
        for _ in range(2):
            x = rng.standard_normal((1, sh.n_embd), dtype=np.float32)
            assert (_bits(gpu.session_forward(k, x)) == _bits(cpu[k].forward(x))).all(), k
    for c in cpu.values():
        c.close()
    gpu.close()


@pytest.mark.gpu
def test_mixed_step_long_context_takes_both_attention_kernels(tmp_models):
    """n_ctx 1024: a 40-token chunk at n_past 500 (T = 540, per-query cluster kernel) next to a chunk that ends exactly at
    T = 512 (the tiled kernel's largest window) and two decode tokens, against a twin handle stepping each session alone."""
    from distributedllm_b200 import capi
    sh = ggjt.SHAPES["tiny128"]
    path = tmp_models("tiny128", ggjt.T_Q4_0, 0, 1, seed=42)
    mixed, twin = capi.Slice(path, 0, 1024, n_sessions=4), capi.Slice(path, 0, 1024, n_sessions=4)
    rng = np.random.default_rng(12)
    for k, n in ((0, 500), (1, 488), (2, 300), (3, 7)):
        for i in range(0, n, 128):
            x = rng.standard_normal((min(128, n - i), sh.n_embd), dtype=np.float32)
            assert (_bits(mixed.session_forward(k, x)) == _bits(twin.session_forward(k, x))).all()
    ids, lens = [2, 0, 1, 3], [1, 40, 24, 1]
    x = rng.standard_normal((sum(lens), sh.n_embd), dtype=np.float32)
    got = mixed.mixed_forward(ids, lens, x)
    for k, g, xs in zip(ids, _split(got, lens), _split(x, lens)):
        assert (_bits(g) == _bits(twin.session_forward(k, xs))).all(), k
    assert [mixed.session_n_past(k) for k in range(4)] == [540, 512, 301, 8]
    for k in range(4):
        x = rng.standard_normal((1, sh.n_embd), dtype=np.float32)
        assert (_bits(mixed.session_forward(k, x)) == _bits(twin.session_forward(k, x))).all(), k
    mixed.close()
    twin.close()


@pytest.mark.gpu
def test_mixed_step_degenerate_cases(tmp_models):
    """All segments of one token = the batched step; one segment = a forward of that session; the fast-prefill switch is
    ignored (a mixed step always runs in exact mode)."""
    from distributedllm_b200 import capi
    sh = ggjt.SHAPES["tiny128b"]                          # every matrix qualifies for the tensor-core prefill
    path = tmp_models("tiny128b", ggjt.T_Q4_0, 0, 1, seed=43)
    mixed, twin = capi.Slice(path, 0, 256, n_sessions=5), capi.Slice(path, 0, 256, n_sessions=5)
    rng = np.random.default_rng(13)
    for k in range(5):
        x = rng.standard_normal((3 + 4 * k, sh.n_embd), dtype=np.float32)
        assert (_bits(mixed.session_forward(k, x)) == _bits(twin.session_forward(k, x))).all()
    ids = [3, 0, 4, 1]
    x = rng.standard_normal((4, sh.n_embd), dtype=np.float32)
    assert (_bits(mixed.mixed_forward(ids, [1, 1, 1, 1], x)) == _bits(twin.batch_forward(ids, x))).all()
    x = rng.standard_normal((37, sh.n_embd), dtype=np.float32)
    assert (_bits(mixed.mixed_forward([2], [37], x)) == _bits(twin.session_forward(2, x))).all()
    mixed.set_fast_prefill(True, 2)
    for ids, lens in (([1], [64]), ([0, 2, 3], [48, 1, 33])):
        x = rng.standard_normal((sum(lens), sh.n_embd), dtype=np.float32)
        got = mixed.mixed_forward(ids, lens, x)
        for k, g, xs in zip(ids, _split(got, lens), _split(x, lens)):
            assert (_bits(g) == _bits(twin.session_forward(k, xs))).all(), k
    mixed.close()
    twin.close()


@pytest.mark.gpu
def test_mixed_step_segment_order_is_free(tmp_models):
    from distributedllm_b200 import capi
    sh = ggjt.SHAPES["tiny128"]
    path = tmp_models("tiny128", ggjt.T_Q4_0, 0, 1, seed=44)
    a, b = capi.Slice(path, 0, 128, n_sessions=4), capi.Slice(path, 0, 128, n_sessions=4)
    rng = np.random.default_rng(14)
    for k in range(4):
        x = rng.standard_normal((2 + 5 * k, sh.n_embd), dtype=np.float32)
        a.session_forward(k, x)
        b.session_forward(k, x)
    seg = {0: 17, 1: 1, 2: 33, 3: 1}
    xs = {k: rng.standard_normal((n, sh.n_embd), dtype=np.float32) for k, n in seg.items()}
    outs = []
    for h, order in ((a, [0, 1, 2, 3]), (b, [3, 2, 1, 0])):
        lens = [seg[k] for k in order]
        got = h.mixed_forward(order, lens, np.concatenate([xs[k] for k in order]))
        outs.append(dict(zip(order, _split(got, lens))))
    for k in seg:
        assert (_bits(outs[0][k]) == _bits(outs[1][k])).all(), k
    a.close()
    b.close()


@pytest.mark.gpu
def test_rejected_mixed_step_changes_nothing(tmp_models):
    from distributedllm_b200 import capi
    sh = ggjt.SHAPES["tiny128"]
    path = tmp_models("tiny128", ggjt.T_Q4_0, 0, 1, seed=45)
    n_ctx = 64
    a, twin = capi.Slice(path, 0, n_ctx, n_sessions=3), capi.Slice(path, 0, n_ctx, n_sessions=3)
    rng = np.random.default_rng(15)
    for k, n in ((0, 5), (1, 50), (2, 1)):
        x = rng.standard_normal((n, sh.n_embd), dtype=np.float32)
        a.session_forward(k, x)
        twin.session_forward(k, x)
    before = [a.session_n_past(k) for k in range(3)]
    bad = [([0, 0], [1, 1], 1),          # a session listed twice
           ([0, 2], [3, 0], 1),          # an empty segment
           ([0, 2], [3, -2], 1),         # a negative one
           ([0, 3], [1, 1], 1),          # a session out of range
           ([-1, 0], [1, 1], 1),
           ([0, 2], [40, 30], 1),        # 70 tokens in one step > n_ctx
           ([0, 1, 2], [2, 15, 1], 5)]   # session 1 would reach 65 > n_ctx
    for ids, lens, code in bad:
        x = np.zeros((max(sum(lens), 0), sh.n_embd), np.float32)
        with pytest.raises(capi.B200Error) as e:
            a.mixed_forward(ids, lens, x)
        assert e.value.code == code, (ids, lens)
        assert [a.session_n_past(k) for k in range(3)] == before, (ids, lens)
    ids, lens = [2, 1, 0], [1, 14, 9]
    x = rng.standard_normal((sum(lens), sh.n_embd), dtype=np.float32)
    got = a.mixed_forward(ids, lens, x)
    for k, g, xs in zip(ids, _split(got, lens), _split(x, lens)):
        assert (_bits(g) == _bits(twin.session_forward(k, xs))).all(), k
    assert [a.session_n_past(k) for k in range(3)] == [14, 64, 2]
    a.close()
    twin.close()


@pytest.mark.gpu
def test_llm_module_propagate_forward_mixed(tmp_models, monkeypatch):
    from distributedllm_b200 import capi
    from distributedllm_b200.compute_node.slices import import_llm
    llm = import_llm()
    sh = ggjt.SHAPES["tiny128"]
    path = tmp_models("tiny128", ggjt.T_Q4_0, 0, 1, seed=46)
    monkeypatch.setenv("B200_SESSIONS", "3")
    monkeypatch.setenv("B200_N_CTX", "64")
    llm.load_slice(path)
    try:
        rng = np.random.default_rng(16)
        priv = [capi.Slice(path, 0, 64) for _ in range(3)]
        x = rng.standard_normal((6, sh.n_embd), dtype=np.float32)
        assert (_bits(np.frombuffer(llm.propagate_forward_session(1, x), np.float32)) == _bits(priv[1].forward(x)).ravel()).all()
        ids, lens = [2, 1, 0], [18, 1, 5]
        x = rng.standard_normal((sum(lens), sh.n_embd), dtype=np.float32)
        got = np.frombuffer(llm.propagate_forward_mixed(ids, lens, x), np.float32).reshape(-1, sh.n_embd)
        for k, g, xs in zip(ids, _split(got, lens), _split(x, lens)):
            assert (_bits(g) == _bits(priv[k].forward(xs))).all(), k
        with pytest.raises(RuntimeError):
            llm.propagate_forward_mixed([0, 0], [1, 1], np.zeros((2, sh.n_embd), np.float32))
        with pytest.raises(ValueError):
            llm.propagate_forward_mixed([0, 1], [2, 1], np.zeros((2, sh.n_embd), np.float32))
        with pytest.raises(ValueError):
            llm.propagate_forward_mixed([0, 1], [1], np.zeros((1, sh.n_embd), np.float32))
        for p in priv:
            p.close()
    finally:
        llm.unload_slice()


WORKER = r'''
import os, sys, ctypes as C
sys.path.insert(0, %(root)r)
import numpy as np, torch, torch.distributed as dist
from distributedllm_b200 import capi, ggjt
from distributedllm_b200.pipeline import layer_ranges, join_pipeline, torch_collectives
rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
torch.cuda.set_device(local)
dist.init_process_group("nccl", device_id=torch.device("cuda", local))
sh = ggjt.SHAPES["tiny128"]
d = %(tmp)r
a, b = layer_ranges(sh.n_layer, world)[rank]
p = os.path.join(d, "s_%%d_%%d.bin" %% (a, b))
ggjt.write_synth_slice(p, sh, a, b, ggjt.T_Q4_0, seed=0)
sl = capi.Slice(p, local, 128, n_sessions=4)
lib = capi.lib()
bcast, gather = torch_collectives(dist, torch.device("cuda", local))
transport = join_pipeline(sl, rank, world, bcast, gather, peer=os.environ.get("B200_PP_PEER", "1") != "0")
if rank == 0:
    whole = os.path.join(d, "whole.bin"); ggjt.write_synth_slice(whole, sh, 0, sh.n_layer - 1, ggjt.T_Q4_0, seed=0)
    ref = capi.Slice(whole, local, 128, n_sessions=4)
rng = np.random.default_rng(22)
buf = torch.zeros((128, sh.n_embd), dtype=torch.float32, device="cuda")
ok = True
steps = [([1, 2], [9, 3]), ([3, 1, 2], [17, 1, 1]), ([0, 2, 3, 1], [33, 16, 1, 1]), ([2, 0], [1, 1])]
for ids, lens in steps:
    x = rng.standard_normal((sum(lens), sh.n_embd), dtype=np.float32)
    if rank == 0:
        buf[:len(x)].copy_(torch.from_numpy(x))
        torch.cuda.synchronize()
    ids_a, lens_a = np.array(ids, np.int32), np.array(lens, np.int32)
    capi.check(lib.b200_pipeline_step_mixed(sl.handle, C.c_void_p(ids_a.ctypes.data), C.c_void_p(lens_a.ctypes.data), len(ids),
                                            C.c_void_p(buf.data_ptr()), 1))
    sl.sync()
    if rank == 0:
        res = torch.empty((len(x), sh.n_embd), dtype=torch.float32, device="cuda")
        n = res.numel() * 4
        C.CDLL("libcudart.so.12").cudaMemcpy(C.c_void_p(res.data_ptr()), C.c_void_p(lib.b200_pipeline_result(sl.handle)), C.c_size_t(n), 3)
        torch.cuda.synchronize()
        got = res.cpu().numpy()
        want = np.concatenate([ref.session_forward(k, xs) for k, xs in zip(ids, np.split(x, np.cumsum(lens)[:-1]))])
        ok = ok and bool((got.view(np.uint32) == want.view(np.uint32)).all())
# a rejected list is rejected on every rank before anything is sent: the pipeline stays usable
ids_a, lens_a = np.array([1, 1], np.int32), np.array([1, 1], np.int32)
rc = lib.b200_pipeline_step_mixed(sl.handle, C.c_void_p(ids_a.ctypes.data), C.c_void_p(lens_a.ctypes.data), 2, C.c_void_p(buf.data_ptr()), 1)
ok = ok and rc == 1
ok = ok and [sl.session_n_past(k) for k in range(4)] == [34, 11, 21, 18]
dist.barrier()
capi.check(lib.b200_pipeline_destroy(sl.handle))
err = lib.b200_pipeline_error(sl.handle)
if rank == 0:
    print(("MIXED_OK" if ok and not err else "MIXED_MISMATCH") + " transport=" + transport)
dist.destroy_process_group()
'''


@pytest.mark.gpu
@pytest.mark.parametrize("peer", [1, 0], ids=["peer", "nccl"])
def test_two_gpu_pipeline_mixed_steps(tmp_path, peer):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    script = tmp_path / "worker.py"
    script.write_text(WORKER % {"root": ROOT, "tmp": str(tmp_path)})
    env = dict(os.environ, B200_PP_PEER=str(peer))
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
                          "--master-addr", "127.0.0.1", "--master-port", str(29571 + peer), str(script)],
                         capture_output=True, text=True, timeout=600, env=env)
    assert "MIXED_OK" in out.stdout, out.stdout[-2000:] + out.stderr[-3000:]
    assert ("transport=peer" if peer else "transport=nccl") in out.stdout, out.stdout[-500:]


def test_mixed_entry_points_refuse_without_a_device():
    """No CPU fallback: without a device the mixed-step entry points answer B200_ENODEV."""
    code = ("import sys, ctypes as C; sys.path.insert(0, %r)\n"
            "from distributedllm_b200 import capi\n"
            "L = capi.lib(); ids = (C.c_int * 1)(0); n = (C.c_int * 1)(1); x = (C.c_float * 4)()\n"
            "print('codes', L.b200_mixed_forward(None, ids, n, 1, x, x), L.b200_mixed_forward_device(None, ids, n, 1, x, x, 1),\n"
            "      L.b200_pipeline_step_mixed(None, ids, n, 1, x, 1))\n" % ROOT)
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    out = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, timeout=120)
    assert "codes 3 3 3" in out.stdout, out.stdout + out.stderr      # B200_ENODEV
