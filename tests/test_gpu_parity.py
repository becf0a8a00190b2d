"""GPU parity: the sm_100a slice forward, called through the C ABI, against the CPU oracle.

Bar (SURVEY.md Appendix B, "exact mode"): hidden states BIT-IDENTICAL to the reference CPU path
for every weight type the slice path supports -- not a tolerance."""
import numpy as np
import pytest

from distributedllm_b200 import ggjt

pytestmark = pytest.mark.gpu


def _bits(a):
    return np.ascontiguousarray(a, dtype=np.float32).view(np.uint32)


def _run_pair(path, calls, shape, n_ctx=512, seed=1):
    from distributedllm_b200 import capi
    from oracle import oracle

    rng = np.random.default_rng(seed)
    gpu = capi.Slice(path, 0, n_ctx)
    cpu = oracle.PortSlice(path, n_ctx)
    bad = tot = 0
    try:
        for n in calls:
            x = rng.standard_normal((n, shape.n_embd), dtype=np.float32)
            a = cpu.forward(x)
            b = gpu.forward(x)
            bad += int((_bits(a) != _bits(b)).sum())
            tot += a.size
            assert np.isfinite(b).all()
    finally:
        gpu.close()
        cpu.close()
    return bad, tot


@pytest.mark.parametrize("shape,wtype", [("tiny", ggjt.T_Q4_0), ("tiny128", ggjt.T_Q4_0), ("tiny3b", ggjt.T_Q4_0),
                                         ("tiny", ggjt.T_Q8_0), ("tiny128", ggjt.T_Q8_0), ("tiny", ggjt.T_F16),
                                         ("tiny3b", ggjt.T_F16), ("tiny128", ggjt.T_F16),
                                         ("tiny", ggjt.T_Q4_1), ("tiny128", ggjt.T_Q4_1), ("tiny3b", ggjt.T_Q4_1)])
def test_bit_exact_prefill_then_decode(tmp_models, shape, wtype):
    sh = ggjt.SHAPES[shape]
    path = tmp_models(shape, wtype, 1, 2)
    bad, tot = _run_pair(path, [40, 1, 1, 7, 1, 20, 3, 1], sh)
    assert bad == 0, "%d of %d floats differ from the oracle" % (bad, tot)


@pytest.mark.parametrize("wtype,version", [(ggjt.T_Q4_1, 2), (ggjt.T_F16, 2), (ggjt.T_Q8_0, 1)],
                         ids=["q4_1", "f16", "q8_0-v1"])
def test_fast_prefill_switch_keeps_other_types_exact(tmp_models, monkeypatch, wtype, version):
    """Fast mode covers Q4_0 (and Q8_0 with the v2 kernel) only; every other slice ignores the switch and stays
    bit-identical to the oracle.  tiny128b passes the shape test, so only the weight type decides."""
    monkeypatch.setenv("B200_FAST_PREFILL", "1")
    monkeypatch.setenv("B200_FAST_MIN_TOKENS", "2")
    monkeypatch.setenv("B200_FAST_V", str(version))
    sh = ggjt.SHAPES["tiny128b"]
    path = tmp_models("tiny128b", wtype, 0, 1)
    bad, tot = _run_pair(path, [40, 1, 1, 7, 1, 130, 3, 1], sh)
    assert bad == 0, "%d of %d floats differ from the oracle" % (bad, tot)


def test_ring_and_simple_kernels_agree(tmp_models, monkeypatch):
    sh = ggjt.SHAPES["tiny3b"]
    path = tmp_models("tiny3b", ggjt.T_Q4_0, 0, 2)
    for ring in ("1", "0"):
        monkeypatch.setenv("B200_RING", ring)
        bad, tot = _run_pair(path, [33, 1, 1, 1, 5], sh)
        assert bad == 0, "ring=%s: %d of %d floats differ" % (ring, bad, tot)


@pytest.mark.parametrize("shape,wtype", [("tiny", ggjt.T_Q4_0), ("tiny128", ggjt.T_Q4_0), ("tiny128", ggjt.T_Q4_1)])
def test_decode_only_long(tmp_models, shape, wtype):
    sh = ggjt.SHAPES[shape]
    path = tmp_models(shape, wtype, 0, 2)
    bad, tot = _run_pair(path, [1] * 40, sh)
    assert bad == 0


@pytest.mark.parametrize("pdl,graph,nq", [("0", "1", "0"), ("1", "0", "0"), ("0", "0", "0"), ("1", "1", "1"), ("0", "0", "1")])
def test_launch_modes_agree(tmp_models, monkeypatch, pdl, graph, nq):
    """Programmatic dependent launch, CUDA-graph replay and the grid-barrier norm+quant epilogue (B200_NQ) are
    scheduling / fusion choices only: all stay bit-exact."""
    monkeypatch.setenv("B200_PDL", pdl)
    monkeypatch.setenv("B200_GRAPH", graph)
    monkeypatch.setenv("B200_NQ", nq)
    sh = ggjt.SHAPES["tiny128"]
    path = tmp_models("tiny128", ggjt.T_Q4_0, 0, 2)
    bad, tot = _run_pair(path, [37, 1, 1, 1, 30, 1, 1], sh)
    assert bad == 0


@pytest.mark.parametrize("mc", ["1", "0"])
@pytest.mark.parametrize("shape", ["tiny", "tiny3b", "tiny128"])
def test_f16_multi_column_kernel_is_a_scheduling_choice(tmp_models, monkeypatch, mc, shape):
    """F16 slices, multi-token calls: 8 / 4 columns per CTA share every weight load (k_gemv_f16_mc) or one column per CTA."""
    monkeypatch.setenv("B200_F16_MC", mc)
    sh = ggjt.SHAPES[shape]
    path = tmp_models(shape, ggjt.T_F16, 0, 1)
    bad, tot = _run_pair(path, [33, 2, 1, 5, 9, 1, 4], sh)
    assert bad == 0, "%d of %d floats differ" % (bad, tot)


@pytest.mark.parametrize("n8", ["1", "0"])
@pytest.mark.parametrize("shape,wtype", [("tiny128", ggjt.T_Q4_0), ("tiny3b", ggjt.T_Q8_0), ("tiny", ggjt.T_Q8_0)])
def test_narrow_matrix_kernel_is_a_scheduling_choice(tmp_models, monkeypatch, n8, shape, wtype):
    """Single-token wo / w2 run 8 threads per row (k_gemv_n8, one AVX lane per thread) instead of 4: the same lane chains."""
    monkeypatch.setenv("B200_N8", n8)
    sh = ggjt.SHAPES[shape]
    path = tmp_models(shape, wtype, 0, 2)
    bad, tot = _run_pair(path, [5, 1, 1, 1, 1, 30, 1, 1], sh)
    assert bad == 0, "%d of %d floats differ" % (bad, tot)


@pytest.mark.parametrize("ring,nq", [("1", "0"), ("0", "0"), ("0", "1")])
def test_q4_1_launch_modes_agree(tmp_models, monkeypatch, ring, nq):
    """Q4_1 slices (unsigned nibbles + the scalar min chain, Q8_1 activations): the fused RMSNorm prologue (B200_NQ=0), the
    grid-barrier epilogue and the ring-less kernels are the same arithmetic."""
    monkeypatch.setenv("B200_RING", ring)
    monkeypatch.setenv("B200_NQ", nq)
    sh = ggjt.SHAPES["tiny3b"]
    path = tmp_models("tiny3b", ggjt.T_Q4_1, 0, 2)
    bad, tot = _run_pair(path, [21, 1, 1, 1, 9, 1], sh)
    assert bad == 0, "%d of %d floats differ" % (bad, tot)
    path = tmp_models("tiny128", ggjt.T_Q4_1, 0, 1)
    bad, tot = _run_pair(path, [1, 1, 1, 40, 1], ggjt.SHAPES["tiny128"])
    assert bad == 0, "%d of %d floats differ" % (bad, tot)


@pytest.mark.parametrize("nc", ["8", "4", "2"])
@pytest.mark.parametrize("shape,wtype", [("tiny128", ggjt.T_Q4_0), ("tiny3b", ggjt.T_Q8_0), ("tiny128", ggjt.T_Q4_1)])
def test_columns_per_cta_is_a_scheduling_choice(tmp_models, monkeypatch, nc, shape, wtype):
    """Multi-token calls pick 8 / 4 / 2 columns per CTA from the matrix width and the batch; columns never interact."""
    monkeypatch.setenv("B200_NC", nc)
    sh = ggjt.SHAPES[shape]
    path = tmp_models(shape, wtype, 0, 1)
    bad, tot = _run_pair(path, [19, 8, 1, 3, 2], sh)
    assert bad == 0


def test_context_overflow_and_clear(tmp_models):
    from distributedllm_b200 import capi

    sh = ggjt.SHAPES["tiny"]
    path = tmp_models("tiny", ggjt.T_Q4_0, 0, 1)
    s = capi.Slice(path, 0, 16)
    x = np.ones((10, sh.n_embd), np.float32)
    y0 = s.forward(x)
    with pytest.raises(capi.B200Error) as e:
        s.forward(x)
    assert e.value.code == 5
    s.clear_context()
    assert s.n_past == 0
    y1 = s.forward(x)
    assert (_bits(y0) == _bits(y1)).all()
    s.close()


def test_edge_cases_empty_ragged_and_full_context(tmp_models):
    """Empty call, a ragged call length (not a multiple of the 8 / 4 / 2 column groups), filling the context to the last
    position in one-token steps and in one call, rewinding: all as the reference behaves (tensor_processor.cpp:1523-1544
    appends at n_past; the reference itself would write past its cache on overflow, we refuse)."""
    from distributedllm_b200 import capi
    from oracle import oracle
    sh = ggjt.SHAPES["tiny128"]
    path = tmp_models("tiny128", ggjt.T_Q4_0, 0, 0)
    n_ctx = 40
    gpu, ref = capi.Slice(path, 0, n_ctx), oracle.PortSlice(path, n_ctx)
    with pytest.raises(capi.B200Error) as e:
        gpu.forward(np.zeros((0, sh.n_embd), np.float32))
    assert e.value.code == 1 and gpu.n_past == 0
    rng = np.random.default_rng(77)
    x = rng.standard_normal((13, sh.n_embd), dtype=np.float32)              # 13 = 8 + 4 + 1 columns
    assert (_bits(gpu.forward(x)) == _bits(ref.forward(x))).all()
    for _ in range(n_ctx - 13):                                            # up to the very last position
        t = rng.standard_normal((1, sh.n_embd), dtype=np.float32)
        assert (_bits(gpu.forward(t)) == _bits(ref.forward(t))).all()
    assert gpu.n_past == n_ctx
    with pytest.raises(capi.B200Error) as e:
        gpu.forward(t)
    assert e.value.code == 5 and gpu.n_past == n_ctx
    # rewind to a previous position and replay: the cache below the rewind point is intact
    gpu.rewind(13)
    ref2 = oracle.PortSlice(path, n_ctx)
    ref2.forward(x)
    t = rng.standard_normal((5, sh.n_embd), dtype=np.float32)
    assert (_bits(gpu.forward(t)) == _bits(ref2.forward(t))).all()
    # the whole context in ONE call
    gpu.clear_context()
    ref3 = oracle.PortSlice(path, n_ctx)
    full = rng.standard_normal((n_ctx, sh.n_embd), dtype=np.float32)
    assert (_bits(gpu.forward(full)) == _bits(ref3.forward(full))).all()
    for r in (ref, ref2, ref3):
        r.close()
    gpu.close()


@pytest.mark.parametrize("tiled", [1, 0], ids=["query-tiled", "cluster-per-query"])
def test_both_prompt_attention_kernels_are_exact(tmp_models, monkeypatch, tiled):
    """Prompt chunks of head-size-128 models run the query-tiled kernel (K / V staged once per 16 queries) while the whole
    context fits its 512-row window, the per-query cluster kernel beyond; both must be the oracle's arithmetic.  Ragged
    chunks: T crosses multiples of 32 inside a call, a 1-token call in between, a chunk that is not a multiple of 16."""
    monkeypatch.setenv("B200_TILED_ATTN", str(tiled))
    sh = ggjt.SHAPES["tiny128"]
    path = tmp_models("tiny128", ggjt.T_Q4_0, 0, 2, seed=17)
    bad, tot = _run_pair(path, [37, 1, 70, 5, 16, 33, 200, 64], sh, n_ctx=512, seed=3)
    assert bad == 0, "%d of %d floats differ" % (bad, tot)


def test_prompt_attention_beyond_the_staged_window(tmp_models):
    """n_ctx 1024: chunks that end beyond position 512 fall back to the cluster kernel mid-prompt; still exact."""
    sh = ggjt.SHAPES["tiny128"]
    path = tmp_models("tiny128", ggjt.T_Q4_0, 0, 1, seed=18)
    bad, tot = _run_pair(path, [300, 200, 40, 1, 100], sh, n_ctx=1024, seed=4)
    assert bad == 0, "%d of %d floats differ" % (bad, tot)
