"""The tcgen05 fast-mode prefill matmuls one at a time, against a float64 reference of the same operation.

b200_debug_fast_matmul runs one weight matmul of a slice with the launches a fast prefill uses: k_prep_q8_f16, then the
tcgen05 kernel (csrc/fastgemm2.cuh, or csrc/fastgemm.cuh with B200_FAST_V=1) and its STORE (qkv), RESID (wo, w2) or
GATE (w1|w3) epilogue.  It returns the output and the fp16 activation operand xh.  The reference rebuilds both operands:
  * xh: RMSNorm (float32 squares, float64 sum) for qkv and w1|w3, the reference's Q8_0 activation quantisation
    (quantize_row_q8_0: d = fp16(amax / 127), q = rint(x * 127 / amax)), then fp16(q * d).  The kernel's xh must be
    bit-identical to it;
  * W16: fp16((n - 8) * d) for Q4_0 and fp16(q * d) for Q8_0, one rounding each, as the dequant warps form them.
Y_ref = W16 . xh in float64 then differs from the kernel only by the order of the fp32 accumulation.  Bounds:
  * STORE / RESID, every element: |y - ref| <= C * sum_k |w_k x_k|  (+ 2^-23 |ref| for the residual add);
    relative RMS over the call <= 1e-5;
  * GATE: y = fp16(silu(fp16(g))) * u with ggml's fp16 SiLU table.  g and u each get the bound above; it is carried
    through the table, and g may land one fp16 step beyond its interval;
  * rows past n_tokens still hold the sentinel, every output row is finite.
Measured on an NVIDIA B200 (1000 W power limit): the largest C any element needed ("required C"), over every N, edge
row and token tile; v2 with 128- or 256-token tiles and v1 gave the same value per matrix:
                      qkv      wo       w1|w3    w2
    tiny128b/c Q4_0   3.3e-7   2.4e-7   4.0e-8   4.1e-7
    tiny128b/c Q8_0   3.4e-7   2.7e-7   6.8e-8   4.8e-7
    3b  (Q4_0)        5.3e-7   5.5e-7   1.1e-7   8.7e-7
    7b  (Q4_0)        6.6e-7   6.1e-7   1.3e-7   8.7e-7
    13b (Q4_0)        6.6e-7   5.8e-7   1.6e-7   1.3e-6
So C = 2^-16 (1.5e-5), 12 x the worst measured.  Relative RMS: at most 6.0e-6 for qkv / wo and 1.65e-5 for w2
(13B, K = 13824: it grows with K), so the bound is 1e-4; w1|w3 reaches 7.8e-5 (g crossing an fp16 step of the SiLU
table) and is held by the per-element bound only.
The checker self-test (CPU) injects faults into the reference output: one 16-wide K slice of one 8-row group dropped,
one token's output swapped with its neighbour's, one 8-row group shifted by one row, and a w1 / w3 pair swapped.  It
asserts that each needs at least 10 x C; on tiny128c the least of them needs 2.1e-2 of sum |w x| (1350 x C)."""
import numpy as np
import pytest

from distributedllm_b200 import ggjt

C_BOUND = 2.0 ** -16
RESID_ULP = 2.0 ** -23
REL_RMS = 1e-4
SENTINEL = 0xFFFFFFFF
NS = [1, 31, 32, 127, 128, 129, 255, 256, 257, 384, 511, 512]
MATS = ["qkv", "wo", "w13", "w2"]
VARIANTS = [(ggjt.T_Q4_0, 2, 128), (ggjt.T_Q4_0, 2, 256), (ggjt.T_Q4_0, 1, 0), (ggjt.T_Q8_0, 2, 128), (ggjt.T_Q8_0, 2, 256)]
VARIANT_IDS = ["q4_0-v2-n128", "q4_0-v2-n256", "q4_0-v1", "q8_0-v2-n128", "q8_0-v2-n256"]


# ---------------------------------------------------------------------------------------------- reference
def prep_ref(x, norm_w=None):
    """The activation operand as k_prep_q8_f16 forms it: [RMSNorm * w ->] Q8_0 -> fp16(q * d)."""
    x = np.ascontiguousarray(x, dtype=np.float32)
    if norm_w is not None:
        ss = (x * x).astype(np.float64).sum(axis=1)
        mean = (ss / x.shape[1]).astype(np.float32)
        scale = np.float32(1) / np.sqrt(mean + np.float32(1e-6))
        x = (x * scale[:, None]) * np.asarray(norm_w, np.float32)[None, :]
    n, k = x.shape
    b = x.reshape(n, k // 32, 32)
    amax = np.abs(b).max(axis=2)
    d = (amax / np.float32(127)).astype(np.float16).astype(np.float32)
    with np.errstate(divide="ignore"):
        idv = np.where(amax != 0, np.float32(127) / amax, np.float32(0)).astype(np.float32)
    q = np.rint(b * idv[..., None]) + np.float32(0)                # round half to even, as the kernel and lrintf; -0 -> +0 (an int)
    return (q * d[..., None]).astype(np.float16).reshape(n, k)


def weights16(f, name, rows=None):
    """Rows of a Q4_0 / Q8_0 matrix of slice file `f` as the fp16 values the dequant warps form."""
    t = f.tensors[name]
    k, n_rows = t.ne
    bs = ggjt.TYPE_BLOCK[t.ttype][1]
    blk = np.frombuffer(f.read_raw(name), np.uint8).reshape(n_rows, k // 32, bs)
    if rows is not None:
        blk = blk[rows]
    d = blk[..., 0:2].copy().view(np.float16)                      # [r, nb, 1]
    if t.ttype == ggjt.T_Q4_0:
        qs = blk[..., 2:]
        q = np.concatenate([qs & 15, qs >> 4], axis=2).astype(np.int16) - 8
    else:
        assert t.ttype == ggjt.T_Q8_0
        q = blk[..., 2:].copy().view(np.int8)
    return (q.astype(np.float16) * d).reshape(-1, k)               # exact product, one fp16 rounding


def silu_table():
    from oracle import oracle
    texp, tsilu = np.zeros(65536, np.uint16), np.zeros(65536, np.uint16)
    L = oracle.port_lib()
    L.orc_tables(texp.ctypes.data, tsilu.ctypes.data)
    return tsilu


def silu16(tsilu, g16):
    return tsilu[np.asarray(g16, np.float16).view(np.uint16)].view(np.float16).astype(np.float64)


class Expect:
    """Reference output with the per-element tolerance `slack + C * unit` of one matmul."""

    def __init__(self, ref, slack, unit, rel_rms=True):
        self.ref, self.slack, self.unit, self.rel_rms = ref, slack, unit, rel_rms

    def required_c(self, y, n=None):
        """Smallest C under which y passes (inf: an element with no C-dependent slack is off)."""
        n = y.shape[0] if n is None else n
        err = np.abs(np.asarray(y, np.float64)[:n] - self.ref[:n])
        excess = err - self.slack[:n]
        unit = self.unit[:n]
        with np.errstate(divide="ignore", invalid="ignore"):
            req = np.where(unit > 0, excess / np.where(unit > 0, unit, 1), np.where(excess > 0, np.inf, 0.0))
        return float(req.max())

    def rel_rms_of(self, y, n):
        d = np.asarray(y, np.float64)[:n] - self.ref[:n]
        return float(np.sqrt(np.mean(d * d)) / np.sqrt(np.mean(self.ref[:n] ** 2)))


def expect_linear(xh, w16, resid=None):
    X, W = xh.astype(np.float64), w16.astype(np.float64)
    ref = X @ W.T
    unit = np.abs(X) @ np.abs(W).T
    slack = np.zeros_like(ref)
    if resid is not None:
        ref = ref + np.asarray(resid, np.float64)
        slack = RESID_ULP * np.abs(ref)
    return Expect(ref, slack, unit)


def gate_parts(xh, w1, w3):
    X = xh.astype(np.float64)
    g, u = X @ w1.astype(np.float64).T, X @ w3.astype(np.float64).T
    sg, su = np.abs(X) @ np.abs(w1.astype(np.float64)).T, np.abs(X) @ np.abs(w3.astype(np.float64)).T
    return g, u, sg, su


def expect_gate(g, u, sg, su, tsilu, c=C_BOUND):
    """y = fp16(silu(fp16(g))) * u; g within c * sg, plus one fp16 step either side; u within c * su."""
    s = silu16(tsilu, g.astype(np.float16))
    lo = np.nextafter((g - c * sg).astype(np.float16), np.float16(-np.inf))
    hi = np.nextafter((g + c * sg).astype(np.float16), np.float16(np.inf))
    ds = np.maximum(np.abs(silu16(tsilu, lo) - s), np.abs(silu16(tsilu, hi) - s))
    ds += np.spacing(np.abs(s).astype(np.float16)).astype(np.float64)    # silu is not monotonic near its minimum
    ref = s * u
    slack = ds * np.abs(u) + RESID_ULP * (np.abs(ref) + ds * np.abs(u))
    return Expect(ref, slack, (np.abs(s) + ds) * su, rel_rms=False)


def layer_inputs(sh, which, n=512, seed=0):
    """Inputs of one matmul: Gaussian rows with edge rows at the token-tile boundaries 0, 127, 128, 255, 256, 511."""
    K = sh.n_ff if which == 3 else sh.n_embd
    rng = np.random.default_rng([seed, which, K])
    x = rng.standard_normal((n, K), dtype=np.float32)
    x[0] = 0.0
    x[0, 37] = 1.75                                     # a single nonzero element
    x[127] = 0.0                                        # all zero
    x[128, 64:96] = 0.0                                 # one all-zero 32-block
    x[255] = 0.625                                      # all equal
    x[256] *= np.float32(1e-7)                          # un-normalised (wo, w2): d rounds to fp16 zero
    x[511] *= np.float32(3e4) / np.abs(x[511]).max()    # amax 3e4: still inside the fp16 range
    resid = rng.standard_normal((n, sh.n_embd), dtype=np.float32) if which in (1, 3) else None
    return x, resid


def layer_names(layer):
    pre = "layers.%d." % layer
    return {k: pre + v for k, v in (("attn_norm", "attention_norm.weight"), ("ffn_norm", "ffn_norm.weight"),
                                     ("wq", "attention.wq.weight"), ("wk", "attention.wk.weight"),
                                     ("wv", "attention.wv.weight"), ("wo", "attention.wo.weight"),
                                     ("w1", "feed_forward.w1.weight"), ("w2", "feed_forward.w2.weight"),
                                     ("w3", "feed_forward.w3.weight"))}


def norm_weight(f, name):
    return np.frombuffer(f.read_raw(name), np.float32)


def build_expect(f, layer, which, x, resid, tsilu, rows=None):
    """(xh, Expect) of matmul `which` of `layer` on inputs x, for output rows `rows` (None: all)."""
    nm = layer_names(f.hparams.first_layer + layer)
    E = f.hparams.n_embd
    if which == 0:
        xh = prep_ref(x, norm_weight(f, nm["attn_norm"]))
        if rows is None:
            w = np.concatenate([weights16(f, nm[k]) for k in ("wq", "wk", "wv")])
        else:
            rows = np.asarray(rows)
            w = np.concatenate([weights16(f, nm[k], rows[(rows >= i * E) & (rows < (i + 1) * E)] - i * E)
                                for i, k in enumerate(("wq", "wk", "wv"))])
        return xh, expect_linear(xh, w)
    if which == 2:
        xh = prep_ref(x, norm_weight(f, nm["ffn_norm"]))
        g, u, sg, su = gate_parts(xh, weights16(f, nm["w1"], rows), weights16(f, nm["w3"], rows))
        return xh, expect_gate(g, u, sg, su, tsilu)
    xh = prep_ref(x)
    r = None if resid is None else (resid if rows is None else resid[:, rows])
    return xh, expect_linear(xh, weights16(f, nm["wo" if which == 1 else "w2"], rows), r)


def check_output(y, xh, n, xh_ref, exp, sample=None):
    """Asserts the operand bits, the sentinel rows, finiteness and the bounds -> (required C, relative RMS) of the first n rows."""
    assert np.array_equal(xh.view(np.uint16), xh_ref[:n].view(np.uint16)), \
        "xh differs from the Q8_0 recipe in %d of %d values" % (int((xh.view(np.uint16) != xh_ref[:n].view(np.uint16)).sum()), xh.size)
    assert (y[n:].view(np.uint32) == SENTINEL).all(), "rows past n_tokens were written"
    body = y[:n]
    assert np.isfinite(body).all(), "%d non-finite outputs" % int((~np.isfinite(body)).sum())
    if sample is not None:
        body = body[:, sample]
    req = exp.required_c(body, n)
    assert req <= C_BOUND, "N=%d: an element needs C = %.3g > %.3g" % (n, req, C_BOUND)
    rel = exp.rel_rms_of(body, n)
    if exp.rel_rms:
        assert rel <= REL_RMS, "N=%d: relative RMS %.3g > %.3g" % (n, rel, REL_RMS)
    return req, rel


# ---------------------------------------------------------------------------------------------- checker self-test (CPU)
@pytest.fixture(scope="module")
def selftest_case(tmp_path_factory):
    sh = ggjt.SHAPES["tiny128c"]
    path = str(tmp_path_factory.mktemp("fastmm") / "tiny128c_q4_0.bin")
    ggjt.write_synth_slice(path, sh, 0, 0, ggjt.T_Q4_0, seed=3)
    return sh, ggjt.read_file(path), silu_table()


def test_prep_recipe_matches_the_oracle_quantiser():
    """prep_ref's Q8_0 step is the oracle's orc_quant_q8_0 (quantize_row_q8_0) bit for bit, edge rows included."""
    from oracle import oracle
    L = oracle.port_lib()
    sh = ggjt.SHAPES["tiny128c"]
    for which in (1, 3):
        x, _ = layer_inputs(sh, which)
        xh = prep_ref(x)
        k = x.shape[1]
        q, d = np.zeros(k, np.int8), np.zeros(k // 32, np.uint16)
        for r in range(0, x.shape[0], 7):
            row = np.ascontiguousarray(x[r])
            L.orc_quant_q8_0(row.ctypes.data, k, q.ctypes.data, d.ctypes.data)
            want = (q.astype(np.float32).reshape(-1, 32) * d.view(np.float16).astype(np.float32)[:, None]).astype(np.float16)
            assert np.array_equal(xh[r].view(np.uint16), want.reshape(-1).view(np.uint16)), (which, r)
    assert not xh[256].any() and np.abs(xh[511].astype(np.float32)).max() > 2e4


@pytest.mark.parametrize("which", [0, 1, 2, 3], ids=MATS)
def test_checker_catches_injected_faults(selftest_case, which):
    sh, f, tsilu = selftest_case
    x, resid = layer_inputs(sh, which)
    xh, exp = build_expect(f, 0, which, x, resid, tsilu)
    assert exp.required_c(exp.ref.astype(np.float32)) <= C_BOUND          # the reference itself, rounded to float32, passes
    nm = layer_names(0)
    X = xh.astype(np.float64)
    g0, k0, t0 = 5, 48, 40                                                  # 8-row group, 16-wide K slice, token
    rows = slice(8 * g0, 8 * g0 + 8)
    faults = {}
    if which == 2:
        w1, w3 = weights16(f, nm["w1"]).astype(np.float64), weights16(f, nm["w3"]).astype(np.float64)
        g, u = X @ w1.T, X @ w3.T
        gd = g.copy()
        gd[:, rows] -= X[:, k0:k0 + 16] @ w1[rows, k0:k0 + 16].T
        faults["dropped K slice"] = silu16(tsilu, gd.astype(np.float16)) * u
        sw = exp.ref.copy()
        sw[:, rows] = silu16(tsilu, u[:, rows].astype(np.float16)) * g[:, rows]
        faults["w1 / w3 swapped"] = sw
    else:
        w = (np.concatenate([weights16(f, nm[k]) for k in ("wq", "wk", "wv")]) if which == 0
             else weights16(f, nm["wo" if which == 1 else "w2"])).astype(np.float64)
        yd = exp.ref.copy()
        yd[:, rows] -= X[:, k0:k0 + 16] @ w[rows, k0:k0 + 16].T
        faults["dropped K slice"] = yd
    ts = exp.ref.copy()
    ts[[t0, t0 + 1]] = ts[[t0 + 1, t0]]
    faults["tokens swapped"] = ts
    sh_ = exp.ref.copy()
    sh_[:, rows] = exp.ref[:, 8 * g0 + 1:8 * g0 + 9]
    faults["row group shifted"] = sh_
    for name, y in faults.items():
        req = exp.required_c(y)
        assert req >= 10 * C_BOUND, "%s: needs C = %.3g only (bound %.3g)" % (name, req, C_BOUND)


# ---------------------------------------------------------------------------------------------- the kernels (GPU)
_expect_cache = {}


def _cached_expect(path, shape, which, tsilu):
    if (path, which) not in _expect_cache:
        f = ggjt.read_file(path)
        x, resid = layer_inputs(ggjt.SHAPES[shape], which, seed=1)
        xh, exp = build_expect(f, 1, which, x, resid, tsilu)
        _expect_cache[(path, which)] = (x, resid, xh, exp)
    return _expect_cache[(path, which)]


@pytest.fixture(scope="module")
def tsilu():
    return silu_table()


@pytest.mark.gpu
@pytest.mark.parametrize("which", [0, 1, 2, 3], ids=MATS)
@pytest.mark.parametrize("variant", VARIANTS, ids=VARIANT_IDS)
@pytest.mark.parametrize("shape", ["tiny128b", "tiny128c"])
def test_fast_matmul_matches_float64_reference(tmp_models, monkeypatch, tsilu, shape, variant, which):
    """Every prefix length N of a 512-row input against the reference of the 512 rows (prep and the matmul are row-wise)."""
    from distributedllm_b200 import capi
    wtype, version, tile = variant
    monkeypatch.setenv("B200_FAST_V", str(version))
    path = tmp_models(shape, wtype, 0, 1)
    x, resid, xh_ref, exp = _cached_expect(path, shape, which, tsilu)
    sl = capi.Slice(path, 0, 512)
    worst = worst_rel = 0.0
    try:
        for n in NS:
            y, xh = sl.debug_fast_matmul(1, which, x[:n], None if resid is None else resid[:n], tile=tile)
            req, rel = check_output(y, xh, n, xh_ref, exp)
            worst, worst_rel = max(worst, req), max(worst_rel, rel)
    finally:
        sl.close()
    print("fast-matmul %s %s %s: required C %.3g, relative RMS %.3g" % (shape, VARIANT_IDS[VARIANTS.index(variant)],
                                                                      MATS[which], worst, worst_rel))


@pytest.mark.gpu
def test_hook_refuses_what_forward_would_not_run_fast(tmp_models, monkeypatch):
    """Slices whose weights never run fast (tiny128: w1|w3 is not a whole number of M tiles; Q4_1; F16; Q8_0 under v1) and
    bad arguments are refused with B200_EINVAL."""
    from distributedllm_b200 import capi
    sh = ggjt.SHAPES["tiny128b"]
    x = np.ones((4, sh.n_embd), np.float32)

    def refused(sl, *args, **kw):
        with pytest.raises(capi.B200Error) as e:
            sl.debug_fast_matmul(*args, **kw)
        return e.value.code == 1

    for shape, wtype in (("tiny128", ggjt.T_Q4_0), ("tiny128b", ggjt.T_Q4_1), ("tiny128b", ggjt.T_F16)):
        sl = capi.Slice(tmp_models(shape, wtype, 0, 0), 0, 64)
        assert refused(sl, 0, 0, x)
        sl.close()
    sl = capi.Slice(tmp_models("tiny128b", ggjt.T_Q4_0, 0, 0), 0, 64)
    assert refused(sl, 1, 0, x)                                                # no layer 1 in this slice
    assert refused(sl, 0, 0, np.ones((65, sh.n_embd), np.float32))            # more tokens than n_ctx
    assert refused(sl, 0, 0, x, tile=64)
    assert refused(sl, 0, 1, x)                                                # wo without its residual
    sl.close()
    monkeypatch.setenv("B200_FAST_V", "1")
    sl = capi.Slice(tmp_models("tiny128b", ggjt.T_Q4_0, 0, 0), 0, 64)
    assert refused(sl, 0, 0, x, tile=256)                                      # v1 has 128-token tiles only
    sl.close()
    sl = capi.Slice(tmp_models("tiny128b", ggjt.T_Q8_0, 0, 0), 0, 64)
    assert refused(sl, 0, 0, x)                                                # v1 is Q4_0 only
    sl.close()


# ---------------------------------------------------------------------------------------------- full-size widths (GPU)
@pytest.fixture(scope="module")
def full_layers(tmp_path_factory):
    root = tmp_path_factory.mktemp("fastmm_full")
    paths = {}

    def get(shape):
        if shape not in paths:
            p = str(root / ("%s_layer0.bin" % shape))
            ggjt.write_fast_q4_slice(p, ggjt.SHAPES[shape], 0, 0, seed=5)
            paths[shape] = p
        return paths[shape]
    return get


@pytest.mark.gpu
@pytest.mark.parametrize("shape", ["3b", "7b", "13b"])
def test_fast_matmul_full_size_widths(full_layers, tsilu, shape):
    """One layer of the real widths, the token tile a forward picks (tile = 0), N = 512 and 300; 7B qkv and w1|w3 at
    N = 512 run the full 256-token tile.  Sampled output rows: the first and last 128 and 256 random ones."""
    from distributedllm_b200 import capi
    sh = ggjt.SHAPES[shape]
    path = full_layers(shape)
    f = ggjt.read_file(path)
    sl = capi.Slice(path, 0, 512)
    rng = np.random.default_rng(9)
    try:
        for which in range(4):
            rows_out = (3 * sh.n_embd, sh.n_embd, sh.n_ff, sh.n_embd)[which]
            sample = np.unique(np.concatenate([np.arange(128), np.arange(rows_out - 128, rows_out),
                                               rng.choice(rows_out, 256, replace=False)]))
            x, resid = layer_inputs(sh, which, seed=2)
            xh_ref, exp = build_expect(f, 0, which, x, resid, tsilu, rows=sample)
            for n in (512, 300):
                y, xh = sl.debug_fast_matmul(0, which, x[:n], None if resid is None else resid[:n])
                req, rel = check_output(y, xh, n, xh_ref, exp, sample=sample)
                print("fast-matmul %s %s N=%d: required C %.3g, relative RMS %.3g" % (shape, MATS[which], n, req, rel))
    finally:
        sl.close()


@pytest.mark.gpu
def test_fast_prefill_full_3b_layer_close_to_exact(full_layers):
    """OpenLLaMA-3B widths pass the fast-path predicate with head size 100: fast matmuls around the generic k_attention,
    against exact mode with the slice-level tolerance of test_gpu_fast_prefill.py."""
    from distributedllm_b200 import capi
    sh = ggjt.SHAPES["3b"]
    path = full_layers("3b")
    x = np.random.default_rng(4).standard_normal((300, sh.n_embd), dtype=np.float32)
    exact, fast = capi.Slice(path, 0, 512), capi.Slice(path, 0, 512)
    fast.set_fast_prefill(True, 32)
    try:
        ye, yf = exact.forward(x), fast.forward(x)
        assert np.isfinite(yf).all()
        assert not np.array_equal(ye, yf)                                 # the fast path ran
        rel_rms = float(np.sqrt(np.mean((yf - ye) ** 2)) / np.sqrt(np.mean(ye ** 2)))
        max_rel = float(np.abs(yf - ye).max() / np.abs(ye).max())
        assert rel_rms <= 1.5e-2, rel_rms
        assert max_rel <= 1e-1, max_rel
    finally:
        exact.close()
        fast.close()
