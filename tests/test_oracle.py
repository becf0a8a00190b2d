"""The oracle is pinned here: the C restatement (oracle/slice_oracle.c) must reproduce, BIT FOR BIT, hidden states
the reference itself produced (tests/golden/slices.npz, dumped from oracle/_ref by gen_golden.py), and the reference's
outputs recorded on further inputs (tests/golden/reference_runs.json, written by gen_reference_runs.py)."""
import hashlib
import json
import os

import numpy as np
import pytest

from distributedllm_b200 import ggjt
from oracle import goldens, oracle

GOLD = os.path.join(os.path.dirname(__file__), "golden")
META = json.load(open(os.path.join(GOLD, "slices.json")))
META.update(json.load(open(os.path.join(GOLD, "slices_q4_1.json"))))
DATA = dict(np.load(os.path.join(GOLD, "slices.npz")))
DATA.update(np.load(os.path.join(GOLD, "slices_q4_1.npz")))


def _bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


@pytest.mark.parametrize("name", sorted(META))
def test_port_matches_reference_goldens(name, tmp_path):
    m = META[name]
    sh = ggjt.SHAPES[m["shape"]]
    path = str(tmp_path / (name + ".bin"))
    ggjt.write_synth_slice(path, sh, m["layers"][0], m["layers"][1], m["wtype"], seed=0)
    assert hashlib.sha256(open(path, "rb").read()).hexdigest() == m["file_sha256"], "synthetic slice file drifted"
    port = oracle.PortSlice(path, 512)
    for i, n in enumerate(m["schedule"]):
        x, y = DATA["%s/x%d" % (name, i)], DATA["%s/y%d" % (name, i)]
        assert x.shape[0] == n
        got = port.forward(x)
        assert (_bits(got) == _bits(y)).all(), "%s call %d: %d floats differ" % (name, i, int((_bits(got) != _bits(y)).sum()))
    port.close()


@pytest.mark.parametrize("shape,wtype", [("tiny", ggjt.T_F32), ("tiny128", ggjt.T_F16), ("tiny3b", ggjt.T_Q8_0),
                                         ("tiny3b", ggjt.T_Q4_1)])
def test_port_matches_live_reference(shape, wtype, tmp_path):
    """Against the outputs the compiled reference gave on these inputs (reference_runs.json: port_live)."""
    sh = ggjt.SHAPES[shape]
    want = goldens.load("port_live")["%s/%s" % (shape, ggjt.TYPE_NAME[wtype])]
    path = str(tmp_path / "m.bin")
    ggjt.write_synth_slice(path, sh, 0, 1, wtype, seed=3)
    port = oracle.PortSlice(path, 512)
    rng = np.random.default_rng(5)
    for i, n in enumerate((34, 1, 2, 1)):
        x = rng.standard_normal((n, sh.n_embd), dtype=np.float32)
        goldens.check(port.forward(x), want[i], "call %d" % i)
    port.close()


def test_slicing_is_transparent(tmp_path):
    """slice [0..3] == slice [0..1] then [2..3] (SURVEY 6: chained slices are bit-identical)."""
    sh = ggjt.SHAPES["tiny"]
    whole, lo, hi = (str(tmp_path / n) for n in ("w.bin", "lo.bin", "hi.bin"))
    ggjt.write_synth_slice(whole, sh, 0, 3, ggjt.T_Q4_0, 0)
    ggjt.write_synth_slice(lo, sh, 0, 1, ggjt.T_Q4_0, 0)
    ggjt.write_synth_slice(hi, sh, 2, 3, ggjt.T_Q4_0, 0)
    a, b, c = oracle.PortSlice(whole), oracle.PortSlice(lo), oracle.PortSlice(hi)
    rng = np.random.default_rng(0)
    for n in (9, 1, 1):
        x = rng.standard_normal((n, sh.n_embd), dtype=np.float32)
        assert (_bits(a.forward(x)) == _bits(c.forward(b.forward(x)))).all()


def test_fp16_round_to_nearest_even():
    L = oracle.port_lib()
    vals = np.concatenate([np.random.default_rng(0).standard_normal(5000).astype(np.float32) * 10.0 ** np.random.default_rng(1).integers(-9, 6, 5000),
                           np.array([0, -0.0, 65504, 65519.99, 65520, 1e-8, 5.96e-8, 2.98e-8, 2.9802322e-8, 6.1e-5, np.inf, -np.inf], np.float32)]).astype(np.float32)
    want = vals.astype(np.float16).view(np.uint16)
    got = np.array([L.orc_fp32_to_fp16(float(v)) for v in vals], np.uint16)
    assert (got == want).all()


def test_q8_0_activation_quant_matches_survey_recipe():
    """amax/127 stored as fp16, 127/amax multiplier, round-half-even (ggml.c:1215-1252)."""
    L = oracle.port_lib()
    rng = np.random.default_rng(2)
    x = rng.standard_normal(256).astype(np.float32)
    x[32:64] = 0
    x[64] = 0.5 * 127 / 127      # exercise a tie
    q = np.zeros(256, np.int8)
    d = np.zeros(8, np.uint16)
    L.orc_quant_q8_0(x.ctypes.data, 256, q.ctypes.data, d.ctypes.data)
    xb = x.reshape(8, 32)
    m = np.abs(xb).max(1).astype(np.float32)
    assert (d == (m / np.float32(127)).astype(np.float16).view(np.uint16)).all()
    idv = np.where(m != 0, np.float32(127) / np.where(m != 0, m, 1), 0).astype(np.float32)
    assert (q.reshape(8, 32) == np.rint((xb * idv[:, None]).astype(np.float32)).astype(np.int8)).all()


def test_q4_1_dot_is_scale_chain_plus_min_chain():
    """ggml_vec_dot_q4_1_q8_1 (ggml.c:2700-2733): unsigned nibbles, 8 fma lanes with d0*d1 (d1 NOT rounded to fp16), and
    the min term m*s added block by block as a scalar float; Q8_1's s = d * sum(q) (ggml.c:1472)."""
    L = oracle.port_lib()
    rng = np.random.default_rng(9)
    k = 128
    w = ggjt.quantize_q4_1(rng.standard_normal((1, k)).astype(np.float32) + 0.3)
    x = rng.standard_normal(k).astype(np.float32)
    x[32:64] = 0
    q, d, s = np.zeros(k, np.int8), np.zeros(k // 32, np.float32), np.zeros(k // 32, np.float32)
    L.orc_quant_q8_1(x.ctypes.data, k, q.ctypes.data, d.ctypes.data, s.ctypes.data)
    amax = np.abs(x.reshape(-1, 32)).max(1).astype(np.float32)
    assert (d.view(np.uint32) == (amax / np.float32(127)).astype(np.float32).view(np.uint32)).all()
    assert (s.view(np.uint32) == (d * q.reshape(-1, 32).sum(1).astype(np.float32)).astype(np.float32).view(np.uint32)).all()
    got = L.orc_dot_q4_1_q8_1(w.ctypes.data, q.ctypes.data, d.ctypes.data, s.ctypes.data, k)
    blocks = w.reshape(-1, 20)
    acc, summs = np.zeros(8, np.float32), np.float32(0)
    for b in range(k // 32):
        d0 = blocks[b, 0:2].copy().view(np.float16).astype(np.float32)[0]
        m0 = blocks[b, 2:4].copy().view(np.float16).astype(np.float32)[0]
        nib = np.concatenate([blocks[b, 4:] & 0x0F, blocks[b, 4:] >> 4]).astype(np.int32)
        summs = np.float32(summs + np.float32(m0 * s[b]))
        si = (nib * q[b * 32:(b + 1) * 32].astype(np.int32)).reshape(8, 4).sum(1)
        dd = np.float32(d0 * d[b])
        acc = (dd.astype(np.float64) * si.astype(np.float64) + acc.astype(np.float64)).astype(np.float32)   # fma: one rounding
    r0, r1, r2, r3 = (np.float32(acc[i + 4] + acc[i]) for i in range(4))
    want = np.float32(np.float32(np.float32(r0 + r2) + np.float32(r1 + r3)) + summs)
    assert np.float32(got).view(np.uint32) == want.view(np.uint32)
    # and the file-format side: the numpy quantiser's blocks decode to within one step of the input
    xw = rng.standard_normal((4, 64)).astype(np.float32)
    blk = ggjt.quantize_q4_1(xw)
    step = (xw.reshape(4, 2, 32).max(2) - xw.reshape(4, 2, 32).min(2)) / 15
    assert (np.abs(ggjt.dequantize_q4_1(blk) - xw).reshape(4, 2, 32).max(2) <= step * 0.51 + 2e-3).all()


def test_fast_q4_1_writer_files_are_valid_for_the_reference(tmp_path):
    """The benchmark generator's Q4_1 files (random 20-byte blocks, ggjt.write_fast_q4_slice) load in the compiled reference
    and the C restatement agrees with it on them, prompt and single-token steps (the reference's outputs are recorded in
    reference_runs.json: fast_q4_1_writer)."""
    sh = ggjt.SHAPES["tiny128"]
    path = str(tmp_path / "fast_q4_1.bin")
    ggjt.write_fast_q4_slice(path, sh, 0, 1, 0, wtype=ggjt.T_Q4_1)
    f = ggjt.read_file(path, sliced=True)
    t = f.tensors["layers.0.feed_forward.w2.weight"]
    assert t.ttype == ggjt.T_Q4_1 and t.nbytes == sh.n_embd * sh.n_ff // 32 * 20
    w = ggjt.dequantize_q4_1(np.frombuffer(f.read_raw("layers.0.attention.wq.weight"), np.uint8).reshape(sh.n_embd, -1, 20))
    assert abs(float(w.mean())) < 2e-3 and 0.7 < float(w.std()) * np.sqrt(sh.n_embd) < 1.3
    want = goldens.load("fast_q4_1_writer")
    port = oracle.PortSlice(path, 512)
    rng = np.random.default_rng(11)
    for i, n in enumerate((20, 1, 1)):
        x = rng.standard_normal((n, sh.n_embd), dtype=np.float32)
        b = port.forward(x)
        assert np.isfinite(b).all()
        goldens.check(b, want[i], "call %d" % i)
    port.close()
