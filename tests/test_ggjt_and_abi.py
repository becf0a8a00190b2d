"""Slice-file format library and the C-ABI surface (no GPU: the library must LOAD and export every symbol
include/b200_slice.h declares, and fail loudly -- not fall back -- when there is no device)."""
import ctypes
import os
import re

import numpy as np

from distributedllm_b200 import ggjt

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_q4_0_quantizer_layout_and_roundtrip():
    rng = np.random.default_rng(0)
    x = rng.standard_normal((4, 64)).astype(np.float32)
    q = ggjt.quantize_q4_0(x)
    assert q.shape == (4, 2, 18)
    d = q[..., :2].copy().view(np.float16).astype(np.float32)[..., 0]
    xb = x.reshape(4, 2, 32)
    idx = np.abs(xb).argmax(2)
    mx = np.take_along_axis(xb, idx[..., None], 2)[..., 0]
    assert np.array_equal(d, (mx / np.float32(-8)).astype(np.float16).astype(np.float32))   # d = max / -8 (ggml.c:957)
    y = ggjt.dequantize_q4_0(q)
    assert np.sqrt(np.mean((x - y) ** 2)) < 0.12         # vendor test-quantize-fns.cpp bounds the same RMSE for unit Gaussians
    # the element with the largest magnitude maps to nibble 0 (-8 * d)
    lo = (q[..., 2:] & 0x0F).astype(int); hi = (q[..., 2:] >> 4).astype(int)
    nib = np.concatenate([lo, hi], 2)
    assert (np.take_along_axis(nib, idx[..., None], 2)[..., 0] == 0).all()


def test_slice_file_roundtrip(tmp_path):
    sh = ggjt.SHAPES["tiny"]
    p = str(tmp_path / "s.bin")
    ggjt.write_synth_slice(p, sh, 1, 2, ggjt.T_Q4_0, seed=0)
    f = ggjt.read_file(p)
    hp = f.hparams
    assert (hp.n_embd, hp.n_head, hp.n_layer, hp.first_layer, hp.ftype, hp.n_ff) == (256, 4, 2, 1, ggjt.FTYPE_Q4_0, 704)
    assert len(f.tensors) == 18 and len(f.vocab) == 512
    t = f.tensors["layers.2.feed_forward.w2.weight"]
    assert t.ne == (704, 256) and t.ttype == ggjt.T_Q4_0 and t.offset % 32 == 0 and t.nbytes == 704 * 256 // 32 * 18
    assert f.tensors["layers.1.attention_norm.weight"].ttype == ggjt.T_F32


def test_slicer_equals_direct_writer(tmp_path):
    sh = ggjt.SHAPES["tiny"]
    full, a, b, e1, e2 = (str(tmp_path / n) for n in ("full.bin", "a.bin", "b.bin", "e1.bin", "e2.bin"))
    ggjt.write_synth_full(full, sh, ggjt.T_Q4_0, seed=0)
    ggjt.slice_model(full, a, 1, 2)
    ggjt.write_synth_slice(b, sh, 1, 2, ggjt.T_Q4_0, seed=0)
    assert open(a, "rb").read() == open(b, "rb").read()
    ggjt.extract_extra_layers(full, e1)
    ggjt.write_synth_extra(e2, sh, ggjt.T_Q4_0, seed=0)
    assert open(e1, "rb").read() == open(e2, "rb").read()
    assert ggjt.read_file(e1).hparams.first_layer == ggjt.NO_FIRST_LAYER


def test_fast_generator_writes_a_loadable_slice(tmp_path):
    from oracle import oracle
    sh = ggjt.ModelShape(512, 256, 32, 2, 2)
    p = str(tmp_path / "fast.bin")
    n = ggjt.write_fast_q4_slice(p, sh, 0, 1, seed=0)
    assert n == os.path.getsize(p)
    s = oracle.PortSlice(p, 32)
    y = s.forward(np.random.default_rng(0).standard_normal((3, 256), dtype=np.float32))
    assert np.isfinite(y).all() and np.abs(y).max() < 100


def _header_symbols():
    text = open(os.path.join(ROOT, "include", "b200_slice.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(b200_[a-z0-9_]+)\s*\(", text)))


def test_library_exports_every_declared_symbol():
    from distributedllm_b200 import capi
    lib = capi.lib()
    names = _header_symbols()
    assert len(names) >= 30
    for n in names:
        assert hasattr(lib, n), "libb200slice.so does not export %s" % n
    assert b"sm_100a" in lib.b200_version()


def test_no_cpu_fallback():
    """Without a B200 every entry point refuses; nothing silently routes to a CPU path."""
    import subprocess, sys
    code = ("import sys; sys.path.insert(0, %r)\n"
            "from distributedllm_b200 import capi\n"
            "try:\n    capi.Slice('/nonexistent.bin')\nexcept capi.B200Error as e:\n    print('code', e.code)\n" % ROOT)
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    out = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, timeout=120)
    assert "code 3" in out.stdout, out.stdout + out.stderr      # B200_ENODEV


def test_product_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "distributedllm_b200")
    for dirpath, _, files in os.walk(pkg):
        for fn in files:
            if fn.endswith((".py", ".cu", ".cuh", ".cpp", ".hpp", ".h")):
                src = open(os.path.join(dirpath, fn), errors="replace").read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b", src, flags=re.M), fn
                assert "liboracle" not in src and "libllmref" not in src, fn


def test_fast_writers_produce_loadable_reference_format_files(tmp_path):
    """The pool-based generators used for the large shapes (bench, full-size tests) write the same container the
    reference's slice_model writes: header + first_layer, tensor directory, 32-byte aligned payloads of the right size."""
    sh = ggjt.ModelShape(512, 256, 32, 4, 3)
    q4, f16, ex = str(tmp_path / "q4.bin"), str(tmp_path / "f16.bin"), str(tmp_path / "extra.bin")
    n = ggjt.write_fast_q4_slice(q4, sh, 1, 2, seed=7)
    assert n == os.path.getsize(q4)
    f = ggjt.read_file(q4, sliced=True)
    assert f.hparams.n_layer == 2 and f.hparams.first_layer == 1 and len(f.tensors) == 18
    w1 = f.tensors["layers.2.feed_forward.w1.weight"]
    assert w1.ttype == ggjt.T_Q4_0 and tuple(w1.ne) == (sh.n_embd, sh.n_ff) and w1.offset % 32 == 0
    assert w1.nbytes == sh.n_embd * sh.n_ff // 32 * 18
    # deterministic, and any layer range of the same (shape, seed) carries the same bytes for a given layer
    ggjt.write_fast_q4_slice(str(tmp_path / "q4b.bin"), sh, 2, 2, seed=7)
    g = ggjt.read_file(str(tmp_path / "q4b.bin"), sliced=True)
    a = open(q4, "rb").read()
    b = open(str(tmp_path / "q4b.bin"), "rb").read()
    t2 = g.tensors["layers.2.feed_forward.w1.weight"]
    assert a[w1.offset:w1.offset + w1.nbytes] == b[t2.offset:t2.offset + t2.nbytes]
    ggjt.write_fast_f16_slice(f16, sh, 0, 0, seed=7)
    h = ggjt.read_file(f16, sliced=True)
    wq = h.tensors["layers.0.attention.wq.weight"]
    assert wq.ttype == ggjt.T_F16 and wq.nbytes == sh.n_embd * sh.n_embd * 2
    vals = np.frombuffer(open(f16, "rb").read()[wq.offset:wq.offset + wq.nbytes], np.float16).astype(np.float32)
    assert np.isfinite(vals).all() and 0.5 < vals.std() * np.sqrt(sh.n_embd) < 2.0
    ggjt.write_fast_q4_extra(ex, sh, seed=7)
    e = ggjt.read_file(ex, sliced=True)
    assert list(e.tensors) == ["tok_embeddings.weight", "norm.weight", "output.weight"] and e.hparams.n_layer == 0


def test_q4_1_quantizer_is_the_reference_quantize_tool(tmp_path):
    """ggjt.quantize_q4_1 (ggml.c:982-1015 restated) against the reference's own `quantize ... q4_1` binary, byte for byte
    (reference_runs.json: quantize_q4_1 holds the SHA-256 of every Q4_1 tensor the tool wrote from this file)."""
    import hashlib
    from oracle import goldens
    want = goldens.load("quantize_q4_1")
    sh = ggjt.SHAPES["tiny3b"]                                   # n_embd = 800: output.weight stays Q4_1 (not Q6_K)
    full = str(tmp_path / "f32.bin")
    ggjt.write_synth_full(full, sh, ggjt.T_F32, seed=0)
    a = ggjt.read_file(full)
    for name, digest in want.items():
        t = a.tensors[name]
        src = np.frombuffer(a.read_raw(name), np.float32).reshape(t.ne[1], t.ne[0])
        assert hashlib.sha256(ggjt.quantize_q4_1(src).tobytes()).hexdigest() == digest, name
    assert len(want) == 2 + 7 * sh.n_layer
