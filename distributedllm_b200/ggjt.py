"""GGJT slice-file format: reader, writer, quantisers, synthetic models.

The on-disk format is the reference's own (it is the contract between
`provision` and the compute node), restated here from the byte layout:

* full model file   -- vendor/llama.cpp/convert.py:1008-1033 (header, vocab,
  tensor records) as read by distllm/slice_model.cpp:126-236: magic 'ggjt',
  version, SEVEN u32 hparams.
* slice file        -- distllm/slice_model.cpp:239-302 (writer) and
  distllm/tensor_processor.cpp:152-248 (reader): same, but EIGHT u32 hparams
  (`first_layer` inserted before `ftype`, `n_layer` = slice length).
* extra-layers file -- slice_model.cpp:341-347, 377-388: n_layer = 0,
  first_layer = 0xFFFFFFFF, tensors tok_embeddings/norm/output.

Quantisers restate ggml.c:941-975 (`quantize_row_q4_0_reference`) and
ggml.c:1100-1140 (`quantize_row_q8_0_reference`), the functions the reference's
`quantize` tool uses to create model files.
"""
from __future__ import annotations

import struct
from dataclasses import dataclass, field
from typing import BinaryIO, Dict, Iterable, List, Optional, Sequence, Tuple

import numpy as np

MAGIC_GGJT = 0x67676A74
FILE_VERSION = 3
NO_FIRST_LAYER = 0xFFFFFFFF

# ggml.h:265-281
T_F32, T_F16, T_Q4_0, T_Q4_1, T_Q8_0, T_Q6_K = 0, 1, 2, 3, 8, 14
# llama.h:108-115
FTYPE_F32, FTYPE_F16, FTYPE_Q4_0, FTYPE_Q4_1, FTYPE_Q8_0 = 0, 1, 2, 3, 7

QK = 32
TYPE_BLOCK = {T_F32: (1, 4), T_F16: (1, 2), T_Q4_0: (32, 18), T_Q4_1: (32, 20),
              T_Q8_0: (32, 34), T_Q6_K: (256, 210)}
TYPE_NAME = {T_F32: "f32", T_F16: "f16", T_Q4_0: "q4_0", T_Q4_1: "q4_1", T_Q8_0: "q8_0", T_Q6_K: "q6_K"}


def tensor_nbytes(ne: Sequence[int], ttype: int) -> int:
    """llama-util / llama_calc_tensor_size: product(ne) * type_size / block_size."""
    blk, sz = TYPE_BLOCK[ttype]
    n = 1
    for d in ne:
        n *= int(d)
    return n * sz // blk


def n_ff_for(n_embd: int, n_mult: int) -> int:
    """tensor_processor.cpp:1250."""
    return ((2 * (4 * n_embd) // 3 + n_mult - 1) // n_mult) * n_mult


# --------------------------------------------------------------------------- quantisers
def quantize_q4_0(x: np.ndarray) -> np.ndarray:
    """[rows, K] f32 -> [rows, K/32, 18] u8 (fp16 d, 16 nibble bytes). ggml.c:941-975."""
    x = np.ascontiguousarray(x, dtype=np.float32)
    rows, k = x.shape
    assert k % QK == 0
    xb = x.reshape(rows, k // QK, QK)
    idx = np.abs(xb).argmax(axis=2)            # first occurrence of amax, as `amax < fabsf(v)`
    mx = np.take_along_axis(xb, idx[..., None], axis=2)[..., 0]
    d = (mx / np.float32(-8)).astype(np.float32)
    with np.errstate(divide="ignore"):
        idv = np.where(d != 0, np.float32(1.0) / np.where(d != 0, d, np.float32(1)), np.float32(0)).astype(np.float32)
    xs = (xb * idv[..., None]).astype(np.float32)
    q = np.minimum(15, np.trunc((xs + np.float32(8.5)).astype(np.float32)).astype(np.int32)).astype(np.uint8)
    out = np.empty((rows, k // QK, 18), dtype=np.uint8)
    out[..., 0:2] = d.astype(np.float16).view(np.uint8).reshape(rows, k // QK, 2)
    out[..., 2:] = q[..., :16] | (q[..., 16:] << 4)
    return out


def dequantize_q4_0(blocks: np.ndarray) -> np.ndarray:
    """[rows, nb, 18] u8 -> [rows, nb*32] f32 (ggml.c dequantize_row_q4_0)."""
    rows, nb, _ = blocks.shape
    d = blocks[..., 0:2].copy().view(np.float16).astype(np.float32)[..., 0]
    qs = blocks[..., 2:]
    lo = (qs & 0x0F).astype(np.int32) - 8
    hi = (qs >> 4).astype(np.int32) - 8
    w = np.concatenate([lo, hi], axis=2).astype(np.float32) * d[..., None]
    return w.reshape(rows, nb * QK)


def quantize_q4_1(x: np.ndarray) -> np.ndarray:
    """[rows, K] f32 -> [rows, K/32, 20] u8 (fp16 d, fp16 min, 16 nibble bytes). ggml.c:982-1015."""
    x = np.ascontiguousarray(x, dtype=np.float32)
    rows, k = x.shape
    assert k % QK == 0
    xb = x.reshape(rows, k // QK, QK)
    mn, mx = xb.min(axis=2), xb.max(axis=2)
    d = ((mx - mn) / np.float32(15)).astype(np.float32)
    idv = np.where(d != 0, np.float32(1.0) / np.where(d != 0, d, np.float32(1)), np.float32(0)).astype(np.float32)
    xs = ((xb - mn[..., None]).astype(np.float32) * idv[..., None]).astype(np.float32)
    q = np.minimum(15, np.trunc((xs + np.float32(0.5)).astype(np.float32)).astype(np.int32)).astype(np.uint8)
    out = np.empty((rows, k // QK, 20), dtype=np.uint8)
    out[..., 0:2] = d.astype(np.float16).view(np.uint8).reshape(rows, k // QK, 2)
    out[..., 2:4] = mn.astype(np.float16).view(np.uint8).reshape(rows, k // QK, 2)
    out[..., 4:] = q[..., :16] | (q[..., 16:] << 4)
    return out


def dequantize_q4_1(blocks: np.ndarray) -> np.ndarray:
    """[rows, nb, 20] u8 -> [rows, nb*32] f32: nibble * d + m, two roundings (ggml.c:1543-1562)."""
    rows, nb, _ = blocks.shape
    d = blocks[..., 0:2].copy().view(np.float16).astype(np.float32)
    m = blocks[..., 2:4].copy().view(np.float16).astype(np.float32)
    qs = blocks[..., 4:]
    n = np.concatenate([qs & 0x0F, qs >> 4], axis=2).astype(np.float32)
    w = ((n * d).astype(np.float32) + m).astype(np.float32)
    return w.reshape(rows, nb * QK)


def quantize_q8_0(x: np.ndarray) -> np.ndarray:
    """[rows, K] f32 -> [rows, K/32, 34] u8. ggml.c:1100-1140 (reference variant: id=1/d, roundf)."""
    x = np.ascontiguousarray(x, dtype=np.float32)
    rows, k = x.shape
    xb = x.reshape(rows, k // QK, QK)
    amax = np.abs(xb).max(axis=2).astype(np.float32)
    d = (amax / np.float32(127)).astype(np.float32)
    idv = np.where(d != 0, np.float32(1.0) / np.where(d != 0, d, np.float32(1)), np.float32(0)).astype(np.float32)
    xs = (xb * idv[..., None]).astype(np.float32)
    q = (np.sign(xs) * np.floor(np.abs(xs) + np.float32(0.5))).astype(np.int8)   # roundf: half away from zero
    out = np.empty((rows, k // QK, 34), dtype=np.uint8)
    out[..., 0:2] = d.astype(np.float16).view(np.uint8).reshape(rows, k // QK, 2)
    out[..., 2:] = q.view(np.uint8)
    return out


def encode_tensor(x: np.ndarray, ttype: int) -> bytes:
    if ttype == T_F32:
        return np.ascontiguousarray(x, dtype=np.float32).tobytes()
    if ttype == T_F16:
        return np.ascontiguousarray(x, dtype=np.float32).astype(np.float16).tobytes()
    if ttype == T_Q4_0:
        return quantize_q4_0(x).tobytes()
    if ttype == T_Q4_1:
        return quantize_q4_1(x).tobytes()
    if ttype == T_Q8_0:
        return quantize_q8_0(x).tobytes()
    raise ValueError(f"cannot encode ggml type {ttype}")


# --------------------------------------------------------------------------- file model
@dataclass
class HParams:
    n_vocab: int
    n_embd: int
    n_mult: int
    n_head: int
    n_layer: int
    n_rot: int
    ftype: int
    first_layer: Optional[int] = None      # None => full-model header (7 fields)

    @property
    def n_ff(self) -> int:
        return n_ff_for(self.n_embd, self.n_mult)


@dataclass
class TensorRecord:
    name: str
    ttype: int
    ne: Tuple[int, ...]        # ne[0] = row length (inner dim), as stored
    offset: int                # file offset of raw data
    nbytes: int


@dataclass
class GGJTFile:
    hparams: HParams
    vocab: List[Tuple[bytes, float]]
    tensors: Dict[str, TensorRecord] = field(default_factory=dict)
    path: str = ""

    def read_raw(self, name: str) -> bytes:
        t = self.tensors[name]
        with open(self.path, "rb") as f:
            f.seek(t.offset)
            return f.read(t.nbytes)


def default_vocab(n_vocab: int) -> List[Tuple[bytes, float]]:
    """A small sentencepiece-shaped vocabulary: <unk>,<s>,</s>, 256 byte tokens, then pieces."""
    v: List[Tuple[bytes, float]] = [(b"<unk>", 0.0), (b"<s>", 0.0), (b"</s>", 0.0)]
    for b in range(256):
        if len(v) >= n_vocab:
            break
        v.append((bytes([b]) if b >= 0x20 and b < 0x7F else b"<0x%02X>" % b, 0.0))
    pieces = [b" ", b"e", b"t", b"a", b"th", b" t", b"he", b" the", b"in", b" a", b"er", b"an", b"re", b"on", b" s"]
    i = 0
    while len(v) < n_vocab:
        p = pieces[i % len(pieces)] + (b"" if i < len(pieces) else str(i).encode())
        v.append((p, -float(i + 1)))
        i += 1
    return v[:n_vocab]


def _write_header(f: BinaryIO, hp: HParams, vocab: Sequence[Tuple[bytes, float]]) -> None:
    f.write(struct.pack("<II", MAGIC_GGJT, FILE_VERSION))
    vals = [hp.n_vocab, hp.n_embd, hp.n_mult, hp.n_head, hp.n_layer, hp.n_rot]
    if hp.first_layer is not None:
        vals.append(hp.first_layer & 0xFFFFFFFF)
    vals.append(hp.ftype)
    f.write(struct.pack("<%dI" % len(vals), *vals))
    assert len(vocab) == hp.n_vocab
    for text, score in vocab:
        f.write(struct.pack("<I", len(text)))
        f.write(text)
        f.write(struct.pack("<f", score))


def _write_tensor(f: BinaryIO, name: str, ttype: int, ne: Sequence[int], raw: bytes) -> None:
    nm = name.encode("utf-8")
    f.write(struct.pack("<III", len(ne), len(nm), ttype))
    f.write(struct.pack("<%dI" % len(ne), *ne))
    f.write(nm)
    pad = (-f.tell()) & 31
    f.write(b"\0" * pad)
    assert len(raw) == tensor_nbytes(ne, ttype), (name, len(raw), tensor_nbytes(ne, ttype))
    f.write(raw)


def write_file(path: str, hp: HParams, vocab: Sequence[Tuple[bytes, float]],
               tensors: Iterable[Tuple[str, int, Sequence[int], bytes]]) -> None:
    with open(path, "wb") as f:
        _write_header(f, hp, vocab)
        for name, ttype, ne, raw in tensors:
            _write_tensor(f, name, ttype, ne, raw)


def read_file(path: str, sliced: Optional[bool] = None) -> GGJTFile:
    """Parse header + tensor directory (no data). `sliced`: 8-field header (slice / extra file);
    None = auto-detect (the interpretation whose vocab walk lands on a valid tensor record)."""
    with open(path, "rb") as f:
        data_size = f.seek(0, 2)
        f.seek(0)
        magic, version = struct.unpack("<II", f.read(8))
        if magic != MAGIC_GGJT or version not in (1, 2, 3):
            raise ValueError("unknown (magic, version) combination: %08x, %08x" % (magic, version))
        if sliced is None:
            sliced = _probe_sliced(path)
        f.seek(8)
        if sliced:
            nv, ne_, nm, nh, nl, nr, fl, ft = struct.unpack("<8I", f.read(32))
            hp = HParams(nv, ne_, nm, nh, nl, nr, ft, fl)
        else:
            nv, ne_, nm, nh, nl, nr, ft = struct.unpack("<7I", f.read(28))
            hp = HParams(nv, ne_, nm, nh, nl, nr, ft, None)
        vocab = []
        for _ in range(hp.n_vocab):
            (ln,) = struct.unpack("<I", f.read(4))
            text = f.read(ln)
            (score,) = struct.unpack("<f", f.read(4))
            vocab.append((text, score))
        out = GGJTFile(hp, vocab, {}, path)
        while f.tell() < data_size:
            n_dims, name_len, ttype = struct.unpack("<III", f.read(12))
            if n_dims < 1 or n_dims > 2:
                raise ValueError("tensor should not be %u-dimensional" % n_dims)
            ne = struct.unpack("<%dI" % n_dims, f.read(4 * n_dims))
            name = f.read(name_len).decode("utf-8")
            if ttype not in TYPE_BLOCK:
                raise ValueError("unrecognized tensor type %u" % ttype)
            f.seek((-f.tell()) & 31, 1)
            off = f.tell()
            nb = tensor_nbytes(ne, ttype)
            f.seek(nb, 1)
            out.tensors[name] = TensorRecord(name, ttype, tuple(ne), off, nb)
        return out


def _probe_sliced(path: str) -> bool:
    for sliced in (True, False):
        try:
            with open(path, "rb") as f:
                size = f.seek(0, 2)
                f.seek(8)
                n = 8 if sliced else 7
                vals = struct.unpack("<%dI" % n, f.read(4 * n))
                nv = vals[0]
                if nv > 10_000_000:
                    continue
                ok = True
                for _ in range(nv):
                    (ln,) = struct.unpack("<I", f.read(4))
                    if ln > 4096:
                        ok = False
                        break
                    f.seek(ln + 4, 1)
                if not ok:
                    continue
                if f.tell() == size:
                    return sliced
                n_dims, name_len, ttype = struct.unpack("<III", f.read(12))
                if 1 <= n_dims <= 2 and name_len < 256 and ttype in TYPE_BLOCK:
                    return sliced
        except struct.error:
            continue
    raise ValueError("not a GGJT file: %s" % path)


# --------------------------------------------------------------------------- slicing
LAYER_TENSORS = ("attention_norm.weight", "attention.wq.weight", "attention.wk.weight",
                 "attention.wv.weight", "attention.wo.weight", "ffn_norm.weight",
                 "feed_forward.w1.weight", "feed_forward.w2.weight", "feed_forward.w3.weight")


def slice_model(src_path: str, dst_path: str, layer_from: int, layer_to: int) -> None:
    """`slice_model slice a b` (slice_model.cpp:389-405, 350-358): keep tensors `layers.{a..b}.*`."""
    src = read_file(src_path, sliced=False)
    hp = src.hparams
    new_hp = HParams(hp.n_vocab, hp.n_embd, hp.n_mult, hp.n_head, layer_to - layer_from + 1, hp.n_rot,
                     hp.ftype, layer_from)
    prefixes = tuple("layers.%d." % i for i in range(layer_from, layer_to + 1))
    with open(dst_path, "wb") as f:
        _write_header(f, new_hp, src.vocab)
        for name, t in src.tensors.items():            # file order is preserved (dict keeps it)
            if name.startswith(prefixes):
                _write_tensor(f, name, t.ttype, t.ne, src.read_raw(name))


def extract_extra_layers(src_path: str, dst_path: str) -> None:
    """`slice_model extra_layers` (slice_model.cpp:341-347, 377-388)."""
    src = read_file(src_path, sliced=False)
    hp = src.hparams
    new_hp = HParams(hp.n_vocab, hp.n_embd, hp.n_mult, hp.n_head, 0, hp.n_rot, hp.ftype, NO_FIRST_LAYER)
    with open(dst_path, "wb") as f:
        _write_header(f, new_hp, src.vocab)
        for name, t in src.tensors.items():
            if name.startswith(("norm", "output", "tok_embeddings")):
                _write_tensor(f, name, t.ttype, t.ne, src.read_raw(name))


# --------------------------------------------------------------------------- synthetic models
@dataclass
class ModelShape:
    n_vocab: int
    n_embd: int
    n_mult: int
    n_head: int
    n_layer: int

    @property
    def n_ff(self) -> int:
        return n_ff_for(self.n_embd, self.n_mult)


SHAPES = {
    "tiny":   ModelShape(512, 256, 32, 4, 4),        # d_head 64, n_ff 704
    "tiny3b": ModelShape(512, 800, 32, 8, 3),        # d_head 100 (OpenLLaMA-3B-like head), n_ff 2144 = 67 blocks
    "tiny128": ModelShape(512, 512, 32, 4, 3),       # d_head 128 (the 7B/13B head size), n_ff 1376 = 43 blocks
    "tiny128b": ModelShape(512, 512, 64, 4, 2),      # d_head 128, n_ff 1408: every matrix is a whole number of 128-row MMA tiles
    "tiny128c": ModelShape(512, 512, 320, 4, 2),     # d_head 128, n_ff 1600 = 12.5 x 128: w2's last 128-wide K block is half empty
    "3b":     ModelShape(32000, 3200, 216, 32, 26),  # OpenLLaMA-3B: n_ff 8640
    "7b":     ModelShape(32000, 4096, 256, 32, 32),
    "13b":    ModelShape(32000, 5120, 256, 40, 40),
}


def _gauss_weights(rng: np.random.Generator, rows: int, k: int, scale: float) -> np.ndarray:
    return (rng.standard_normal((rows, k), dtype=np.float32) * np.float32(scale)).astype(np.float32)


def synth_layer_tensors(shape: ModelShape, layer: int, wtype: int, seed: int):
    """Yield (name, type, ne, raw) for one transformer layer: N(0, 1/sqrt(fan_in)) matrices,
    norm weights 1 + 0.1*N(0,1) (SURVEY.md 8d)."""
    rng = np.random.default_rng([seed, layer])
    e, ff = shape.n_embd, shape.n_ff
    pre = "layers.%d." % layer
    dims = {"attention.wq.weight": (e, e), "attention.wk.weight": (e, e), "attention.wv.weight": (e, e),
            "attention.wo.weight": (e, e), "feed_forward.w1.weight": (ff, e), "feed_forward.w2.weight": (e, ff),
            "feed_forward.w3.weight": (ff, e)}
    for nm in LAYER_TENSORS:
        if nm.endswith("norm.weight"):
            w = (1.0 + 0.1 * rng.standard_normal(e)).astype(np.float32)
            yield pre + nm, T_F32, (e,), w.tobytes()
        else:
            rows, k = dims[nm]
            w = _gauss_weights(rng, rows, k, 1.0 / np.sqrt(k))
            yield pre + nm, wtype, (k, rows), encode_tensor(w, wtype)


_FTYPE_OF = {T_F32: FTYPE_F32, T_F16: FTYPE_F16, T_Q4_0: FTYPE_Q4_0, T_Q4_1: FTYPE_Q4_1, T_Q8_0: FTYPE_Q8_0}


def write_synth_slice(path: str, shape: ModelShape, layer_from: int, layer_to: int, wtype: int = T_Q4_0,
                      seed: int = 0, vocab: Optional[Sequence[Tuple[bytes, float]]] = None) -> None:
    """Write a slice file for layers [layer_from, layer_to] straight from the generator (the
    result is byte-identical to full-model -> slice_model, because every layer is seeded
    independently)."""
    vocab = list(vocab) if vocab is not None else default_vocab(shape.n_vocab)
    hp = HParams(shape.n_vocab, shape.n_embd, shape.n_mult, shape.n_head, layer_to - layer_from + 1,
                 shape.n_embd // shape.n_head, _FTYPE_OF[wtype], layer_from)
    with open(path, "wb") as f:
        _write_header(f, hp, vocab)
        for layer in range(layer_from, layer_to + 1):
            for name, t, ne, raw in synth_layer_tensors(shape, layer, wtype, seed):
                _write_tensor(f, name, t, ne, raw)


def synth_extra_tensors(shape: ModelShape, wtype: int, seed: int):
    rng = np.random.default_rng([seed, 1_000_003])
    e, v = shape.n_embd, shape.n_vocab
    emb = _gauss_weights(rng, v, e, 1.0)
    yield "tok_embeddings.weight", wtype, (e, v), encode_tensor(emb, wtype)
    yield "norm.weight", T_F32, (e,), (1.0 + 0.1 * rng.standard_normal(e)).astype(np.float32).tobytes()
    out = _gauss_weights(rng, v, e, 1.0 / np.sqrt(e))
    yield "output.weight", wtype, (e, v), encode_tensor(out, wtype)


def write_synth_extra(path: str, shape: ModelShape, wtype: int = T_Q4_0, seed: int = 0,
                      vocab: Optional[Sequence[Tuple[bytes, float]]] = None) -> None:
    vocab = list(vocab) if vocab is not None else default_vocab(shape.n_vocab)
    hp = HParams(shape.n_vocab, shape.n_embd, shape.n_mult, shape.n_head, 0, shape.n_embd // shape.n_head,
                 _FTYPE_OF[wtype], NO_FIRST_LAYER)
    write_file(path, hp, vocab, synth_extra_tensors(shape, wtype, seed))


def write_synth_full(path: str, shape: ModelShape, wtype: int = T_F32, seed: int = 0,
                     vocab: Optional[Sequence[Tuple[bytes, float]]] = None) -> None:
    """A full (un-sliced) model file, for feeding the reference `quantize` / `slice_model`."""
    vocab = list(vocab) if vocab is not None else default_vocab(shape.n_vocab)
    hp = HParams(shape.n_vocab, shape.n_embd, shape.n_mult, shape.n_head, shape.n_layer,
                 shape.n_embd // shape.n_head, _FTYPE_OF[wtype], None)

    def gen():
        ex = {n: (t, ne, raw) for n, t, ne, raw in synth_extra_tensors(shape, wtype, seed)}
        yield ("tok_embeddings.weight",) + ex["tok_embeddings.weight"]
        yield ("norm.weight",) + ex["norm.weight"]
        yield ("output.weight",) + ex["output.weight"]
        for layer in range(shape.n_layer):
            yield from synth_layer_tensors(shape, layer, wtype, seed)

    write_file(path, hp, vocab, gen())


_POOL_BLOCKS = 1 << 21          # 2 Mi blocks = 36 MiB per pool


def _fast_q4_pool(seed: int, k: int) -> np.ndarray:
    """A pool of random Q4_0 blocks: uniform nibbles, fp16 scale = +-mag*(1 + j/512), j in [-128,128),
    mag = 1/(4.6*sqrt(fan_in)) so that weights have std ~ 1/sqrt(fan_in)."""
    rng = np.random.default_rng([seed, k, 77])
    blocks = rng.integers(0, 256, size=(_POOL_BLOCKS, 18), dtype=np.uint8)
    mag = 1.0 / (4.6 * np.sqrt(k))
    lut = (mag * (1.0 + (np.arange(256, dtype=np.float32) - 128.0) / 512.0)).astype(np.float16).view(np.uint16)
    d = lut[blocks[:, 1]] | ((blocks[:, 0] & 1).astype(np.uint16) << 15)
    blocks[:, 0] = (d & 0xFF).astype(np.uint8)
    blocks[:, 1] = (d >> 8).astype(np.uint8)
    return blocks


def _fast_q41_pool(seed: int, k: int) -> np.ndarray:
    """Q4_1 twin of _fast_q4_pool: 20-byte blocks, fp16 step d = mag*(1 + j/512) > 0 and fp16 minimum
    m = -(7.5 + i/256)*d (i in [-128,128)), so nibble*d + m is centred with std ~ 1/sqrt(fan_in)."""
    rng = np.random.default_rng([seed, k, 79])
    blocks = rng.integers(0, 256, size=(_POOL_BLOCKS, 20), dtype=np.uint8)
    mag = 1.0 / (4.6 * np.sqrt(k))
    d = (mag * (1.0 + (blocks[:, 1].astype(np.float32) - 128.0) / 512.0)).astype(np.float16)
    m = (-(7.5 + (blocks[:, 3].astype(np.float32) - 128.0) / 256.0) * d.astype(np.float32)).astype(np.float16)
    blocks[:, 0:2] = d.view(np.uint8).reshape(-1, 2)
    blocks[:, 2:4] = m.view(np.uint8).reshape(-1, 2)
    return blocks


def write_fast_q4_slice(path: str, shape: ModelShape, layer_from: int, layer_to: int, seed: int = 0,
                        wtype: int = T_Q4_0) -> int:
    """Large-model generator for benchmarks.  Quantising 6.5e9 Gaussians takes minutes, so Q4_0
    blocks are written directly: each matrix is a window (at a per-tensor pseudo-random block
    offset, wrapping) into a 36 MiB pool of random blocks built once per fan-in.  The file is the
    ground truth for both the B200 path and the CPU reference, so the distribution only has to keep
    activations finite; any layer range of the same (shape, seed) is reproducible.  Returns bytes written.
    `wtype` = T_Q4_1 writes 20-byte Q4_1 blocks from _fast_q41_pool instead."""
    assert wtype in (T_Q4_0, T_Q4_1)
    bsz = TYPE_BLOCK[wtype][1]
    vocab = default_vocab(shape.n_vocab)
    hp = HParams(shape.n_vocab, shape.n_embd, shape.n_mult, shape.n_head, layer_to - layer_from + 1,
                 shape.n_embd // shape.n_head, _FTYPE_OF[wtype], layer_from)
    e, ff = shape.n_embd, shape.n_ff
    dims = {"attention.wq.weight": (e, e), "attention.wk.weight": (e, e), "attention.wv.weight": (e, e),
            "attention.wo.weight": (e, e), "feed_forward.w1.weight": (ff, e), "feed_forward.w2.weight": (e, ff),
            "feed_forward.w3.weight": (ff, e)}
    make_pool = _fast_q4_pool if wtype == T_Q4_0 else _fast_q41_pool
    pools = {k: memoryview(make_pool(seed, k)).cast("B") for k in sorted({e, ff})}
    pool_bytes = _POOL_BLOCKS * bsz
    with open(path, "wb") as f:
        _write_header(f, hp, vocab)
        for layer in range(layer_from, layer_to + 1):
            pre = "layers.%d." % layer
            rng = np.random.default_rng([seed, layer, 78])
            for nm in LAYER_TENSORS:
                if nm.endswith("norm.weight"):
                    w = (1.0 + 0.1 * rng.standard_normal(e)).astype(np.float32)
                    _write_tensor(f, pre + nm, T_F32, (e,), w.tobytes())
                    continue
                rows, k = dims[nm]
                nbytes = rows * k // QK * bsz
                start = int(rng.integers(0, _POOL_BLOCKS)) * bsz
                name = (pre + nm).encode("utf-8")
                f.write(struct.pack("<III", 2, len(name), wtype))
                f.write(struct.pack("<2I", k, rows))
                f.write(name)
                f.write(b"\0" * ((-f.tell()) & 31))
                left, pos = nbytes, start
                while left:
                    n = min(left, pool_bytes - pos)
                    f.write(pools[k][pos:pos + n])
                    left -= n
                    pos = 0
        return f.tell()


def write_fast_f16_slice(path: str, shape: ModelShape, layer_from: int, layer_to: int, seed: int = 0) -> int:
    """F16 twin of write_fast_q4_slice (BASELINE config 4: un-quantised 7B): each matrix is a window into a pool of
    16 Mi fp16 values ~ N(0, 1/fan_in), one pool per fan-in.  Returns bytes written."""
    vocab = default_vocab(shape.n_vocab)
    hp = HParams(shape.n_vocab, shape.n_embd, shape.n_mult, shape.n_head, layer_to - layer_from + 1,
                 shape.n_embd // shape.n_head, FTYPE_F16, layer_from)
    e, ff = shape.n_embd, shape.n_ff
    dims = {"attention.wq.weight": (e, e), "attention.wk.weight": (e, e), "attention.wv.weight": (e, e),
            "attention.wo.weight": (e, e), "feed_forward.w1.weight": (ff, e), "feed_forward.w2.weight": (e, ff),
            "feed_forward.w3.weight": (ff, e)}
    n_pool = 1 << 24
    pools = {}
    for k in sorted({e, ff}):
        rng = np.random.default_rng([seed, k, 79])
        pools[k] = memoryview((rng.standard_normal(n_pool, dtype=np.float32) / np.float32(np.sqrt(k))).astype(np.float16)).cast("B")
    pool_bytes = n_pool * 2
    with open(path, "wb") as f:
        _write_header(f, hp, vocab)
        for layer in range(layer_from, layer_to + 1):
            pre = "layers.%d." % layer
            rng = np.random.default_rng([seed, layer, 80])
            for nm in LAYER_TENSORS:
                if nm.endswith("norm.weight"):
                    w = (1.0 + 0.1 * rng.standard_normal(e)).astype(np.float32)
                    _write_tensor(f, pre + nm, T_F32, (e,), w.tobytes())
                    continue
                rows, k = dims[nm]
                nbytes = rows * k * 2
                start = int(rng.integers(0, n_pool)) * 2
                name = (pre + nm).encode("utf-8")
                f.write(struct.pack("<III", 2, len(name), T_F16))
                f.write(struct.pack("<2I", k, rows))
                f.write(name)
                f.write(b"\0" * ((-f.tell()) & 31))
                left, pos = nbytes, start
                while left:
                    n = min(left, pool_bytes - pos)
                    f.write(pools[k][pos:pos + n])
                    left -= n
                    pos = 0
        return f.tell()


def write_fast_q4_extra(path: str, shape: ModelShape, seed: int = 0) -> int:
    """Extra-layers file (tok_embeddings, norm, output -- all Q4_0 / f32) for the large shapes, from the same block
    pool as write_fast_q4_slice.  Embedding rows come out with std ~ 1/sqrt(n_embd); the first RMSNorm rescales them."""
    vocab = default_vocab(shape.n_vocab)
    hp = HParams(shape.n_vocab, shape.n_embd, shape.n_mult, shape.n_head, 0, shape.n_embd // shape.n_head,
                 FTYPE_Q4_0, NO_FIRST_LAYER)
    e, v = shape.n_embd, shape.n_vocab
    pool = memoryview(_fast_q4_pool(seed, e)).cast("B")
    pool_bytes = _POOL_BLOCKS * 18
    rng = np.random.default_rng([seed, 81])
    with open(path, "wb") as f:
        _write_header(f, hp, vocab)
        for nm in ("tok_embeddings.weight", "norm.weight", "output.weight"):
            if nm == "norm.weight":
                _write_tensor(f, nm, T_F32, (e,), (1.0 + 0.1 * rng.standard_normal(e)).astype(np.float32).tobytes())
                continue
            name = nm.encode("utf-8")
            f.write(struct.pack("<III", 2, len(name), T_Q4_0))
            f.write(struct.pack("<2I", e, v))
            f.write(name)
            f.write(b"\0" * ((-f.tell()) & 31))
            left, pos = v * e // QK * 18, int(rng.integers(0, _POOL_BLOCKS)) * 18
            while left:
                n = min(left, pool_bytes - pos)
                f.write(pool[pos:pos + n])
                left -= n
                pos = 0
        return f.tell()
