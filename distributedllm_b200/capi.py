"""ctypes binding of libb200slice.so (include/b200_slice.h).  No torch, no CPU fallback:
importing works anywhere, every call needs a B200."""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libb200slice.so")

ERRORS = {1: "EINVAL", 2: "EFILE", 3: "ENODEV", 4: "ECUDA", 5: "ECONTEXT", 6: "ENCCL"}


class B200Error(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__("b200 error %d (%s): %s" % (code, ERRORS.get(code, "?"), msg))
        self.code = code


class SliceInfo(C.Structure):
    _fields_ = [(n, C.c_int32) for n in ("n_embd", "n_head", "n_ff", "n_layer", "first_layer", "n_ctx", "n_past",
                                          "weight_type", "device")] + [("weight_bytes", C.c_int64),
                                                                        ("kv_bytes_per_pos", C.c_int64)]


_lib: Optional[C.CDLL] = None


def lib() -> C.CDLL:
    """Load the native library; raises if it has not been built (there is no fallback)."""
    global _lib
    if _lib is None:
        if not os.path.isfile(LIB_PATH):
            raise ImportError("libb200slice.so is not built: run `python -m distributedllm_b200.build`")
        L = C.CDLL(LIB_PATH)
        vp, ci, cf = C.c_void_p, C.c_int, C.c_float
        L.b200_last_error.restype = C.c_char_p
        L.b200_version.restype = C.c_char_p
        L.b200_slice_load.argtypes = [C.c_char_p, ci, ci, C.POINTER(vp)]
        L.b200_slice_load_ex.argtypes = [C.c_char_p, ci, ci, ci, C.POINTER(vp)]
        L.b200_session_count.argtypes = [vp]
        L.b200_session_n_past.argtypes = [vp, ci]
        L.b200_session_clear.argtypes = [vp, ci]
        L.b200_session_rewind.argtypes = [vp, ci, ci]
        L.b200_session_forward.argtypes = [vp, ci, vp, ci, vp]
        L.b200_session_forward_device.argtypes = [vp, ci, vp, ci, vp, ci]
        L.b200_batch_forward.argtypes = [vp, vp, ci, vp, vp]
        L.b200_batch_forward_device.argtypes = [vp, vp, ci, vp, vp, ci]
        L.b200_mixed_forward.argtypes = [vp, vp, vp, ci, vp, vp]
        L.b200_mixed_forward_device.argtypes = [vp, vp, vp, ci, vp, vp, ci]
        L.b200_slice_unload.argtypes = [vp]
        L.b200_slice_clear.argtypes = [vp]
        L.b200_slice_rewind.argtypes = [vp, ci]
        L.b200_slice_info.argtypes = [vp, C.POINTER(SliceInfo)]
        L.b200_slice_forward.argtypes = [vp, vp, ci, vp]
        L.b200_slice_forward_device.argtypes = [vp, vp, ci, vp, ci]
        L.b200_slice_sync.argtypes = [vp]
        L.b200_slice_last_ms.argtypes = [vp]
        L.b200_slice_last_ms.restype = cf
        L.b200_slice_launch_count.argtypes = [vp]
        L.b200_slice_launch_count.restype = C.c_int64
        L.b200_slice_set_fast_prefill.argtypes = [vp, ci, ci]
        L.b200_slice_mark.argtypes = [vp, ci]
        L.b200_slice_mark_elapsed_ms.argtypes = [vp]
        L.b200_slice_mark_elapsed_ms.restype = cf
        L.b200_slice_profile.argtypes = [vp, ci]
        L.b200_slice_profile_read.argtypes = [vp, vp, vp, ci]
        L.b200_debug_read.argtypes = [vp, ci, C.c_size_t, C.c_size_t, vp]
        L.b200_debug_trace_enable.argtypes = [vp, ci]
        L.b200_debug_skip_attention.argtypes = [vp, ci]
        L.b200_debug_trace_read.argtypes = [vp, vp, vp, vp, ci]
        L.b200_slice_dev_in.argtypes = [vp]
        L.b200_slice_dev_in.restype = vp
        L.b200_slice_dev_out.argtypes = [vp]
        L.b200_slice_dev_out.restype = vp
        L.b200_pipeline_result.argtypes = [vp]
        L.b200_pipeline_result.restype = vp
        L.b200_device_init.argtypes = [ci]
        L.b200_debug_ptrace_read.argtypes = [vp, vp, C.c_size_t]
        for name, args in (("b200_pipeline_unique_id", [vp]), ("b200_pipeline_init", [vp, ci, ci, vp]),
                           ("b200_pipeline_step", [vp, vp, ci, ci]),
                           ("b200_pipeline_mailbox_export", [vp, vp]), ("b200_pipeline_mailbox_connect", [vp, vp, ci]),
                           ("b200_pipeline_collect", [vp, ci, vp]), ("b200_pipeline_pingpong", [vp, ci, ci, vp]), ("b200_pipeline_transport", [vp]), ("b200_pipeline_set_transport", [vp, ci]), ("b200_pipeline_error", [vp]),
                           ("b200_pipeline_step_session", [vp, ci, vp, ci, ci]), ("b200_pipeline_step_batch", [vp, vp, ci, vp, ci]),
                           ("b200_pipeline_step_mixed", [vp, vp, vp, ci, vp, ci]), ("b200_pipeline_destroy", [vp]),
                           ("b200_extra_load", [C.c_char_p, ci, C.POINTER(vp)]), ("b200_extra_unload", [vp]),
                           ("b200_extra_dims", [vp, C.POINTER(ci), C.POINTER(ci)]),
                           ("b200_extra_embed", [vp, vp, ci, vp]), ("b200_extra_logits", [vp, vp, ci, ci, vp]),
                           ("b200_extra_next_token", [vp, vp, ci, C.POINTER(C.c_int32)]),
                           ("b200_extra_tokenize", [vp, C.c_char_p, vp, ci]),
                           ("b200_debug_fast_matmul", [vp, ci, ci, ci, vp, ci, vp, vp, vp])):
            if hasattr(L, name):
                getattr(L, name).argtypes = args
        if hasattr(L, "b200_extra_token_text"):
            L.b200_extra_token_text.argtypes = [vp, C.c_int32, C.POINTER(ci)]
            L.b200_extra_token_text.restype = C.POINTER(C.c_char)
        _lib = L
    return _lib


def check(rc: int) -> None:
    if rc != 0:
        raise B200Error(rc, (lib().b200_last_error() or b"").decode("utf-8", "replace"))


def _ptr(a: np.ndarray) -> C.c_void_p:
    return C.c_void_p(a.ctypes.data)


def _segments(sessions, n_tokens):
    ids = np.ascontiguousarray(sessions, dtype=np.int32).reshape(-1)
    lens = np.ascontiguousarray(n_tokens, dtype=np.int32).reshape(-1)
    if ids.shape != lens.shape:
        raise ValueError("mixed step: %d sessions but %d token counts" % (ids.size, lens.size))
    return ids, lens


class Slice:
    """One slice resident on one GPU (mirrors llm.load_slice / propagate_forward / clear_context)."""

    def __init__(self, path: str, device: int = 0, n_ctx: int = 0, n_sessions: int = 1):
        self._h = C.c_void_p()
        check(lib().b200_slice_load_ex(os.fsencode(path), device, n_ctx, n_sessions, C.byref(self._h)))
        self.info = self._info()
        self.n_sessions = n_sessions

    # ---- sessions / batched steps (additive API, include/b200_slice.h) ----
    def session_forward(self, session: int, x: np.ndarray) -> np.ndarray:
        x = np.ascontiguousarray(x, dtype=np.float32).reshape(-1, self.n_embd)
        out = np.empty_like(x)
        check(lib().b200_session_forward(self._h, session, _ptr(x), x.shape[0], _ptr(out)))
        return out

    def batch_forward(self, sessions, x: np.ndarray) -> np.ndarray:
        """One token for each listed session: x is [len(sessions)][n_embd]."""
        ids = np.ascontiguousarray(sessions, dtype=np.int32)
        x = np.ascontiguousarray(x, dtype=np.float32).reshape(len(ids), self.n_embd)
        out = np.empty_like(x)
        check(lib().b200_batch_forward(self._h, _ptr(ids), len(ids), _ptr(x), _ptr(out)))
        return out

    def batch_forward_device(self, sessions, d_in: int, d_out: int, sync: bool = False) -> None:
        ids = np.ascontiguousarray(sessions, dtype=np.int32)
        check(lib().b200_batch_forward_device(self._h, _ptr(ids), len(ids), C.c_void_p(d_in), C.c_void_p(d_out), int(sync)))

    def mixed_forward(self, sessions, n_tokens, x: np.ndarray) -> np.ndarray:
        """n_tokens[i] tokens of sessions[i] in one pass: x is [sum(n_tokens)][n_embd], the segments back to back."""
        ids, lens = _segments(sessions, n_tokens)
        x = np.ascontiguousarray(x, dtype=np.float32).reshape(int(lens.sum()), self.n_embd)
        out = np.empty_like(x)
        check(lib().b200_mixed_forward(self._h, _ptr(ids), _ptr(lens), len(ids), _ptr(x), _ptr(out)))
        return out

    def mixed_forward_device(self, sessions, n_tokens, d_in: int, d_out: int, sync: bool = False) -> None:
        ids, lens = _segments(sessions, n_tokens)
        check(lib().b200_mixed_forward_device(self._h, _ptr(ids), _ptr(lens), len(ids), C.c_void_p(d_in), C.c_void_p(d_out), int(sync)))

    def session_n_past(self, session: int) -> int:
        return lib().b200_session_n_past(self._h, session)

    def session_clear(self, session: int = -1) -> None:
        check(lib().b200_session_clear(self._h, session))

    def session_rewind(self, session: int, n_past: int) -> None:
        check(lib().b200_session_rewind(self._h, session, n_past))

    def _info(self) -> SliceInfo:
        i = SliceInfo()
        check(lib().b200_slice_info(self._h, C.byref(i)))
        return i

    @property
    def n_embd(self) -> int:
        return self.info.n_embd

    @property
    def n_past(self) -> int:
        return self._info().n_past

    @property
    def handle(self) -> C.c_void_p:
        return self._h

    def forward(self, x: np.ndarray) -> np.ndarray:
        """HOST buffers in and out: [n_tokens][n_embd] float32."""
        x = np.ascontiguousarray(x, dtype=np.float32).reshape(-1, self.n_embd)
        out = np.empty_like(x)
        check(lib().b200_slice_forward(self._h, _ptr(x), x.shape[0], _ptr(out)))
        return out

    def forward_device(self, d_in: int, n_tokens: int, d_out: int, sync: bool = False) -> None:
        check(lib().b200_slice_forward_device(self._h, C.c_void_p(d_in), n_tokens, C.c_void_p(d_out), int(sync)))

    def sync(self) -> None:
        check(lib().b200_slice_sync(self._h))

    def clear_context(self) -> None:
        check(lib().b200_slice_clear(self._h))

    def rewind(self, n_past: int) -> None:
        check(lib().b200_slice_rewind(self._h, n_past))

    @property
    def dev_in(self) -> int:
        return lib().b200_slice_dev_in(self._h)

    @property
    def dev_out(self) -> int:
        return lib().b200_slice_dev_out(self._h)

    @property
    def pipeline_result(self) -> int:
        """Device pointer of the step's final activation: dev_out, or on rank 0 of a ring pipeline the last slice's output."""
        return lib().b200_pipeline_result(self._h)

    def set_fast_prefill(self, on: bool, min_tokens: int = 0) -> None:
        check(lib().b200_slice_set_fast_prefill(self._h, int(on), min_tokens))

    def mark(self, which: int) -> None:
        check(lib().b200_slice_mark(self._h, which))

    def mark_elapsed_ms(self) -> float:
        return float(lib().b200_slice_mark_elapsed_ms(self._h))

    def profile(self, enable: bool) -> None:
        check(lib().b200_slice_profile(self._h, int(enable)))

    def profile_read(self):
        ms = np.zeros(7, np.float32)
        cnt = np.zeros(7, np.int32)
        check(lib().b200_slice_profile_read(self._h, _ptr(ms), _ptr(cnt), 7))
        return ms, cnt

    def debug_read(self, which: int, count: int, dtype=np.float32) -> np.ndarray:
        out = np.zeros(count, np.uint32)
        check(lib().b200_debug_read(self._h, which, 0, count, _ptr(out)))
        return out.view(dtype)

    def debug_fast_matmul(self, layer: int, which: int, x: np.ndarray, resid: Optional[np.ndarray] = None, tile: int = 0):
        """One fast-mode weight matmul (which: 0 qkv, 1 wo, 2 w1|w3, 3 w2) -> (y, xh).  y is
        [round_up(n_tokens, 256)][rows] float32, rows past n_tokens hold the sentinel 0xFFFFFFFF; xh is the fp16
        activation operand [n_tokens][K]."""
        i = self.info
        K = i.n_ff if which == 3 else i.n_embd
        rows = (3 * i.n_embd, i.n_embd, i.n_ff, i.n_embd)[which] if 0 <= which <= 3 else 0
        x = np.ascontiguousarray(x, dtype=np.float32).reshape(-1, K)
        n = x.shape[0]
        r = None if resid is None else np.ascontiguousarray(resid, dtype=np.float32).reshape(n, i.n_embd)
        y = np.empty(((n + 255) // 256 * 256, rows), np.float32)
        xh = np.empty((n, K), np.float16)
        check(lib().b200_debug_fast_matmul(self._h, layer, which, tile, _ptr(x), n, None if r is None else _ptr(r),
                                           _ptr(y), _ptr(xh)))
        return y, xh

    def skip_attention(self, on: bool) -> None:
        check(lib().b200_debug_skip_attention(self._h, int(on)))

    def trace_enable(self, on: bool) -> None:
        check(lib().b200_debug_trace_enable(self._h, int(on)))

    def trace_read(self, max_launches: int = 512):
        """-> (stamps [n][ctas][8] uint64 ns, class ids [n], cta counts [n])"""
        buf = np.zeros((max_launches, 1024, 8), np.uint64)
        cls = np.zeros(max_launches, np.int32)
        ctas = np.zeros(max_launches, np.int32)
        n = lib().b200_debug_trace_read(self._h, _ptr(buf), _ptr(cls), _ptr(ctas), max_launches)
        return buf[:n], cls[:n], ctas[:n]

    def ptrace_read(self, n_sm: int = 148):
        """-> stamps [n_cta][n_layer][16] uint64 ns of the last persistent step (B200_PTRACE=1)."""
        L = self.info.n_layer
        buf = np.zeros((n_sm, L, 16), np.uint64)
        n = lib().b200_debug_ptrace_read(self._h, _ptr(buf), buf.size)
        return buf[: n // L] if L else buf[:0]

    def last_ms(self) -> float:
        return float(lib().b200_slice_last_ms(self._h))

    def launch_count(self) -> int:
        return int(lib().b200_slice_launch_count(self._h))

    def close(self) -> None:
        if self._h:
            check(lib().b200_slice_unload(self._h))
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
