"""ctypes binding of libb200sdr.so (include/b200sdr.h, include/rtlws_compat.h).

PyTorch is used for device memory and streams only; every computation happens inside the
library's CUDA kernels.  There is no fallback: if the shared library is missing or the
machine has no CUDA device, calls raise.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libb200sdr.so")

WINDOW_RECT = 0
WINDOW_HANN = 1

CHAIN_TILE = 5120          # samples: 5 frames of 1024 = 128 audio samples at R = 10
HALF_BAND_N = 11

# every symbol include/b200sdr.h and include/rtlws_compat.h declare
EXPORTED_SYMBOLS = [
    "b200_init", "b200_last_error", "b200_launch_count", "b200_sm_count",
    "b200_spectrum_plan_create", "b200_spectrum_plan_destroy", "b200_spectrum_plan_rows", "b200_spectrum_exec",
    "b200_spectrum_exec_cs32", "b200_spectrum_exec_rf32",
    "b200_fm_history_samples", "b200_fm_history_reset", "b200_fm_history_carry", "b200_fm_exec",
    "b200_fm_channel_tune", "b200_fm_channels_exec",
    "b200_iq_history_reset", "b200_iq_history_carry", "b200_fm_channel_filter_design",
    "b200_fm_channels_fir_history_samples", "b200_fm_channels_exec_fir", "b200_session_set_channel_filter",
    "b200_fm_channels_exec_runs", "b200_stream_set_channel_sink", "b200_stream_set_channels",
    "b200_stream_set_channel_filter",
    "b200_chain_exec", "b200_chain_exec_r", "b200_chain_tile_samples",
    "b200_session_create", "b200_session_create_r", "b200_session_destroy", "b200_session_reset", "b200_session_chain", "b200_session_products",
    "b200_session_channels",
    "b200_stream_create", "b200_stream_create_r", "b200_stream_destroy", "b200_stream_set_sinks", "b200_stream_set_payload_sink", "b200_stream_push", "b200_stream_poll",
    "b200_stream_flush", "b200_stream_pending_samples",
    "b200_wire_spectrum_header", "b200_wire_spectrum_message", "b200_wire_spectrum_messages",
    "b200_wire_audio_messages", "b200_wire_audio_fragment", "b200_wire_reference_drain_index",
    "b200_host_alloc", "b200_host_free",
    "b200_fm_exec_cs32", "b200_fm_demod_create", "b200_fm_demod_destroy", "b200_fm_demod_reset", "b200_fm_demod_block",
    "b200_debug_atan2", "b200_audio_post", "b200_audio_post_out_samples", "b200_audio_resample_taps",
    "b200_audio_post_rows", "b200_stream_set_audio_post",
    "b200_shard_count", "b200_shard_stream", "b200_comm_unique_id", "b200_comm_create", "b200_comm_create_all",
    "b200_comm_destroy", "b200_comm_world", "b200_comm_rank", "b200_comm_nccl_version", "b200_comm_gather_rows",
    "b200_comm_gather_rows_all", "b200_multi_create", "b200_multi_destroy", "b200_multi_chain",
    "spectrum_alloc", "spectrum_add_cmplx_u8", "spectrum_add_cmplx_s32", "spectrum_add_real_f32", "spectrum_free",
    "cic_decimate", "halfband_decimate",
    "rf_decimator_alloc", "rf_decimator_add_callback", "rf_decimator_set_parameters",
    "rf_decimator_decimate_cmplx_u8", "rf_decimator_remove_callbacks", "rf_decimator_free",
]


class B200Error(RuntimeError):
    pass


class CmplxS32(C.Structure):
    _fields_ = [("re", C.c_int32), ("im", C.c_int32)]


class CicDelayLine(C.Structure):
    """struct cic_delay_line (resample.h:8-12)."""
    _fields_ = [("integrator_prev_out", CmplxS32), ("comb_prev_in", CmplxS32)]


RF_CALLBACK = C.CFUNCTYPE(None, C.POINTER(CmplxS32), C.c_int)
SPECTRUM_SINK = C.CFUNCTYPE(None, C.c_void_p, C.c_int, C.c_int64, C.c_int, C.POINTER(C.c_float))
AUDIO_SINK = C.CFUNCTYPE(None, C.c_void_p, C.c_int, C.c_int64, C.c_int, C.POINTER(C.c_float))
PAYLOAD_SINK = C.CFUNCTYPE(None, C.c_void_p, C.c_int, C.c_int64, C.c_int, C.POINTER(C.c_ubyte))
CHANNEL_SINK = C.CFUNCTYPE(None, C.c_void_p, C.c_int, C.c_int32, C.c_int64, C.c_int, C.POINTER(C.c_float))

FM_MAX_CHANNELS = 32
FM_MAX_RUNS = 64


AUDIO_POST_MAX_ROWS = 1024


class AudioPostRow(C.Structure):
    """b200_audio_post_row: one row of the table of b200_audio_post_rows."""
    _fields_ = [("audio_row", C.c_int32), ("out_row", C.c_int32), ("state_row", C.c_int32), ("fresh", C.c_int32)]


class FmChannelRun(C.Structure):
    """b200_fm_channel_run: one row of the runs table of b200_fm_channels_exec_runs."""
    _fields_ = [("stream", C.c_int32), ("n_channels", C.c_int32), ("first_sample", C.c_int64),
                ("audio_row", C.c_int64), ("phase_inc", C.c_uint32 * FM_MAX_CHANNELS)]

_lib = None


def lib() -> C.CDLL:
    """Load libb200sdr.so (built by __graft_entry__.build()); raises if it is not there."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise B200Error(f"{LIB_PATH} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                        "(there is no CPU fallback)")
    L = C.CDLL(LIB_PATH)
    vp, i32, i64, u64, f32p = C.c_void_p, C.c_int, C.c_int64, C.c_uint64, C.c_void_p
    L.b200_init.argtypes = [i32]
    L.b200_last_error.restype = C.c_char_p
    L.b200_launch_count.restype = u64
    L.b200_sm_count.restype = i32
    L.b200_spectrum_plan_create.restype = vp
    L.b200_spectrum_plan_create.argtypes = [i32, i32, i32, i64, i32, i32]
    L.b200_spectrum_plan_destroy.argtypes = [vp]
    L.b200_spectrum_plan_rows.restype = i64
    L.b200_spectrum_plan_rows.argtypes = [vp, i64]
    for name in ("b200_spectrum_exec", "b200_spectrum_exec_cs32", "b200_spectrum_exec_rf32"):
        getattr(L, name).argtypes = [vp, vp, i64, i32, i64, f32p, f32p, vp, vp]
    L.b200_fm_history_samples.argtypes = [i32]
    L.b200_fm_history_reset.argtypes = [vp, i64, i32, i32, vp]
    L.b200_fm_history_carry.argtypes = [vp, i64, i32, i64, i32, vp]
    L.b200_fm_exec.argtypes = [vp, i64, i32, i64, i32, f32p, i64, vp, i64, vp]
    L.b200_fm_channel_tune.argtypes = [C.c_double, C.c_double, C.POINTER(C.c_uint32)]
    L.b200_fm_channels_exec.argtypes = [vp, i64, i32, i64, i32, i64, vp, i32, f32p, i64, f32p, i64, vp]
    L.b200_iq_history_reset.argtypes = [vp, i64, i32, i32, vp]
    L.b200_iq_history_carry.argtypes = [vp, i64, i32, i64, i32, vp]
    L.b200_fm_channel_filter_design.argtypes = [i32, i32, C.c_double, C.c_double, C.c_double, vp]
    L.b200_fm_channels_fir_history_samples.argtypes = [i32, i32]
    L.b200_fm_channels_exec_fir.argtypes = [vp, i64, i32, i64, i32, i64, vp, i32, f32p, i64, f32p, i64, vp, i32, vp]
    L.b200_session_set_channel_filter.argtypes = [vp, vp, i32]
    L.b200_fm_channels_exec_runs.argtypes = [vp, i64, i32, i64, i32, vp, i32, f32p, i64, i64, vp, i32, vp]
    L.b200_stream_set_channel_sink.argtypes = [vp, i32, CHANNEL_SINK]
    L.b200_stream_set_channels.argtypes = [vp, i32, i32, vp, vp]
    L.b200_stream_set_channel_filter.argtypes = [vp, vp, i32]
    L.b200_chain_exec.argtypes = [vp, i64, i32, i64, i32, f32p, f32p, i64, vp, i32, vp]
    L.b200_chain_exec_r.argtypes = [vp, i64, i32, i64, i32, i32, f32p, f32p, i64, vp, i32, vp]
    L.b200_chain_tile_samples.restype = i64
    L.b200_chain_tile_samples.argtypes = [i32]
    L.b200_session_create.restype = vp
    L.b200_session_create.argtypes = [i32, i64]
    L.b200_session_create_r.restype = vp
    L.b200_session_create_r.argtypes = [i32, i64, i32]
    L.b200_stream_create_r.restype = vp
    L.b200_stream_create_r.argtypes = [i32, i64, i32, i32]
    L.b200_session_destroy.argtypes = [vp]
    L.b200_session_reset.argtypes = [vp]
    L.b200_session_chain.argtypes = [vp, vp, i64, i32, vp, vp]
    L.b200_session_products.argtypes = [vp, vp, i64, i32, i32, vp, vp]
    L.b200_session_channels.argtypes = [vp, vp, i64, vp, i32, vp]
    L.b200_stream_create.restype = vp
    L.b200_stream_create.argtypes = [i32, i64, i32]
    L.b200_stream_destroy.argtypes = [vp]
    L.b200_stream_set_sinks.restype = None
    L.b200_stream_set_sinks.argtypes = [vp, SPECTRUM_SINK, AUDIO_SINK, vp]
    L.b200_stream_set_payload_sink.argtypes = [vp, i32, PAYLOAD_SINK]
    L.b200_stream_push.argtypes = [vp, i32, vp, i32]
    L.b200_stream_poll.argtypes = [vp]
    L.b200_stream_flush.argtypes = [vp]
    L.b200_stream_pending_samples.restype = i64
    L.b200_stream_pending_samples.argtypes = [vp, i32]
    L.b200_wire_spectrum_header.argtypes = [C.c_char_p, i32, C.c_uint32, C.c_uint32, i32]
    L.b200_wire_spectrum_message.argtypes = [vp, i32, C.c_uint32, C.c_uint32, i32, vp, i32]
    L.b200_wire_spectrum_messages.argtypes = [vp, i64, i32, i32, vp, vp, vp, vp, i64, vp, vp]
    L.b200_wire_audio_messages.argtypes = [vp, i64, i32, i64, i32, i32, i32, vp, i64, vp]
    L.b200_wire_audio_fragment.argtypes = [i32, C.POINTER(C.c_int32), C.POINTER(C.c_int32), C.POINTER(C.c_int32)]
    L.b200_wire_reference_drain_index.restype = i64
    L.b200_wire_reference_drain_index.argtypes = [i64, i32]
    L.b200_host_alloc.restype = vp
    L.b200_host_alloc.argtypes = [u64]
    L.b200_host_free.argtypes = [vp]
    L.b200_fm_exec_cs32.argtypes = [vp, i64, i32, i64, vp, vp, i64, vp, i64, vp, i64, i32, vp]
    L.b200_fm_demod_create.restype = vp
    L.b200_fm_demod_destroy.restype = None
    L.b200_fm_demod_destroy.argtypes = [vp]
    L.b200_fm_demod_reset.argtypes = [vp]
    L.b200_fm_demod_block.argtypes = [vp, vp, i32, vp, vp]
    L.b200_debug_atan2.argtypes = [vp, i32, vp, i32, vp]
    L.b200_audio_post.argtypes = [vp, i64, i32, i64, C.c_double, i32, vp, vp, i64, vp]
    L.b200_audio_post_out_samples.restype = i64
    L.b200_audio_post_out_samples.argtypes = [i64, i32]
    L.b200_audio_resample_taps.argtypes = [vp]
    L.b200_audio_post_rows.argtypes = [vp, i64, i64, i64, C.c_double, i32, vp, i32, vp, i64, vp, i64, i64, vp]
    L.b200_stream_set_audio_post.argtypes = [vp, i32, C.c_double]
    L.b200_shard_count.argtypes = [i32, i32, i32]
    L.b200_shard_stream.argtypes = [i32, i32, i32, i32]
    L.b200_comm_unique_id.argtypes = [vp]
    L.b200_comm_create.restype = vp
    L.b200_comm_create.argtypes = [vp, i32, i32]
    L.b200_comm_create_all.argtypes = [i32, C.POINTER(vp)]
    L.b200_comm_destroy.restype = None
    L.b200_comm_destroy.argtypes = [vp]
    L.b200_comm_world.argtypes = [vp]
    L.b200_comm_rank.argtypes = [vp]
    L.b200_comm_gather_rows.argtypes = [vp, vp, i32, i32, vp, i32, vp]
    L.b200_comm_gather_rows_all.argtypes = [C.POINTER(vp), i32, C.POINTER(vp), i32, i32, vp, i32, C.POINTER(vp)]
    L.b200_multi_create.restype = vp
    L.b200_multi_create.argtypes = [i32, i32, i64, i32, i32]
    L.b200_multi_destroy.restype = None
    L.b200_multi_destroy.argtypes = [vp]
    L.b200_multi_chain.argtypes = [vp, vp, i64, vp, vp, vp]
    # reference-named interface
    L.spectrum_alloc.restype = vp
    L.spectrum_alloc.argtypes = [i32]
    L.spectrum_free.argtypes = [vp]
    for name in ("spectrum_add_cmplx_u8", "spectrum_add_cmplx_s32", "spectrum_add_real_f32"):
        getattr(L, name).argtypes = [vp, vp, vp, i32]
    L.cic_decimate.argtypes = [i32, vp, i32, vp, i32, C.POINTER(CicDelayLine)]
    L.halfband_decimate.restype = None
    L.halfband_decimate.argtypes = [vp, vp, i32, vp]
    L.rf_decimator_alloc.restype = vp
    L.rf_decimator_add_callback.argtypes = [vp, RF_CALLBACK]
    L.rf_decimator_set_parameters.argtypes = [vp, C.c_double, i32]
    L.rf_decimator_decimate_cmplx_u8.argtypes = [vp, vp, i32]
    L.rf_decimator_remove_callbacks.argtypes = [vp]
    L.rf_decimator_free.argtypes = [vp]
    _lib = L
    return L


def last_error() -> str:
    return lib().b200_last_error().decode()


def _check(rc: int, what: str) -> None:
    if rc != 0:
        raise B200Error(f"{what} -> {rc}: {last_error()}")


def _torch():
    import torch
    if not torch.cuda.is_available():
        raise B200Error("no CUDA device: libb200sdr has no CPU fallback")
    return torch


def _stream_ptr(stream=None):
    torch = _torch()
    s = torch.cuda.current_stream() if stream is None else stream
    return C.c_void_p(s.cuda_stream)


def init(device: int = 0) -> None:
    _check(lib().b200_init(device), "b200_init")


def launch_count() -> int:
    return int(lib().b200_launch_count())


# --------------------------------------------------------------------------------------
# batched spectrum
# --------------------------------------------------------------------------------------

class SpectrumPlan:
    """b200_spectrum_plan_*: N-point frames, K accumulated per row (spectrum.c + cbb_main.c:48-59,112-128)."""

    def __init__(self, N: int = 1024, hop: int | None = None, K: int = 1, row_hop: int | None = None,
                 window: int = WINDOW_RECT, gain_db: int = 0):
        self.N, self.K = N, K
        self.hop = N if hop is None else hop
        self.row_hop = K * self.hop if row_hop is None else row_hop
        self.h = lib().b200_spectrum_plan_create(N, self.hop, K, self.row_hop, window, gain_db)
        if not self.h:
            raise B200Error(f"b200_spectrum_plan_create: {last_error()}")

    def close(self):
        if getattr(self, "h", None):
            lib().b200_spectrum_plan_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:      # interpreter shutdown: the module globals may already be gone
            pass

    def rows(self, n_samples: int) -> int:
        return int(lib().b200_spectrum_plan_rows(self.h, n_samples))

    def _run(self, fn, x, n_rows, db, power, db_u8, out, stream) -> dict:
        """Allocate the requested [n_streams, n_rows, N] outputs (unless `out` has them) and call the C exec `fn`
        on x[s] (stream s starts x.stride(0) elements after stream s - 1)."""
        torch = _torch()
        n_streams, n_samples = x.shape[0], x.shape[1]
        if n_rows is None:
            n_rows = self.rows(n_samples)
        res = {} if out is None else out
        if db and "db" not in res:
            res["db"] = torch.empty((n_streams, n_rows, self.N), dtype=torch.float32, device=x.device)
        if power and "power" not in res:
            res["power"] = torch.empty((n_streams, n_rows, self.N), dtype=torch.float32, device=x.device)
        if db_u8 and "db_u8" not in res:
            res["db_u8"] = torch.empty((n_streams, n_rows, self.N), dtype=torch.uint8, device=x.device)
        ptr = lambda k: C.c_void_p(res[k].data_ptr()) if k in res else None
        stride = x.stride(0) * x.element_size() if n_streams > 1 else 0
        _check(fn(self.h, C.c_void_p(x.data_ptr()), stride, n_streams, n_rows, ptr("db"), ptr("power"), ptr("db_u8"),
                  _stream_ptr(stream)), fn.__name__)
        return res

    def exec(self, iq, n_rows: int | None = None, db: bool = True, power: bool = False, db_u8: bool = False,
             out: dict | None = None, stream=None) -> dict:
        """iq: cuda uint8 tensor [n_streams, n_samples, 2] (rows may be strided views).

        Returns a dict with the requested [n_streams, n_rows, N] tensors."""
        torch = _torch()
        assert iq.is_cuda and iq.dtype == torch.uint8 and iq.dim() == 3 and iq.shape[2] == 2
        assert iq.stride(2) == 1 and iq.stride(1) == 2
        return self._run(lib().b200_spectrum_exec, iq, n_rows, db, power, db_u8, out, stream)

    def exec_cs32(self, x, n_rows: int | None = None, db: bool = False, power: bool = True, db_u8: bool = False,
                  out: dict | None = None, stream=None) -> dict:
        """x: cuda int32 tensor [n_streams, n_samples, 2] (spectrum_add_cmplx_s32 semantics; rows may be strided
        views).  Outputs as for exec(); power only by default."""
        torch = _torch()
        assert x.is_cuda and x.dtype == torch.int32 and x.dim() == 3 and x.shape[2] == 2
        assert x.stride(2) == 1 and x.stride(1) == 2
        return self._run(lib().b200_spectrum_exec_cs32, x, n_rows, db, power, db_u8, out, stream)

    def exec_rf32(self, x, n_rows: int | None = None, db: bool = False, power: bool = True, db_u8: bool = False,
                  out: dict | None = None, stream=None) -> dict:
        """x: cuda float32 tensor [n_streams, n_samples] (spectrum_add_real_f32 semantics; rows may be strided
        views).  Outputs as for exec(); power only by default."""
        torch = _torch()
        assert x.is_cuda and x.dtype == torch.float32 and x.dim() == 2 and x.stride(1) == 1
        return self._run(lib().b200_spectrum_exec_rf32, x, n_rows, db, power, db_u8, out, stream)


# --------------------------------------------------------------------------------------
# device ring of independent streams: [history | batch] per stream
# --------------------------------------------------------------------------------------

class StreamRing:
    """Device-resident IQ of `n_streams` independent dongles laid out as the FM branch wants it:
    each row is [history (32*R samples, or `history`) | batch (n_samples)], rows 16-byte aligned.
    A FIR channel filter of T taps wants history=fm_channels_fir_history_samples(R, T)."""

    def __init__(self, n_streams: int, n_samples: int, R: int = 10, device="cuda", history: int | None = None):
        torch = _torch()
        self.n_streams, self.n_samples, self.R = n_streams, n_samples, R
        self.hist = int(lib().b200_fm_history_samples(R)) if history is None else int(history)
        if self.hist < int(lib().b200_fm_history_samples(R)) or self.hist % 8 != 0:
            raise B200Error(f"StreamRing: history {self.hist} must be a multiple of 8 and at least 32 R = {32 * R}")
        row = self.hist + n_samples
        row = (row + 7) // 8 * 8
        self.buf = torch.empty((n_streams, row, 2), dtype=torch.uint8, device=device)
        self.batch = self.buf[:, self.hist:self.hist + n_samples, :]
        self.stride_bytes = self.buf.stride(0)
        self.reset()

    def reset(self, stream=None) -> None:
        """Every stream back to its start (history = 128: the reference's zeroed delay lines)."""
        _check(lib().b200_iq_history_reset(C.c_void_p(self.batch.data_ptr()), self.stride_bytes, self.n_streams,
                                           self.hist, _stream_ptr(stream)), "b200_iq_history_reset")

    def carry(self, stream=None) -> None:
        """History <- tail of the batch (call after a batch has been processed)."""
        _check(lib().b200_iq_history_carry(C.c_void_p(self.batch.data_ptr()), self.stride_bytes, self.n_streams,
                                           self.n_samples, self.hist, _stream_ptr(stream)), "b200_iq_history_carry")

    def load(self, iq) -> None:
        """Copy a [n_streams, n_samples, 2] uint8 array/tensor into the batch area."""
        torch = _torch()
        t = torch.as_tensor(iq)
        self.batch.copy_(t.reshape(self.n_streams, self.n_samples, 2), non_blocking=True)


def fm_exec(ring: StreamRing, audio=None, decimated: bool = False, dec=None, stream=None):
    """b200_fm_exec over a StreamRing -> (audio [n_streams, n/(4R)] f32, decimated [n_streams, n/R, 2] i32 | None).
    `audio` / `dec` may be given, also as row slices of wider tensors; a given `dec` implies decimated=True."""
    torch = _torch()
    n_audio = ring.n_samples // (4 * ring.R)
    if audio is None:
        audio = torch.empty((ring.n_streams, n_audio), dtype=torch.float32, device=ring.buf.device)
    if dec is None and decimated:
        dec = torch.empty((ring.n_streams, ring.n_samples // ring.R, 2), dtype=torch.int32, device=ring.buf.device)
    if dec is not None:
        assert dec.dtype == torch.int32 and dec.shape == (ring.n_streams, ring.n_samples // ring.R, 2)
        assert dec.stride(2) == 1 and dec.stride(1) == 2 and dec.stride(0) % 2 == 0
    _check(lib().b200_fm_exec(C.c_void_p(ring.batch.data_ptr()), ring.stride_bytes, ring.n_streams, ring.n_samples,
                              ring.R, C.c_void_p(audio.data_ptr()), audio.stride(0),
                              C.c_void_p(dec.data_ptr()) if dec is not None else None,
                              dec.stride(0) // 2 if dec is not None else 0, _stream_ptr(stream)), "b200_fm_exec")
    return audio, dec


def fm_channel_tune(offset_hz: float, fs: float) -> int:
    """b200_fm_channel_tune: the phase increment (uint32) that brings baseband +offset_hz to DC; host arithmetic."""
    inc = C.c_uint32()
    _check(lib().b200_fm_channel_tune(float(offset_hz), float(fs), C.byref(inc)), "b200_fm_channel_tune")
    return int(inc.value)


FM_MAX_CHANNEL_TAPS = 1024


def fm_channel_filter(R: int, n_taps: int, cutoff_hz: float, atten_db: float = 60.0, fs: float = 2_048_000.0):
    """b200_fm_channel_filter_design: Kaiser-windowed sinc low-pass taps (float32 numpy [n_taps], summing to R) for
    fm_channels_exec(taps=...) / Session.set_channel_filter; host arithmetic."""
    h = np.empty(n_taps if n_taps > 0 else 1, dtype=np.float32)
    _check(lib().b200_fm_channel_filter_design(R, n_taps, float(cutoff_hz), float(atten_db), float(fs), h.ctypes.data),
           "b200_fm_channel_filter_design")
    return h


def fm_channels_fir_history_samples(R: int, n_taps: int) -> int:
    """History (input samples) a stream needs in front of its batch for a T-tap channel filter."""
    h = int(lib().b200_fm_channels_fir_history_samples(R, n_taps))
    if h < 0:
        raise B200Error(f"b200_fm_channels_fir_history_samples({R}, {n_taps}): {last_error()}")
    return h


def _channel_taps(ring: StreamRing, taps, what: str) -> int:
    """The tap count of an FIR channel filter (0 for the boxcar), after refusing a ring whose history is too short
    for it: the kernel would read before the rows."""
    if taps is None:
        return 0
    torch = _torch()
    assert taps.is_cuda and taps.dtype == torch.float32 and taps.dim() == 1 and taps.is_contiguous()
    T = taps.shape[0]
    need = fm_channels_fir_history_samples(ring.R, T)
    if ring.hist < need:
        raise B200Error(f"{what}: {T} taps at R = {ring.R} need a ring history of {need} samples, the ring has "
                        f"{ring.hist}")
    return T


def fm_channels_exec(ring: StreamRing, phase_inc, first_sample: int, audio=None, baseband: bool = False, stream=None,
                     taps=None):
    """b200_fm_channels_exec over a StreamRing: phase_inc is a cuda int32 tensor [n_streams, n_channels] holding the
    uint32 increments' bits; first_sample is the absolute index of the batch's first sample (a multiple of 4R).
    taps (a cuda float32 tensor [T]) selects b200_fm_channels_exec_fir, whose ring needs the longer history of
    fm_channels_fir_history_samples(R, T).  A given audio must be float32 [S, C, n/(4R)] on the ring's device, its
    rows may be slices of wider rows.
    -> (audio [S, C, n/(4R)] f32, baseband [S, C, n/R, 2] f32 | None)."""
    torch = _torch()
    assert phase_inc.is_cuda and phase_inc.dtype == torch.int32 and phase_inc.dim() == 2
    assert phase_inc.shape[0] == ring.n_streams and phase_inc.is_contiguous()
    S, Ch = phase_inc.shape
    n_audio = ring.n_samples // (4 * ring.R)
    if audio is None:
        audio = torch.empty((S, Ch, n_audio), dtype=torch.float32, device=ring.buf.device)
    _check_output("fm_channels_exec audio", audio, torch.float32, (S, Ch, n_audio), ring.buf.device, row_slices=True)
    bb = None
    if baseband:
        bb = torch.empty((S, Ch, ring.n_samples // ring.R, 2), dtype=torch.float32, device=ring.buf.device)
    T = _channel_taps(ring, taps, "fm_channels_exec")
    args = (C.c_void_p(ring.batch.data_ptr()), ring.stride_bytes, ring.n_streams, ring.n_samples, ring.R, first_sample,
            C.c_void_p(phase_inc.data_ptr()), Ch, C.c_void_p(audio.data_ptr()), audio.stride(1),
            C.c_void_p(bb.data_ptr()) if bb is not None else None, bb.stride(1) // 2 if bb is not None else 0)
    if T:
        _check(lib().b200_fm_channels_exec_fir(*args, C.c_void_p(taps.data_ptr()), T, _stream_ptr(stream)),
               "b200_fm_channels_exec_fir")
    else:
        _check(lib().b200_fm_channels_exec(*args, _stream_ptr(stream)), "b200_fm_channels_exec")
    return audio, bb


def fm_channels_exec_runs(ring: StreamRing, runs, audio=None, taps=None, stream=None):
    """b200_fm_channels_exec_runs over a StreamRing: runs is a sequence of (stream, first_sample, phase_inc list),
    each with its own position and 1..32 uint32 increments; run k's channels get the next len(phase_inc) audio rows,
    in order.  taps (a cuda float32 tensor [T]) selects the FIR filter, whose ring needs the history of
    fm_channels_fir_history_samples(R, T).  -> audio [sum of the channel counts, n/(4R)] f32."""
    torch = _torch()
    runs = list(runs)
    table = (FmChannelRun * max(1, len(runs)))()
    row = 0
    for k, (s, first, incs) in enumerate(runs):
        incs = [int(v) & 0xFFFFFFFF for v in incs]
        table[k].stream, table[k].n_channels, table[k].first_sample, table[k].audio_row = s, len(incs), first, row
        for c, v in enumerate(incs[:FM_MAX_CHANNELS]):
            table[k].phase_inc[c] = v
        row += len(incs)
    n_audio = ring.n_samples // (4 * ring.R)
    if audio is None:
        audio = torch.empty((max(row, 1), n_audio), dtype=torch.float32, device=ring.buf.device)
    _check_output("fm_channels_exec_runs audio", audio, torch.float32, (max(row, 1), n_audio), ring.buf.device,
                  row_slices=True)
    T = _channel_taps(ring, taps, "fm_channels_exec_runs")
    _check(lib().b200_fm_channels_exec_runs(C.c_void_p(ring.batch.data_ptr()), ring.stride_bytes, ring.n_streams,
                                            ring.n_samples, ring.R, table, len(runs), C.c_void_p(audio.data_ptr()),
                                            audio.stride(0), audio.shape[0],
                                            C.c_void_p(taps.data_ptr()) if taps is not None else None, T,
                                            _stream_ptr(stream)), "b200_fm_channels_exec_runs")
    return audio


def _check_output(what: str, t, dtype, shape: tuple, device, row_slices: bool = False) -> None:
    """Refuse an output tensor the kernels would write past: they see only its data pointer (and row stride).
    row_slices: rows (the last dimension) may be slices of wider rows, with unit column stride, and the leading
    dimensions pack them one row stride apart; otherwise the tensor must be contiguous."""
    packed = all(t.stride(d) == t.shape[d + 1] * t.stride(d + 1) for d in range(t.dim() - 2))
    layout_ok = t.stride(-1) == 1 and packed if row_slices else t.is_contiguous()
    if t.dtype != dtype or tuple(t.shape) != shape or not layout_ok or t.device != device:
        raise B200Error(f"{what}: want {dtype} {shape} {'with unit column stride' if row_slices else 'contiguous'} "
                        f"on {device}, got {t.dtype} {tuple(t.shape)} strides {t.stride()} on {t.device}")


def chain_exec(ring: StreamRing, gain_db: int = 0, db=None, audio=None, avg_u8=None, K_avg: int = 6, stream=None):
    """b200_chain_exec: per-frame dB spectra (N = 1024) + FM audio from one pass over the ring's batch.
    Given outputs must be on the ring's device: db contiguous float32 [n_streams, n/1024, 1024], audio float32
    [n_streams, n/(4R)] (rows may be slices of wider rows), avg_u8 contiguous uint8 [n_streams, 1024]."""
    torch = _torch()
    S, dev = ring.n_streams, ring.buf.device
    n_audio = ring.n_samples // (4 * ring.R)
    if db is None:
        db = torch.empty((S, ring.n_samples // 1024, 1024), dtype=torch.float32, device=dev)
    if audio is None:
        audio = torch.empty((S, n_audio), dtype=torch.float32, device=dev)
    _check_output("chain_exec db", db, torch.float32, (S, ring.n_samples // 1024, 1024), dev)
    _check_output("chain_exec audio", audio, torch.float32, (S, n_audio), dev, row_slices=True)
    if avg_u8 is not None:
        _check_output("chain_exec avg_u8", avg_u8, torch.uint8, (S, 1024), dev)
    _check(lib().b200_chain_exec_r(C.c_void_p(ring.batch.data_ptr()), ring.stride_bytes, ring.n_streams,
                                   ring.n_samples, ring.R, gain_db, C.c_void_p(db.data_ptr()), C.c_void_p(audio.data_ptr()),
                                   audio.stride(0), C.c_void_p(avg_u8.data_ptr()) if avg_u8 is not None else None,
                                   K_avg, _stream_ptr(stream)), "b200_chain_exec_r")
    return db, audio


FM_STATE_FLOATS = 48
FM_SKIP_STAGE2 = 1
AUDIO_DEEMPH_50US, AUDIO_DEEMPH_75US, AUDIO_RESAMPLE_48K = 1, 2, 4
AUDIO_POST_STATE_FLOATS = 64
COMM_ID_BYTES = 128


def fm_exec_cs32(dec, state, audio=None, demod: bool = False, phase: bool = False, flags: int = 0, stream=None):
    """b200_fm_exec_cs32: decimated cmplx_s32 [n_streams, n, 2] (cuda int32) + carried state
    [n_streams, FM_STATE_FLOATS] -> dict(audio, demod?, phase?).  audio_main.c:110-139."""
    torch = _torch()
    assert dec.is_cuda and dec.dtype == torch.int32 and dec.dim() == 3 and dec.shape[2] == 2 and dec.stride(1) == 2
    assert state.is_cuda and state.dtype == torch.float32 and state.shape == (dec.shape[0], FM_STATE_FLOATS)
    n_streams, n = dec.shape[0], dec.shape[1]
    res = {}
    skip = bool(flags & FM_SKIP_STAGE2)
    if not skip:
        res["audio"] = audio if audio is not None else torch.empty((n_streams, n // 4), dtype=torch.float32, device=dec.device)
    if demod:
        res["demod"] = torch.empty((n_streams, n), dtype=torch.float32, device=dec.device)
    if phase:
        res["phase"] = torch.empty((n_streams, n), dtype=torch.float32, device=dec.device)
    ptr = lambda k: C.c_void_p(res[k].data_ptr()) if k in res else None
    stride = lambda k: res[k].stride(0) if k in res else 0
    _check(lib().b200_fm_exec_cs32(C.c_void_p(dec.data_ptr()), dec.stride(0) // 2, n_streams, n,
                                   C.c_void_p(state.data_ptr()), ptr("audio"), stride("audio"), ptr("demod"),
                                   stride("demod"), ptr("phase"), stride("phase"), flags, _stream_ptr(stream)),
           "b200_fm_exec_cs32")
    return res


def debug_atan2(y, x, which: int):
    """atan2_approx of integer pairs as kernel family `which` evaluates it (b200_debug_atan2)."""
    torch = _torch()
    yx = torch.stack([torch.as_tensor(y, dtype=torch.int32), torch.as_tensor(x, dtype=torch.int32)], dim=-1).contiguous().cuda()
    out = torch.empty(yx.shape[:-1], dtype=torch.float32, device="cuda")
    _check(lib().b200_debug_atan2(C.c_void_p(yx.data_ptr()), out.numel(), C.c_void_p(out.data_ptr()), which,
                                  _stream_ptr()), "b200_debug_atan2")
    return out.cpu().numpy()


class FmDemod:
    """b200_fm_demod_*: the body of an rf_decimator_callback -- host cmplx_s32 blocks in, host audio out."""

    def __init__(self):
        _torch()
        self.h = lib().b200_fm_demod_create()
        if not self.h:
            raise B200Error(f"b200_fm_demod_create: {last_error()}")

    def block(self, signal: np.ndarray, want_audio: bool = True, want_demod: bool = False):
        signal = np.ascontiguousarray(signal, dtype=np.int32).reshape(-1, 2)
        n = len(signal)
        audio = np.empty(n // 4, dtype=np.float32) if want_audio else None
        demod = np.empty(n, dtype=np.float32) if want_demod else None
        _check(lib().b200_fm_demod_block(self.h, signal.ctypes.data, n, audio.ctypes.data if want_audio else None,
                                         demod.ctypes.data if want_demod else None), "b200_fm_demod_block")
        return audio, demod

    def reset(self):
        _check(lib().b200_fm_demod_reset(self.h), "b200_fm_demod_reset")

    def close(self):
        if getattr(self, "h", None):
            lib().b200_fm_demod_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def audio_post(audio, state, flags: int, rate_hz: float = 51200.0, out=None, stream=None):
    """b200_audio_post: opt-in de-emphasis / 15:16 resampling of [n_streams, n] f32 audio rows (extensions,
    not in the reference).  state: cuda float32 [n_streams, AUDIO_POST_STATE_FLOATS], zero = stream start."""
    torch = _torch()
    assert audio.is_cuda and audio.dtype == torch.float32 and audio.dim() == 2 and audio.stride(1) == 1
    n_streams, n = audio.shape
    n_out = int(lib().b200_audio_post_out_samples(n, flags))
    if n_out < 0:
        raise B200Error("audio_post: the resampler takes multiples of 16 samples")
    if out is None:
        out = torch.empty((n_streams, n_out), dtype=torch.float32, device=audio.device)
    _check(lib().b200_audio_post(C.c_void_p(audio.data_ptr()), audio.stride(0), n_streams, n, rate_hz, flags,
                                 C.c_void_p(state.data_ptr()), C.c_void_p(out.data_ptr()), out.stride(0),
                                 _stream_ptr(stream)), "b200_audio_post")
    return out


def audio_post_rows(audio, rows, state, flags: int, rate_hz: float = 51200.0, out=None, stream=None):
    """b200_audio_post_rows: audio_post over a table of rows.  rows is a sequence of (audio_row, out_row, state_row,
    fresh); row k reads audio[audio_row], writes out[out_row] and advances state[state_row] (or starts from zero state
    if fresh).  audio: cuda float32 [n_audio_rows, n] (rows may be slices of wider rows), state: cuda float32
    [n_state_rows, AUDIO_POST_STATE_FLOATS], out (allocated if not given, one row per table row): float32
    [n_out_rows, audio_post_out_samples(n)] rows with unit column stride."""
    torch = _torch()
    assert audio.is_cuda and audio.dtype == torch.float32 and audio.dim() == 2 and audio.stride(1) == 1
    n = audio.shape[1]
    n_out = int(lib().b200_audio_post_out_samples(n, flags))
    if n_out < 0:
        raise B200Error("audio_post_rows: the resampler takes multiples of 16 samples")
    rows = list(rows)
    table = (AudioPostRow * max(1, len(rows)))()
    for k, (a, o, st, fresh) in enumerate(rows):
        table[k].audio_row, table[k].out_row, table[k].state_row, table[k].fresh = a, o, st, int(bool(fresh))
    if out is None:
        out = torch.empty((max(1, len(rows)), n_out), dtype=torch.float32, device=audio.device)
    _check_output("audio_post_rows out", out, torch.float32, (out.shape[0], n_out), audio.device, row_slices=True)
    _check_output("audio_post_rows state", state, torch.float32, (state.shape[0], AUDIO_POST_STATE_FLOATS),
                  audio.device)
    _check(lib().b200_audio_post_rows(C.c_void_p(audio.data_ptr()), audio.stride(0), audio.shape[0], n, rate_hz, flags,
                                      table, len(rows), C.c_void_p(state.data_ptr()), state.shape[0],
                                      C.c_void_p(out.data_ptr()), out.stride(0), out.shape[0], _stream_ptr(stream)),
           "b200_audio_post_rows")
    return out


def resample_taps() -> np.ndarray:
    h = np.empty(240, dtype=np.float32)
    assert lib().b200_audio_resample_taps(h.ctypes.data) == 240
    return h


class Comm:
    """b200_comm_*: the NCCL communicator behind the one exchange of the path (gather of per-stream rows).
    One process per GPU: `Comm.unique_id()` on rank 0, distribute the 128 bytes, `Comm(id, world, rank)`."""

    def __init__(self, id128: bytes, world: int, rank: int):
        _torch()
        assert len(id128) == COMM_ID_BYTES
        self.world, self.rank = world, rank
        buf = (C.c_ubyte * COMM_ID_BYTES).from_buffer_copy(id128)
        self.h = lib().b200_comm_create(buf, world, rank)
        if not self.h:
            raise B200Error(f"b200_comm_create: {last_error()}")

    @staticmethod
    def unique_id() -> bytes:
        buf = (C.c_ubyte * COMM_ID_BYTES)()
        _check(lib().b200_comm_unique_id(buf), "b200_comm_unique_id")
        return bytes(buf)

    def gather_rows(self, send, n_streams_total: int, recv=None, root: int = 0, stream=None):
        """send: cuda tensor [n_local, row...] (contiguous); recv (root): [n_streams_total, row...]."""
        row_bytes = int(send[0].numel() * send.element_size()) if send.shape[0] else int(recv[0].numel() * recv.element_size())
        _check(lib().b200_comm_gather_rows(self.h, C.c_void_p(send.data_ptr()), n_streams_total, row_bytes,
                                           C.c_void_p(recv.data_ptr()) if recv is not None else None, root,
                                           _stream_ptr(stream)), "b200_comm_gather_rows")

    def close(self):
        if getattr(self, "h", None):
            lib().b200_comm_destroy(self.h)
            self.h = None


class Multi:
    """b200_multi_*: one process, G GPUs, host arrays in global stream order (stream s on device s mod G)."""

    def __init__(self, n_gpus: int, n_streams: int, max_samples: int, gain_db: int = 0, K_avg: int = 6):
        _torch()
        self.n_gpus, self.n_streams = n_gpus, n_streams
        self.h = lib().b200_multi_create(n_gpus, n_streams, max_samples, gain_db, K_avg)
        if not self.h:
            raise B200Error(f"b200_multi_create: {last_error()}")

    def chain(self, h_iq: np.ndarray, n_samples: int, want_db: bool = True, want_audio: bool = True, want_avg: bool = True):
        h_iq = np.ascontiguousarray(h_iq, dtype=np.uint8)
        db = np.empty((self.n_streams, n_samples // 1024, 1024), np.float32) if want_db else None
        audio = np.empty((self.n_streams, n_samples // 40), np.float32) if want_audio else None
        avg = np.empty((self.n_streams, 1024), np.uint8) if want_avg else None
        p = lambda a: a.ctypes.data if a is not None else None
        _check(lib().b200_multi_chain(self.h, h_iq.ctypes.data, n_samples, p(db), p(audio), p(avg)), "b200_multi_chain")
        return db, audio, avg

    def close(self):
        if getattr(self, "h", None):
            lib().b200_multi_destroy(self.h)
            self.h = None


def shard_count(n_streams: int, world: int, rank: int) -> int:
    return int(lib().b200_shard_count(n_streams, world, rank))


def shard_stream(n_streams: int, world: int, rank: int, i: int) -> int:
    return int(lib().b200_shard_stream(n_streams, world, rank, i))


class Session:
    """b200_session_*: the host-buffer entry point (PCIe copies inside)."""

    def __init__(self, n_streams: int, max_samples: int, R: int = 10):
        _torch()
        self.n_streams, self.max_samples, self.R = n_streams, max_samples, R
        self.h = lib().b200_session_create_r(n_streams, max_samples, R)
        if not self.h:
            raise B200Error(f"b200_session_create_r: {last_error()}")

    def close(self):
        if getattr(self, "h", None):
            lib().b200_session_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:      # interpreter shutdown: the module globals may already be gone
            pass

    def reset(self):
        lib().b200_session_reset(self.h)

    def chain(self, h_iq, n_samples: int, h_db=None, h_audio=None, gain_db: int = 0) -> None:
        """h_iq / h_db / h_audio: host tensors or numpy arrays (pinned for asynchronous copies)."""
        def hp(x):
            if x is None:
                return None
            return C.c_void_p(x.data_ptr() if hasattr(x, "data_ptr") else x.ctypes.data)
        _check(lib().b200_session_chain(self.h, hp(h_iq), n_samples, gain_db, hp(h_db), hp(h_audio)),
               "b200_session_chain")


    def products(self, h_iq, n_samples: int, h_audio, h_avg_u8, gain_db: int = 0, K_avg: int = 6) -> None:
        """b200_session_products: audio + the K-frame averaged payload bytes per stream (the reference's own products)."""
        def hp(x):
            if x is None:
                return None
            return C.c_void_p(x.data_ptr() if hasattr(x, "data_ptr") else x.ctypes.data)
        _check(lib().b200_session_products(self.h, hp(h_iq), n_samples, gain_db, K_avg, hp(h_audio), hp(h_avg_u8)),
               "b200_session_products")

    def set_channel_filter(self, h_taps) -> None:
        """b200_session_set_channel_filter: later channels() calls use these FIR taps (host float32); None or an
        empty array goes back to the boxcar.  Only at stream position 0 (after creation or reset())."""
        h = np.zeros(0, np.float32) if h_taps is None else np.ascontiguousarray(h_taps, dtype=np.float32).reshape(-1)
        _check(lib().b200_session_set_channel_filter(self.h, h.ctypes.data if h.size else None, int(h.size)),
               "b200_session_set_channel_filter")

    def channels(self, h_iq, n_samples: int, phase_inc, h_audio=None):
        """b200_session_channels: phase_inc [n_streams, n_channels] (host, uint32 bits) -> h_audio
        [n_streams, n_channels, n_samples / (4R)] f32 (allocated if not given), mixed at the session's position."""
        inc = np.ascontiguousarray(np.asarray(phase_inc).astype(np.int64) & 0xFFFFFFFF, dtype=np.uint32)
        assert inc.ndim == 2 and inc.shape[0] == self.n_streams
        if h_audio is None:
            h_audio = np.empty((self.n_streams, inc.shape[1], n_samples // (4 * self.R)), np.float32)
        h_iq = np.ascontiguousarray(h_iq, dtype=np.uint8) if isinstance(h_iq, np.ndarray) else h_iq
        p = lambda x: C.c_void_p(x.data_ptr() if hasattr(x, "data_ptr") else x.ctypes.data)
        _check(lib().b200_session_channels(self.h, p(h_iq), n_samples, inc.ctypes.data, inc.shape[1], p(h_audio)),
               "b200_session_channels")
        return h_audio


class PushStream:
    """b200_stream_*: signal_source-style pushes in, spectra and audio out through sinks."""

    def __init__(self, n_streams: int, batch_samples: int, gain_db: int = 0, R: int = 10, payload_K: int = 0,
                 frames: bool = True, channel_capacity: int = 0):
        """payload_K > 0: also collect the K-frame averaged u8 payload of every batch (self.payloads);
        frames=False: no per-frame dB sink (the rows stay on the device);
        channel_capacity > 0: FM channels, up to that many per dongle (set_channels), collected in
        self.channel_audio[stream][channel id] as (first_sample, [n] copy) tuples."""
        _torch()
        self.n_streams, self.batch, self.R = n_streams, batch_samples, R
        self.h = lib().b200_stream_create_r(n_streams, batch_samples, gain_db, R)
        if not self.h:
            raise B200Error(f"b200_stream_create_r: {last_error()}")
        self.payloads = [[] for _ in range(n_streams)]     # (first_frame, K, [1024] u8 copy)
        self._frames = frames
        self._payload_K = payload_K
        self.spectra = [[] for _ in range(n_streams)]      # (first_frame, [n_frames, 1024] copy)
        self.audio = [[] for _ in range(n_streams)]        # (first_sample, [n] copy)
        self.channel_audio = [{} for _ in range(n_streams)]   # id -> [(first_sample, [n] copy)]

        def on_spectrum(user, stream, first, n, ptr):
            self.spectra[stream].append((first, np.ctypeslib.as_array(ptr, shape=(n, 1024)).copy()))

        def on_audio(user, stream, first, n, ptr):
            self.audio[stream].append((first, np.ctypeslib.as_array(ptr, shape=(n,)).copy()))

        def on_payload(user, stream, first, k, ptr):
            self.payloads[stream].append((first, k, np.ctypeslib.as_array(ptr, shape=(1024,)).copy()))

        self._on_spectrum = SPECTRUM_SINK(on_spectrum)
        self._cb = (self._on_spectrum if self._frames else SPECTRUM_SINK(), AUDIO_SINK(on_audio), PAYLOAD_SINK(on_payload))
        lib().b200_stream_set_sinks(self.h, self._cb[0], self._cb[1], None)
        if self._payload_K > 0:
            _check(lib().b200_stream_set_payload_sink(self.h, self._payload_K, self._cb[2]), "b200_stream_set_payload_sink")

        def on_channel(user, stream, cid, first, n, ptr):
            self.channel_audio[stream].setdefault(cid, []).append((first, np.ctypeslib.as_array(ptr, shape=(n,)).copy()))

        self._on_channel = CHANNEL_SINK(on_channel)
        if channel_capacity > 0:
            _check(lib().b200_stream_set_channel_sink(self.h, channel_capacity, self._on_channel),
                   "b200_stream_set_channel_sink")

    def set_channels(self, stream: int, phase_inc, ids) -> None:
        """b200_stream_set_channels: dongle `stream`'s listeners from now on (increments as uint32 bits, distinct
        int32 ids); empty lists clear the set.  Takes effect with the batch whose last sample is pushed next."""
        inc = np.ascontiguousarray(np.asarray(phase_inc, dtype=np.int64).reshape(-1) & 0xFFFFFFFF, dtype=np.uint32)
        cid = np.ascontiguousarray(np.asarray(ids, dtype=np.int64).reshape(-1), dtype=np.int32)
        assert inc.size == cid.size
        _check(lib().b200_stream_set_channels(self.h, stream, int(inc.size), inc.ctypes.data if inc.size else None,
                                              cid.ctypes.data if cid.size else None), "b200_stream_set_channels")

    def set_channel_filter(self, h_taps) -> None:
        """b200_stream_set_channel_filter: FIR taps (host float32) for every channel; None or empty goes back to the
        boxcar.  Only before anything is pushed."""
        h = np.zeros(0, np.float32) if h_taps is None else np.ascontiguousarray(h_taps, dtype=np.float32).reshape(-1)
        _check(lib().b200_stream_set_channel_filter(self.h, h.ctypes.data if h.size else None, int(h.size)),
               "b200_stream_set_channel_filter")

    def set_audio_post(self, flags: int, rate_hz: float = 51200.0) -> None:
        """b200_stream_set_audio_post: de-emphasis and / or 48 kHz output (AUDIO_* flags; 0 = raw audio) for the
        centre and channel audio sinks.  rate_hz is fs / (4R).  Only before anything is pushed."""
        _check(lib().b200_stream_set_audio_post(self.h, flags, rate_hz), "b200_stream_set_audio_post")

    def enable_frames(self) -> None:
        """Install the per-frame dB sink on a stream that was created without one (frames=False): the library
        allocates the row buffers now; batches submitted before this call deliver no rows."""
        self._frames = True
        self._cb = (self._on_spectrum, self._cb[1], self._cb[2])
        lib().b200_stream_set_sinks(self.h, self._cb[0], self._cb[1], None)

    def push(self, stream: int, samples: np.ndarray) -> None:
        samples = np.ascontiguousarray(samples, dtype=np.uint8)
        _check(lib().b200_stream_push(self.h, stream, samples.ctypes.data, samples.size // 2), "b200_stream_push")

    def poll(self) -> None:
        _check(lib().b200_stream_poll(self.h), "b200_stream_poll")

    def flush(self) -> None:
        _check(lib().b200_stream_flush(self.h), "b200_stream_flush")

    def pending(self, stream: int) -> int:
        return int(lib().b200_stream_pending_samples(self.h, stream))

    def close(self):
        if getattr(self, "h", None):
            lib().b200_stream_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:      # interpreter shutdown: the module globals may already be gone
            pass


# --------------------------------------------------------------------------------------
# the reference's interface, same names (numpy in / numpy out, synchronous)
# --------------------------------------------------------------------------------------

def spectrum_alloc(N: int):
    h = lib().spectrum_alloc(N)
    if not h:
        raise B200Error(f"spectrum_alloc({N}) failed")
    return h


def spectrum_free(s) -> None:
    lib().spectrum_free(s)


def spectrum_add_cmplx_u8(s, src: np.ndarray, power_spectrum: np.ndarray, length: int) -> int:
    src = np.ascontiguousarray(src, dtype=np.uint8)
    assert power_spectrum.dtype == np.float64 and power_spectrum.flags.c_contiguous
    return lib().spectrum_add_cmplx_u8(s, src.ctypes.data, power_spectrum.ctypes.data, length)


def spectrum_add_cmplx_s32(s, src: np.ndarray, power_spectrum: np.ndarray, length: int) -> int:
    src = np.ascontiguousarray(src, dtype=np.int32)
    assert power_spectrum.dtype == np.float64 and power_spectrum.flags.c_contiguous
    return lib().spectrum_add_cmplx_s32(s, src.ctypes.data, power_spectrum.ctypes.data, length)


def spectrum_add_real_f32(s, src: np.ndarray, power_spectrum: np.ndarray, length: int) -> int:
    src = np.ascontiguousarray(src, dtype=np.float32)
    assert power_spectrum.dtype == np.float64 and power_spectrum.flags.c_contiguous
    return lib().spectrum_add_real_f32(s, src.ctypes.data, power_spectrum.ctypes.data, length)


def cic_decimate(R: int, src: np.ndarray, src_len: int, dst: np.ndarray, dst_len: int, delay: CicDelayLine) -> int:
    src = np.ascontiguousarray(src, dtype=np.uint8)
    assert dst.dtype == np.int32 and dst.flags.c_contiguous
    return lib().cic_decimate(R, src.ctypes.data, src_len, dst.ctypes.data, dst_len, C.byref(delay))


def halfband_decimate(inp: np.ndarray, out: np.ndarray, output_len: int, delay: np.ndarray) -> None:
    inp = np.ascontiguousarray(inp, dtype=np.float32)
    assert out.dtype == np.float32 and delay.dtype == np.float32 and len(delay) == HALF_BAND_N - 1
    lib().halfband_decimate(inp.ctypes.data, out.ctypes.data, output_len, delay.ctypes.data)


class RfDecimator:
    """rf_decimator_* (rf_decimator.h:11-21): re-blocking to 100 ms, CIC on the GPU, host callbacks."""

    def __init__(self):
        self.h = lib().rf_decimator_alloc()
        self._keep = []

    def add_callback(self, fn) -> None:
        def tramp(ptr, n):
            arr = np.ctypeslib.as_array(C.cast(ptr, C.POINTER(C.c_int32)), shape=(n, 2))
            fn(arr, n)
        cb = RF_CALLBACK(tramp)
        self._keep.append(cb)
        lib().rf_decimator_add_callback(self.h, cb)

    def set_parameters(self, sample_rate: float, down_factor: int) -> int:
        return lib().rf_decimator_set_parameters(self.h, sample_rate, down_factor)

    def decimate_cmplx_u8(self, signal: np.ndarray, length: int | None = None) -> int:
        signal = np.ascontiguousarray(signal, dtype=np.uint8)
        n = signal.size // 2 if length is None else length
        return lib().rf_decimator_decimate_cmplx_u8(self.h, signal.ctypes.data, n)

    def remove_callbacks(self) -> None:
        lib().rf_decimator_remove_callbacks(self.h)
        self._keep.clear()

    def free(self) -> None:
        if self.h:
            lib().rf_decimator_free(self.h)
            self.h = None
