"""rtl-ws_b200 -- B200-native (sm_100a) IQ processing path for rtl-ws.

The product is the C-ABI shared library ``libb200sdr.so`` built from ``csrc/`` (CUDA
kernels + host C++); this package is its thin ctypes binding plus the synthetic IQ
generators used by the tests and the benchmark.  The directory name carries a hyphen, so
import it through ``__graft_entry__.load_package()`` (tests/conftest.py does) under the
module name ``rtl_ws_b200``.
"""
from . import audio, binding, replay, sharding, synth, wire  # noqa: F401
from .binding import (  # noqa: F401
    B200Error, SpectrumPlan, StreamRing, Session, PushStream, RfDecimator, CicDelayLine,
    fm_exec, chain_exec, fm_channel_tune, fm_channels_exec, FM_MAX_CHANNELS, fm_channel_filter,
    fm_channels_exec_runs, FmChannelRun, FM_MAX_RUNS,
    fm_channels_fir_history_samples, FM_MAX_CHANNEL_TAPS, init, lib, launch_count, fm_exec_cs32, FmDemod, debug_atan2, audio_post, resample_taps,
    audio_post_rows, AudioPostRow, AUDIO_POST_MAX_ROWS, Comm, Multi,
    shard_count, shard_stream, FM_STATE_FLOATS, FM_SKIP_STAGE2, AUDIO_DEEMPH_50US, AUDIO_DEEMPH_75US,
    AUDIO_RESAMPLE_48K, AUDIO_POST_STATE_FLOATS,
    spectrum_alloc, spectrum_free, spectrum_add_cmplx_u8, spectrum_add_cmplx_s32, spectrum_add_real_f32,
    cic_decimate, halfband_decimate,
    WINDOW_RECT, WINDOW_HANN, CHAIN_TILE, LIB_PATH, EXPORTED_SYMBOLS,
)
