"""SURVEY.md section 8f row 3 on the GPU: virtual dongles (libb200replay.so, rtl_sensor.h) deliver 262144-byte
buffers exactly as the reference's signal source hands them to its callbacks; the callback body is
b200_stream_push.  Results against the CPU oracle, for several dongles at once and through the reference's
unmodified signal_source.c."""
import ctypes as C
import json
import os
import subprocess
import threading
import time

import numpy as np
import pytest

from oracle import pyoracle as _po

pytestmark = pytest.mark.gpu

BUF = 262144


def collect(ps, s):
    frames = np.concatenate([r for _, r in sorted(ps.spectra[s], key=lambda t: t[0])]) if ps.spectra[s] else np.zeros((0, 1024))
    audio = np.concatenate([a for _, a in sorted(ps.audio[s], key=lambda t: t[0])]) if ps.audio[s] else np.zeros(0)
    return frames, audio


def check_stream(po, iq, frames, audio):
    n = (len(iq) // 204800) * 204800          # whole batches only (the tail stays pending)
    want_rows = po.Spectrum(1024).rows(iq[:n])
    assert frames.shape == want_rows.shape
    ref_db = 10 * np.log10(want_rows)
    ok = want_rows > 1e-6 * want_rows.mean(axis=1, keepdims=True)
    assert np.abs(frames[ok] - ref_db[ok]).max() <= 0.01
    _, dec, _ = po.cic_decimate(10, iq[:n])
    _, _, ref_audio, _ = po.fm_demodulate(dec, po.FmState())
    assert audio.shape == ref_audio.shape and np.abs(audio - ref_audio).max() <= 1e-4


def test_virtual_dongles_feed_the_push_stream(pkg, cuda, po, synth):
    rp = pkg.replay
    n_dongles, n_buffers = 4, 8                                     # 8 x 131072 samples = 5 batches of 204800 + a tail
    caps = [synth.s3_fm(n_buffers * BUF // 2, seed=300 + i) for i in range(n_dongles)]
    ps = pkg.PushStream(n_dongles, 204800)
    lock = threading.Lock()                                         # b200_stream_* is single-producer

    def body(i, buf):
        with lock:
            ps.push(i, buf)

    dongles = [rp.VirtualDongle(40 + i, c) for i, c in enumerate(caps)]
    before = pkg.launch_count()
    threads = [threading.Thread(target=d.read_async, args=(lambda b, i=i: body(i, b),)) for i, d in enumerate(dongles)]
    [t.start() for t in threads]
    [t.join() for t in threads]
    ps.flush()
    # a submission is one chain launch and one history carry.  Dongles that fill a batch together go out as one group
    # (stream.cu), so the 5 batches of each dongle take between 5 and 5 * n_dongles submissions, depending on how the
    # reader threads interleave
    launches = pkg.launch_count() - before
    assert 2 * 5 <= launches <= 2 * 5 * n_dongles, launches
    for i, c in enumerate(caps):
        assert ps.pending(i) == (n_buffers * BUF // 2) % 204800
        frames, audio = collect(ps, i)
        check_stream(po, c, frames, audio)
    [d.close() for d in dongles]
    ps.close()


@pytest.mark.skipif(not os.path.exists(_po.REPLAY_SO), reason="oracle/_ref/libreplay_rtlws.so not built")
def test_reference_signal_source_drives_the_gpu_path(pkg, cuda, po, synth):
    """The reference's signal_source.c (unmodified) reading from the replay sensor, with a registered
    signal_source_callback whose body is b200_stream_push -- INTEGRATION.md section 2, run for real."""
    rp = pkg.replay
    iq = synth.s3_fm(7 * BUF // 2, seed=310)
    L = rp.lib(mode=C.RTLD_GLOBAL)
    ss = C.CDLL(_po.REPLAY_SO)
    ps = pkg.PushStream(1, 204800)
    CB = C.CFUNCTYPE(None, C.POINTER(C.c_ubyte), C.c_int)
    cb = CB(lambda p, n: ps.push(0, np.ctypeslib.as_array(p, shape=(2 * n,))))
    d = rp.VirtualDongle(50, iq)
    L.b200_replay_gate(50, 0)
    ss.signal_source_start.argtypes = [C.c_void_p]
    ss.signal_source_start(d.dev)
    ss.signal_source_add_callback(cb)
    L.b200_replay_gate(50, 1)
    deadline = time.time() + 20
    while d.delivered_bytes() < 7 * BUF and time.time() < deadline:
        time.sleep(0.005)
    ss.signal_source_stop()
    ps.flush()
    frames, audio = collect(ps, 0)
    check_stream(po, iq, frames, audio)
    d.close()
    ps.close()


def test_c_host_example_virtual_dongles(pkg, cuda, tmp_path):
    """examples/virtual_dongles.c: a plain-C host (reader threads as in signal_source.c, rtl_read_async callbacks
    pushing into b200_stream, sinks cutting wire messages) compiled against the two libraries and run."""
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    lib_dir = os.path.join(root, "rtl-ws_b200")
    exe = str(tmp_path / "virtual_dongles")
    subprocess.run(["gcc", "-O2", "-pthread", "-o", exe, os.path.join(root, "examples", "virtual_dongles.c"),
                    "-I" + os.path.join(root, "include"), "-L" + lib_dir, "-lb200sdr", "-lb200replay",
                    "-Wl,-rpath," + lib_dir, "-lm"], check=True)
    n_dongles, seconds = 5, 1.0
    out = subprocess.run([exe, str(n_dongles), str(seconds)], check=True, capture_output=True, text=True, timeout=120)
    r = json.loads(out.stdout.strip().splitlines()[-1])
    n_buffers = int(seconds * 2048000 * 2 / 262144)
    batches = n_buffers * 131072 // 204800
    assert r["dongles"] == n_dongles and r["iq_samples"] == n_dongles * n_buffers * 131072
    assert r["audio_samples"] == n_dongles * batches * 5120
    assert r["spectrum_messages"] == n_dongles * batches and r["spectrum_bytes"] == r["spectrum_messages"] * (31 + 1024)
    assert r["audio_messages"] == n_dongles * (batches * 5120 // 4096) and r["audio_bytes"] == r["audio_messages"] * 16392
    assert 0.1 < r["audio_rms"] < 1.0                      # a 25 kHz-deviation FM signal through the +-1 limiter
    assert r["kernel_launches"] >= 2 * n_dongles * batches
