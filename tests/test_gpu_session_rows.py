"""The device IQ rows of a host-buffer session ([history | batch] per stream) and the public history calls.

A session's channel filter sets the history every session call carries, so a batch shorter than it is refused by all
of them; sessions of more than 16 streams submit groups of several streams per lane; the history calls check their
arguments before they launch anything, and say why in b200_last_error().
"""
import ctypes as C

import numpy as np
import pytest

from test_gpu_fm_channels import FS, incs_tensor

B200_ERR_ARG, B200_ERR_ALIGN = -1, -4


def dev(torch, h):
    return torch.as_tensor(np.ascontiguousarray(h, np.float32)).cuda()


@pytest.mark.gpu
def test_filter_history_binds_every_session_call(pkg, synth, cuda):
    """R = 1, batches of up to 2048 samples (tile 1024) and 1024 taps: the history is 1056 samples, so a batch of
    1024 is refused by chain, products and channels before anything is launched, and the position stays at 0."""
    torch = cuda
    R, T, n = 1, 1024, 2048
    H = pkg.fm_channels_fir_history_samples(R, T)
    assert H == 1056
    h = pkg.fm_channel_filter(R, T, 0.4 * FS, 60.0)
    iq = synth.s3_fm(n, seed=7, carrier=100e3)[None]
    incs = np.array([[pkg.fm_channel_tune(f, FS) for f in (100e3, -300e3)]], dtype=np.int64)
    sess = pkg.Session(1, n, R=R)
    sess.set_channel_filter(h)
    short = np.ascontiguousarray(iq[:, :1024])
    torch.cuda.synchronize()
    before = pkg.launch_count()
    with pytest.raises(pkg.B200Error):
        sess.chain(short, 1024, np.empty((1, 1, 1024), np.float32), np.empty((1, 1024 // (4 * R)), np.float32))
    with pytest.raises(pkg.B200Error):
        sess.products(short, 1024, np.empty((1, 1024 // (4 * R)), np.float32), np.empty((1, 1024), np.uint8), K_avg=1)
    with pytest.raises(pkg.B200Error):
        sess.channels(short, 1024, incs)
    assert pkg.launch_count() == before

    got = sess.channels(iq, n, incs)
    ring = pkg.StreamRing(1, n, R=R, history=H)
    ring.load(iq)
    want, _ = pkg.fm_channels_exec(ring, incs_tensor(torch, incs), 0, taps=dev(torch, h))
    assert np.array_equal(got, want.cpu().numpy())
    sess.close()


@pytest.mark.gpu
def test_session_groups_of_several_streams(pkg, synth, cuda):
    """40 streams: groups of ceil(40 / 16) = 3 streams, the last one of 1.  With a 200-tap filter, channel batches
    equal the device form batch by batch; chain batches between them equal a filterless session's."""
    torch = cuda
    R, T, S = 10, 200, 40
    n = 2 * int(pkg.lib().b200_chain_tile_samples(R))
    n_audio = n // (4 * R)
    h = pkg.fm_channel_filter(R, T, 80e3, 60.0)
    parts = [np.stack([synth.s3_fm(n, seed=1000 * k + s, carrier=-250e3 + 10e3 * s) for s in range(S)])
             for k in range(6)]
    incs = np.array([[pkg.fm_channel_tune(f, FS) for f in (-250e3 + 10e3 * s, 300e3)] for s in range(S)],
                    dtype=np.int64)
    sess = pkg.Session(S, n, R=R)
    sess.set_channel_filter(h)
    plain = pkg.Session(S, n, R=R)
    ring = pkg.StreamRing(S, n, R=R, history=pkg.fm_channels_fir_history_samples(R, T))
    taps, d_incs = dev(torch, h), incs_tensor(torch, incs)
    for k in range(6):
        ring.load(parts[k])
        if k % 2 == 0:
            got = sess.channels(parts[k], n, incs)
            want, _ = pkg.fm_channels_exec(ring, d_incs, k * n, taps=taps)
            assert np.array_equal(got, want.cpu().numpy()), k
            plain.chain(parts[k], n, None, np.empty((S, n_audio), np.float32))
        else:
            outs = []
            for s in (sess, plain):
                db, au = np.empty((S, n // 1024, 1024), np.float32), np.empty((S, n_audio), np.float32)
                s.chain(parts[k], n, db, au)
                outs.append((db, au))
            assert all(np.array_equal(x, y) for x, y in zip(*outs)), k
        ring.carry()
    sess.close()
    plain.close()


def test_history_calls_refuse_before_launch(pkg):
    """b200_fm_history_reset / _carry refuse a down factor outside [1, 256] and a NULL pointer; all four history calls
    refuse a pointer that is not 16-byte aligned, and say so in b200_last_error().  Refused calls never touch the
    pointer, so fake addresses are safe."""
    L = pkg.lib()
    fake, stride, n = 1 << 20, 1 << 20, 1 << 20
    before = pkg.launch_count()
    for R, p in ((0, fake), (257, fake), (10, None)):
        ptr = C.c_void_p(p) if p else None
        assert L.b200_fm_history_reset(ptr, stride, 1, R, None) == B200_ERR_ARG, (R, p)
        assert L.b200_fm_history_carry(ptr, stride, 1, n, R, None) == B200_ERR_ARG, (R, p)
    odd = C.c_void_p(fake + 1)
    calls = {
        "history reset": [lambda: L.b200_iq_history_reset(odd, stride, 1, 320, None),
                          lambda: L.b200_fm_history_reset(odd, stride, 1, 10, None)],
        "history carry": [lambda: L.b200_iq_history_carry(odd, stride, 1, n, 320, None),
                          lambda: L.b200_fm_history_carry(odd, stride, 1, n, 10, None)],
    }
    for name, fns in calls.items():
        for fn in fns:
            assert not L.b200_session_create_r(0, 5120, 10)     # a different error first
            other = pkg.binding.last_error()
            assert fn() == B200_ERR_ALIGN, name
            msg = pkg.binding.last_error()
            assert msg != other and name in msg, (name, msg)
    assert pkg.launch_count() == before
