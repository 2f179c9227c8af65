"""FM channels with a FIR channel filter (b200_fm_channels_exec_fir, b200_session_set_channel_filter).

Definition (include/b200sdr.h): with y[n] the mixed sample of b200_fm_channels_exec and h[0..T-1] real taps,
b[m] = sum_{k<T} h[k] y[mR + R - T + k]; the demodulator after b is unchanged.  T = R with h = 1 is the boxcar.
mix_fir below restates that in float64; the rest of the oracle (demodulate, offsets_for, ...) is
test_gpu_fm_channels.py's.
"""
import ctypes as C
import math

import numpy as np
import pytest

from test_gpu_fm_channels import FS, batch_len, demodulate, incs_tensor, mix_boxcar, offsets_for, tone_power
from test_gpu_fm_rates import SM_SMEM, WALK, short_tile, sm_count, tiles_per_stream

FC_T = 62


def mixed(iq, inc, n0=0):
    """y[n] of the definition, float64, for u8 IQ [n, 2] whose first sample has absolute index n0."""
    iq = np.asarray(iq).reshape(-1, 2)
    n = (np.arange(len(iq), dtype=np.int64) + np.int64(n0)).astype(np.uint64)
    phi = (np.uint64(inc & 0xFFFFFFFF) * n) & np.uint64(0xFFFFFFFF)
    phs = phi.astype(np.int64) - (phi >= 2**31).astype(np.int64) * 2**32
    x = (iq[:, 0].astype(np.float64) - 128.0) + 1j * (iq[:, 1].astype(np.float64) - 128.0)
    if inc & 0xFFFFFFFF:
        x = x * np.exp(-1j * np.pi * phs.astype(np.float64) / 2.0**31)
    return x


def mix_fir(iq, R, inc, h, n0=0):
    """f64 baseband b[m] = sum_{k<T} h[k] y[mR + R - T + k] of a batch whose history mixes to zero (all 128: stream
    start, or a ring reset at any position)."""
    h = np.asarray(h, np.float64)
    T = len(h)
    P = max(T - R, 0)
    y = np.concatenate([np.zeros(P, np.complex128), mixed(iq, inc, n0)])
    M = (len(y) - P) // R
    out = np.empty(M, np.complex128)
    k = np.arange(T)
    step = max(1, (1 << 21) // T)
    for m0 in range(0, M, step):
        m = np.arange(m0, min(M, m0 + step))
        out[m] = (y[(m * R + R - T + P)[:, None] + k[None, :]] * h).sum(axis=1)
    return out


def kaiser_transition_hz(T, atten_db, fs=FS):
    """Kaiser's transition width for T taps and atten_db of stopband: T - 1 = (A - 7.95) / (2.285 dw)."""
    return (atten_db - 7.95) / (2.285 * (T - 1)) / (2 * np.pi) * fs


# Selectivity: a wanted station (1 kHz tone) at 0 Hz and a neighbour 20 dB stronger (2.5 kHz tone), both with the 75
# kHz deviation of broadcast FM, R = 10.  The float64 oracle gives these audio margins (wanted tone over the
# neighbour's tone, in dB) in the wanted channel:
#   neighbour at +200 kHz: boxcar -12.5, designed 80 kHz / 60 dB / 167 taps 42.3, 80 kHz / 70 dB / 199 taps 42.0
#   neighbour at +300 kHz: boxcar -12.5, 167 taps 42.3, 199 taps 42.2
# With the boxcar the neighbour captures the discriminator.  The GPU must show at least:
SELECTIVITY_MARGIN_DB = 30.0
SEL_R = 10
SEL_N = 4 * SEL_R * FC_T * 40
SEL_FILTERS = ((167, 60.0), (199, 70.0))


def neighbour_scene(synth, offset_hz, seed=70):
    w = synth.s3_fm(SEL_N, seed=seed, deviation=75e3, amplitude=10.0, sigma=0.5, tones=(1000.0,)).astype(np.float64)
    nb = synth.s3_fm(SEL_N, seed=seed + 1, deviation=75e3, carrier=offset_hz, amplitude=100.0, sigma=0.5,
                     tones=(2500.0,)).astype(np.float64)
    x = (w[:, 0] - 127.5) + 1j * (w[:, 1] - 127.5) + (nb[:, 0] - 127.5) + 1j * (nb[:, 1] - 127.5)
    return synth._quantise(x + (127.5 + 127.5j))


def wanted_margin(audio, rate=FS / (4 * SEL_R)):
    a = np.asarray(audio, np.float64)[256:]
    return 10 * np.log10(tone_power(a, 1000.0, rate) / tone_power(a, 2500.0, rate))


# ------------------------------------------------------------------------------------------------------------------
# CPU: the oracle, the design, the selectivity that motivates the filter
# ------------------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("R", [1, 7, 10, 256])
@pytest.mark.parametrize("inc", [0, 123_456_789, 2**31, 2**32 - 977])
def test_oracle_with_boxcar_taps_is_mix_boxcar(synth, R, inc):
    iq = synth.s1_noise(4 * R * 64, seed=R)
    for n0 in (0, 4 * R * 1000):
        assert np.array_equal(mix_fir(iq, R, inc, np.ones(R), n0), mix_boxcar(iq, R, inc, n0))


@pytest.mark.parametrize("R,T,cutoff,atten", [(10, 167, 80e3, 60.0), (10, 199, 80e3, 70.0), (10, 101, 60e3, 40.0),
                                              (1, 33, 500e3, 50.0), (64, 1024, 10e3, 80.0), (3, 200, 250e3, 60.0)])
def test_filter_design(pkg, R, T, cutoff, atten):
    h = pkg.fm_channel_filter(R, T, cutoff, atten)
    assert h.dtype == np.float32 and h.shape == (T,)
    assert np.array_equal(h, h[::-1])
    assert abs(h.astype(np.float64).sum() - R) <= 1e-6 * R
    nfft = 1 << 18
    H = np.abs(np.fft.rfft(h.astype(np.float64), nfft))
    f = np.arange(len(H)) * FS / nfft
    gain_db = 20 * np.log10(np.maximum(H, 1e-300) / H[0])
    stop = f >= cutoff + kaiser_transition_hz(T, atten)
    assert gain_db[stop].max() <= -(atten - 1.0), gain_db[stop].max()
    # the -6 dB point sits at the cutoff
    assert abs(gain_db[np.argmin(np.abs(f - cutoff))] + 6.02) < 0.5


def test_filter_design_refusals(pkg):
    L = pkg.lib()
    out = np.full(8, 7.0, np.float32)
    ok = (10, 8, 80e3, 60.0, FS)
    assert L.b200_fm_channel_filter_design(*ok, out.ctypes.data) == 0
    out[:] = 7.0
    for args in ((0, 8, 80e3, 60.0, FS), (257, 8, 80e3, 60.0, FS), (10, 0, 80e3, 60.0, FS), (10, 1025, 80e3, 60.0, FS),
                 (10, 8, 0.0, 60.0, FS), (10, 8, FS / 2, 60.0, FS), (10, 8, -1e3, 60.0, FS), (10, 8, float("nan"), 60.0, FS),
                 (10, 8, 80e3, float("nan"), FS), (10, 8, 80e3, -1.0, FS), (10, 8, 80e3, 60.0, 0.0),
                 (10, 8, 80e3, 60.0, -FS), (10, 8, 80e3, 60.0, float("nan")), (10, 8, 80e3, 60.0, float("inf"))):
        assert L.b200_fm_channel_filter_design(*args, out.ctypes.data) == -1, args
        assert (out == 7.0).all()
    assert L.b200_fm_channel_filter_design(*ok, None) == -1


def test_history_samples(pkg):
    H = pkg.fm_channels_fir_history_samples
    assert H(10, 10) == 320 and H(10, 1) == 320 and H(10, 200) == 512
    assert H(7, 300) == 224 + 293 + 3                       # rounded up to a multiple of 8
    assert H(1, 1024) == 1056 and H(256, 1024) == 8192 + 768
    assert all(H(R, T) % 8 == 0 and H(R, T) >= 32 * R + max(T - R, 0) for R in (1, 3, 7, 109) for T in (1, 5, 77, 1024))
    L = pkg.lib()
    for R, T in ((0, 10), (257, 10), (10, 0), (10, 1025)):
        assert L.b200_fm_channels_fir_history_samples(R, T) == -1


def test_history_calls_refuse_bad_lengths(pkg):
    """b200_iq_history_reset / _carry refuse a length that is not a positive multiple of 8 or is past
    B200_IQ_MAX_HISTORY_SAMPLES (its byte count would overflow an int) before touching the pointer."""
    L = pkg.lib()
    fake = C.c_void_p(1 << 20)
    for h in (0, -8, 4, 12, 2**30, 2**31 - 8):
        assert L.b200_iq_history_reset(fake, 1 << 20, 1, h, None) == -1, h
        assert L.b200_iq_history_carry(fake, 1 << 20, 1, 2**31, h, None) == -1, h


@pytest.mark.parametrize("offset", [200e3, 300e3])
def test_selectivity_oracle(pkg, synth, offset):
    iq = neighbour_scene(synth, offset)
    box = wanted_margin(demodulate(mix_boxcar(iq, SEL_R, 0)))
    assert box < SELECTIVITY_MARGIN_DB, box
    for T, A in SEL_FILTERS:
        h = pkg.fm_channel_filter(SEL_R, T, 80e3, A)
        m = wanted_margin(demodulate(mix_fir(iq, SEL_R, 0, h)))
        assert m > SELECTIVITY_MARGIN_DB + 6.0, (T, A, m)


# ------------------------------------------------------------------------------------------------------------------
# GPU
# ------------------------------------------------------------------------------------------------------------------

def fir_ring(pkg, iq, R, T):
    ring = pkg.StreamRing(iq.shape[0], iq.shape[1], R=R, history=pkg.fm_channels_fir_history_samples(R, T))
    ring.load(iq)
    return ring


def design(pkg, R, T):
    """A low-pass for channel tests: cutoff 0.4 fs / R (below fs / 2), 60 dB."""
    return pkg.fm_channel_filter(R, T, min(0.4 * FS / R, 0.45 * FS), 60.0)


def dev(torch, h):
    return torch.as_tensor(np.ascontiguousarray(h, np.float32)).cuda()


@pytest.mark.gpu
@pytest.mark.parametrize("R", [1, 3, 5, 7, 10, 12, 16, 64, 256])
def test_boxcar_taps_are_the_boxcar(pkg, synth, cuda, R):
    """T = R, h = 1: at inc = 0 the baseband is the integer CIC output and the audio b200_fm_channels_exec's, bit for
    bit; at other offsets within the boxcar's tolerance of the oracle."""
    torch = cuda
    n = batch_len(R, 62 * 3 + 10)
    S, Ch = 3, 2
    iq = np.stack([synth.s3_fm(n, seed=10 + s) if s != 1 else synth.s1_noise(n, seed=10 + s) for s in range(S)])
    ring = fir_ring(pkg, iq, R, R)
    ones = dev(torch, np.ones(R))
    _, dec = pkg.fm_exec(ring, decimated=True)
    zero = incs_tensor(torch, np.zeros((S, Ch)))
    box_audio, _ = pkg.fm_channels_exec(ring, zero, 0)
    audio, bb = pkg.fm_channels_exec(ring, zero, 0, baseband=True, taps=ones)
    torch.cuda.synchronize()
    dec = dec.cpu().numpy()
    for c in range(Ch):
        assert np.array_equal(bb[:, c].cpu().numpy(), dec.astype(np.float32))
    assert torch.equal(audio, box_audio)
    incs = offsets_for(R, S, Ch, np.random.default_rng(R))
    audio, bb = pkg.fm_channels_exec(ring, incs_tensor(torch, incs), 4 * R * 77, baseband=True, taps=ones)
    audio, bb = audio.cpu().numpy(), bb.cpu().numpy()
    for s in range(S):
        for c in range(Ch):
            ref = mix_boxcar(iq[s], R, int(incs[s, c]), 4 * R * 77)
            err = max(np.abs(bb[s, c, :, 0] - ref.real).max(), np.abs(bb[s, c, :, 1] - ref.imag).max())
            assert err <= 4e-6 * 128 * R, (s, c, err)
            assert np.abs(audio[s, c] - demodulate(bb[s, c])).max() <= 1e-4


def oracle_cases():
    out = []
    for R in (10, 1, 7, 109, 110, 256):
        for T in sorted({1, R - 1, R + 1, 8 * R + 3, 200, 1024}):
            if 1 <= T <= 1024:
                out.append((R, T))
    return out


def check_against_oracle(bb, audio, iq, incs, R, h, first, streams, channels):
    tol_bb = 4e-6 * 128 * float(np.abs(h.astype(np.float64)).sum())
    for s in streams:
        for c in channels:
            ref = mix_fir(iq[s], R, int(incs[s, c]), h, first)
            err = max(np.abs(bb[s, c, :, 0] - ref.real).max(), np.abs(bb[s, c, :, 1] - ref.imag).max())
            assert err <= tol_bb, (s, c, err, tol_bb)
            assert np.abs(audio[s, c] - demodulate(bb[s, c])).max() <= 1e-4, (s, c)


@pytest.mark.gpu
@pytest.mark.parametrize("R,T", oracle_cases())
def test_fir_against_oracle(pkg, synth, cuda, R, T):
    torch = cuda
    rng = np.random.default_rng(R * 2000 + T)
    S, Ch = 3, 3
    n = batch_len(R, 62 * 2 + 6)
    iq = np.stack([synth.s3_fm(n, seed=20 + s, carrier=150_000.0 * (s - 1)) if s != 2 else synth.s1_noise(n, seed=22)
                   for s in range(S)])
    incs = offsets_for(R, S, Ch, rng)
    h = design(pkg, R, T)
    ring = fir_ring(pkg, iq, R, T)
    audio, bb = pkg.fm_channels_exec(ring, incs_tensor(torch, incs), 0, baseband=True, taps=dev(torch, h))
    check_against_oracle(bb.cpu().numpy(), audio.cpu().numpy(), iq, incs, R, h, 0, range(S), range(Ch))


def fir_ctas_per_sm(R, T):
    """Upper bound on resident FIR CTAs per SM: the shared memory of one channel per group (the least the launcher
    uses) and 7 CTAs of 288 threads."""
    L = T - R
    stage = 2 * (280 * R + L + ((-L) & 7))
    stages = 2 if 2 * stage <= 120 * 1024 else 1
    smem = stages * stage + T * 16 + (288 + 144) * 4 + 16
    return max(1, min(2048 // 288, SM_SMEM // (smem + 1024)))


@pytest.mark.gpu
@pytest.mark.parametrize("R,T", [(10, 200), (7, 300), (110, 1024), (256, 1024)])
def test_fir_walk_tiles(pkg, cuda, synth, R, T):
    """Every resident CTA walks at least 3 tiles (refills and mbarrier parity flips), an odd prime number of tiles per
    stream so CTAs cross stream boundaries mid-walk, and a short last tile."""
    torch = cuda
    S, Ch = 3, 3
    workers = sm_count(pkg) * fir_ctas_per_sm(R, T)
    tps = tiles_per_stream(workers, S)
    n_audio = (tps - 1) * FC_T + short_tile(FC_T)
    n = 4 * R * n_audio
    assert n % 8 == 0 and -(-n_audio // FC_T) == tps and S * tps >= WALK * workers
    iq = np.stack([synth.s3_fm(n, seed=80 + s, carrier=-120e3 * s) for s in range(S)])
    incs = offsets_for(R, S, Ch, np.random.default_rng(T))
    h = design(pkg, R, T)
    first = 4 * R * 4321
    ring = fir_ring(pkg, iq, R, T)
    audio, bb = pkg.fm_channels_exec(ring, incs_tensor(torch, incs), first, baseband=True, taps=dev(torch, h))
    check_against_oracle(bb.cpu().numpy(), audio.cpu().numpy(), iq, incs, R, h, first, (0, S - 1), range(Ch))


@pytest.mark.gpu
@pytest.mark.parametrize("R,T", [(10, 200), (7, 300), (3, 1024)])
def test_fir_batches_equal_one_long_batch(pkg, synth, cuda, R, T):
    """Three batches with carry against one long batch, bit for bit.  (7, 300) and (3, 1024) reach back T - R > 32 R
    samples, past the boxcar's history."""
    torch = cuda
    H = pkg.fm_channels_fir_history_samples(R, T)
    n = max(batch_len(R, 62 * 2 + 20), batch_len(R, -(-H // (4 * R))))
    S = 2
    iq = np.stack([synth.s3_fm(3 * n, seed=30 + s, carrier=-200_000.0) for s in range(S)])
    incs = incs_tensor(torch, [[round(f / FS * 2**32) & 0xFFFFFFFF for f in (-200e3, 0.0, 333e3, 1e6)]] * S)
    taps = dev(torch, design(pkg, R, T))
    a_long, b_long = pkg.fm_channels_exec(fir_ring(pkg, iq, R, T), incs, 0, baseband=True, taps=taps)
    ring = pkg.StreamRing(S, n, R=R, history=H)
    parts_a, parts_b = [], []
    for k in range(3):
        ring.load(np.ascontiguousarray(iq[:, k * n:(k + 1) * n]))
        a, b = pkg.fm_channels_exec(ring, incs, k * n, baseband=True, taps=taps)
        parts_a.append(a.clone())
        parts_b.append(b.clone())
        ring.carry()
    torch.cuda.synchronize()
    assert torch.equal(torch.cat(parts_a, dim=2), a_long)
    assert torch.equal(torch.cat(parts_b, dim=2), b_long)


@pytest.mark.gpu
@pytest.mark.parametrize("first", [(2**33 // 40 + 1234) * 40, (2**62 // 40 - 5000) * 40])
def test_fir_far_stream_positions(pkg, synth, cuda, first):
    torch = cuda
    R, T, n = 10, 200, batch_len(10, 62 * 3)
    iq = synth.s3_fm(n, seed=44, carrier=300e3)[None]
    incs = np.array([[round(300e3 / FS * 2**32), round(-777_777.0 / FS * 2**32) & 0xFFFFFFFF, 2**31 - 1]])
    h = design(pkg, R, T)
    ring = fir_ring(pkg, iq, R, T)         # history all 128: mixes to zero at any position
    audio, bb = pkg.fm_channels_exec(ring, incs_tensor(torch, incs), first, baseband=True, taps=dev(torch, h))
    check_against_oracle(bb.cpu().numpy(), audio.cpu().numpy(), iq, incs, R, h, first, (0,), range(3))


@pytest.mark.gpu
@pytest.mark.parametrize("R,T", [(10, 160), (12, 1024)])
def test_fir_channels_are_independent(pkg, synth, cuda, R, T):
    torch = cuda
    n = batch_len(R, 62 * 3)
    S, Ch = 2, 11
    rng = np.random.default_rng(9)
    iq = np.stack([synth.s3_fm(n, seed=50 + s, carrier=90e3) for s in range(S)])
    incs = rng.integers(0, 2**32, size=(S, Ch), dtype=np.int64)
    taps = dev(torch, design(pkg, R, T))
    ring = fir_ring(pkg, iq, R, T)
    a_all, b_all = pkg.fm_channels_exec(ring, incs_tensor(torch, incs), 40 * R, baseband=True, taps=taps)
    for c in range(Ch):
        a1, b1 = pkg.fm_channels_exec(ring, incs_tensor(torch, incs[:, c:c + 1]), 40 * R, baseband=True, taps=taps)
        assert torch.equal(a1[:, 0], a_all[:, c]) and torch.equal(b1[:, 0], b_all[:, c])
    perm = rng.permutation(Ch)
    a_p, b_p = pkg.fm_channels_exec(ring, incs_tensor(torch, incs[:, perm]), 40 * R, baseband=True, taps=taps)
    assert torch.equal(a_p, a_all[:, perm]) and torch.equal(b_p, b_all[:, perm])


@pytest.mark.gpu
@pytest.mark.parametrize("offset", [200e3, 300e3])
def test_selectivity(pkg, synth, cuda, offset):
    torch = cuda
    iq = neighbour_scene(synth, offset)[None]
    zero = incs_tensor(torch, np.zeros((1, 1)))
    for T, A in SEL_FILTERS:
        ring = fir_ring(pkg, iq, SEL_R, T)
        audio, _ = pkg.fm_channels_exec(ring, zero, 0, taps=dev(torch, pkg.fm_channel_filter(SEL_R, T, 80e3, A)))
        m = wanted_margin(audio.cpu().numpy()[0, 0])
        assert m > SELECTIVITY_MARGIN_DB, (T, A, m)
    box, _ = pkg.fm_channels_exec(fir_ring(pkg, iq, SEL_R, SEL_R), zero, 0)
    assert wanted_margin(box.cpu().numpy()[0, 0]) < SELECTIVITY_MARGIN_DB


@pytest.mark.gpu
def test_fir_arguments_refused_before_launch(pkg, synth, cuda):
    torch = cuda
    R, n, S, T = 10, 4960, 2, 200
    ring = fir_ring(pkg, np.stack([synth.s1_noise(n, seed=s) for s in range(S)]), R, T)
    incs = incs_tensor(torch, np.zeros((S, 32)))
    audio = torch.empty((S * 33, n // 40 + 8), dtype=torch.float32, device="cuda")
    taps = torch.ones(1026, dtype=torch.float32, device="cuda")
    bb = torch.empty((S * 2, n // R, 2), dtype=torch.float32, device="cuda")
    L = pkg.lib()
    iq = ring.batch.data_ptr()

    def call(iq=iq, stride=ring.stride_bytes, n_samples=n, first=0, inc=incs.data_ptr(), Ch=2, au=audio.data_ptr(),
             R=R, tp=taps.data_ptr(), T=T, ast=audio.stride(0), bbp=0, bbs=0):
        return L.b200_fm_channels_exec_fir(C.c_void_p(iq), stride, S, n_samples, R, first,
                                           C.c_void_p(inc) if inc else None, Ch, C.c_void_p(au) if au else None,
                                           ast, C.c_void_p(bbp) if bbp else None, bbs,
                                           C.c_void_p(tp) if tp else None, T, None)

    torch.cuda.synchronize()
    assert call() == 0
    torch.cuda.synchronize()
    before = pkg.launch_count()
    cases = [(dict(T=0), -1), (dict(tp=0, T=0), -1), (dict(T=1025), -1), (dict(T=-3), -1), (dict(tp=0), -1), (dict(tp=taps.data_ptr() + 2), -4),
             (dict(Ch=0), -1), (dict(Ch=33), -1), (dict(first=-40), -1), (dict(first=20), -1), (dict(first=41), -1),
             (dict(n_samples=n - 20), -1), (dict(n_samples=-40), -1),
             (dict(R=5, n_samples=60), -1), (dict(R=0), -1), (dict(R=257), -1),
             (dict(inc=0), -1), (dict(au=0), -1), (dict(iq=iq + 2), -4), (dict(stride=ring.stride_bytes + 8), -4),
             (dict(inc=incs.data_ptr() + 2), -4), (dict(au=audio.data_ptr() + 2), -4),
             # rows closer than a row's length would overlap
             (dict(ast=n // 40 - 1), -1), (dict(bbp=bb.data_ptr(), bbs=n // R - 1), -1)]
    for kw, want in cases:
        assert call(**kw) == want, kw
        assert pkg.binding.last_error()
    assert pkg.launch_count() == before


@pytest.mark.gpu
def test_binding_refuses_a_ring_history_too_short(pkg, synth, cuda):
    """A ring with the boxcar's 32 R of history cannot feed 167 taps (480 samples): the kernel would read before the
    rows, so the binding refuses before anything is launched.  StreamRing itself refuses a history below 32 R or not
    a multiple of 8."""
    torch = cuda
    R, n, S = 10, 4960, 2
    ring = pkg.StreamRing(S, n, R=R)
    ring.load(np.stack([synth.s1_noise(n, seed=s) for s in range(S)]))
    taps = dev(torch, pkg.fm_channel_filter(R, 167, 80e3, 60.0))
    inc = incs_tensor(torch, np.zeros((S, 1)))
    torch.cuda.synchronize()
    before = pkg.launch_count()
    with pytest.raises(pkg.B200Error):
        pkg.fm_channels_exec(ring, inc, 0, taps=taps)
    for h in (32 * R - 8, 32 * R + 4):
        with pytest.raises(pkg.B200Error):
            pkg.StreamRing(S, n, R=R, history=h)
    assert pkg.launch_count() == before
    ok = fir_ring(pkg, ring.batch.cpu().numpy(), R, 167)
    pkg.fm_channels_exec(ok, inc, 0, taps=taps)
    assert pkg.launch_count() > before


@pytest.mark.gpu
def test_session_channel_filter(pkg, synth, cuda):
    torch = cuda
    R, T, S = 10, 200, 3
    n = 2 * int(pkg.lib().b200_chain_tile_samples(R))
    iq = np.stack([synth.s3_fm(4 * n, seed=60 + s, carrier=-250e3) for s in range(S)])
    parts = [np.ascontiguousarray(iq[:, k * n:(k + 1) * n]) for k in range(4)]
    incs = np.array([[pkg.fm_channel_tune(f, FS) for f in (-250e3, 0.0, 410e3)]] * S, dtype=np.int64)
    h = pkg.fm_channel_filter(R, T, 80e3, 70.0)

    # the session form equals the device form
    sess = pkg.Session(S, n, R=R)
    sess.set_channel_filter(h)
    got = [sess.channels(parts[k], n, incs) for k in range(4)]
    ring = pkg.StreamRing(S, n, R=R, history=pkg.fm_channels_fir_history_samples(R, T))
    for k in range(4):
        ring.load(parts[k])
        a, _ = pkg.fm_channels_exec(ring, incs_tensor(torch, incs), k * n, taps=dev(torch, h))
        assert np.array_equal(a.cpu().numpy(), got[k]), k
        ring.carry()
    # only at position 0
    with pytest.raises(pkg.B200Error):
        sess.set_channel_filter(h)
    assert pkg.lib().b200_session_set_channel_filter(C.c_void_p(sess.h), None, 0) == -1

    # chain and products read only the last 32 R history samples: the same with and without a filter
    plain = pkg.Session(S, n, R=R)
    sess.reset()
    sess.set_channel_filter(h)
    n_audio = n // (4 * R)
    for k in range(4):
        outs = []
        for s in (plain, sess):
            if k % 2 == 0:
                db, au = np.empty((S, n // 1024, 1024), np.float32), np.empty((S, n_audio), np.float32)
                s.chain(parts[k], n, db, au)
                outs.append((db, au))
            else:
                au, avg = np.empty((S, n_audio), np.float32), np.empty((S, 1024), np.uint8)
                s.products(parts[k], n, au, avg)
                outs.append((au, avg))
        assert all(np.array_equal(x, y) for x, y in zip(*outs)), k
    # channel calls interleaved with them still see the filtered history: position 4n of the same IQ
    more = np.stack([synth.s3_fm(n, seed=90 + s) for s in range(S)])
    a = sess.channels(more, n, incs)
    ring.load(more)
    want, _ = pkg.fm_channels_exec(ring, incs_tensor(torch, incs), 4 * n, taps=dev(torch, h))
    assert np.array_equal(a, want.cpu().numpy())

    # n_taps = 0 goes back to the boxcar
    sess.reset()
    sess.set_channel_filter(None)
    plain.reset()
    for k in range(2):
        assert np.array_equal(sess.channels(parts[k], n, incs), plain.channels(parts[k], n, incs)), k
    sess.close()
    plain.close()

    # a history longer than the session's largest batch is refused (R = 1: 1056 samples, batches of 1024)
    small = pkg.Session(1, 1024, R=1)
    with pytest.raises(pkg.B200Error):
        small.set_channel_filter(np.ones(1024, np.float32))
    small.set_channel_filter(np.ones(64, np.float32))
    small.close()
