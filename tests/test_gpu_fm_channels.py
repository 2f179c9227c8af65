"""FM channels at frequency offsets inside one dongle's band (b200_fm_channels_exec, b200_session_channels).

Definition (include/b200sdr.h): sample n of a stream (int64 from stream start) is mixed with
exp(-j 2 pi phi(n) / 2^32), phi(n) = (uint32)(inc * (uint64) n); the channel baseband is the reference's boxcar of R
mixed samples (resample.c:21-40, no 1/128), and the audio is the reference's demodulator (audio_main.c:110-139) on it.
The oracle below restates that in float64: mix, boxcar, atan2_approx, first difference, limiter, the 11-tap half-band
twice.  Its atan2_approx is the device's form (copysign, so -0.0 behaves as on the device; branch on |y| < |x|).
"""
import numpy as np
import pytest

HB = np.array([0.01824, 0.0, -0.11614, 0.0, 0.34790, 0.5, 0.34790, 0.0, -0.11614, 0.0, 0.01824])
FS = 2_048_000.0


def mix_boxcar(iq, R, inc, n0=0):
    """f64 baseband b[m] = sum_{k<R} y[mR + k] of u8 IQ [n, 2] whose first sample has absolute index n0."""
    iq = np.asarray(iq).reshape(-1, 2)
    n = (np.arange(len(iq), dtype=np.int64) + np.int64(n0)).astype(np.uint64)
    phi = (np.uint64(inc & 0xFFFFFFFF) * n) & np.uint64(0xFFFFFFFF)
    phs = phi.astype(np.int64) - (phi >= 2**31).astype(np.int64) * 2**32          # [-2^31, 2^31)
    x = (iq[:, 0].astype(np.float64) - 128.0) + 1j * (iq[:, 1].astype(np.float64) - 128.0)
    if inc & 0xFFFFFFFF:
        x = x * np.exp(-1j * np.pi * phs.astype(np.float64) / 2.0**31)
    return x.reshape(-1, R).sum(axis=1)


def atan2_approx(y, x):
    y = np.asarray(y, dtype=np.float64)
    x = np.asarray(x, dtype=np.float64)
    lt = np.abs(y) < np.abs(x)
    den = np.where(lt, x * x + 0.28 * y * y, y * y + 0.28 * x * x)
    with np.errstate(divide="ignore", invalid="ignore"):
        q = x * y / den
    r = np.where(lt, q + np.where(x < 0, np.copysign(np.pi, y), 0.0), np.copysign(np.pi / 2, y) - q)
    return np.where(den == 0, 0.0, r)


def halfband(x):
    return np.convolve(x, HB)[:len(x)][::2]


def demodulate(b):
    """audio_main.c:110-139 in float64 from stream start (zero delay lines) on complex baseband b."""
    b = np.asarray(b)
    if b.dtype != np.complex128:
        b = b[..., 0].astype(np.float64) + 1j * b[..., 1].astype(np.float64)
    ph = atan2_approx(b.imag, b.real)
    d = np.clip(np.diff(ph, prepend=0.0), -1.0, 1.0)
    return halfband(halfband(d))


def reference_audio(iq, R, inc, n0=0):
    return demodulate(mix_boxcar(iq, R, inc, n0))


def tone_power(a, f, rate):
    t = np.arange(len(a)) / rate
    return abs(np.dot(a, np.exp(-2j * np.pi * f * t))) ** 2 / len(a) ** 2


def three_stations(n, seed=40):
    """Three s3_fm-style stations at distinct carriers inside +-fs/2, each with its own tone."""
    from importlib import import_module
    synth = import_module("rtl_ws_b200.synth")
    x = np.zeros(n, dtype=np.complex128)
    for i, (car, tone) in enumerate(STATIONS):
        u = synth.s3_fm(n, seed=seed + i, carrier=car, amplitude=40.0, sigma=1.0, tones=(tone,)).astype(np.float64)
        x += (u[:, 0] - 127.5) + 1j * (u[:, 1] - 127.5)
    return synth._quantise(x + (127.5 + 127.5j))


STATIONS = ((-500_000.0, 1_000.0), (100_000.0, 2_500.0), (700_000.0, 4_000.0))
# own tone over the strongest other station's tone in a channel's audio, in dB.  The float64 oracle on the CPU gives
# 32.8, 51.9 and 50.2 dB for the three channels (test_station_separation_oracle checks 6 dB above this threshold);
# the GPU must show at least this:
STATION_MARGIN_DB = 26.0


def station_margins(audio_rows, rate):
    skip = 256
    out = []
    for c, row in enumerate(audio_rows):
        p = [tone_power(np.asarray(row[skip:], np.float64), tone, rate) for _, tone in STATIONS]
        others = max(p[i] for i in range(len(STATIONS)) if i != c)
        out.append(10 * np.log10(p[c] / others))
    return out


# ------------------------------------------------------------------------------------------------------------------
# CPU: the oracle pinned to the reference, the tune encoding
# ------------------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("R", [10, 5, 12])
@pytest.mark.parametrize("kind", ["s3_fm", "s1_noise"])
def test_oracle_at_zero_offset_is_the_reference(po, synth, R, kind):
    n = 4 * R * 8 * 64
    iq = synth.s3_fm(n, seed=7) if kind == "s3_fm" else synth.s1_noise(n, seed=7)
    b = mix_boxcar(iq, R, 0)
    _, dec, _ = po.cic_decimate(R, iq)
    assert np.array_equal(b.real, dec[:, 0].astype(np.float64))
    assert np.array_equal(b.imag, dec[:, 1].astype(np.float64))
    _, _, ref_audio, _ = po.fm_demodulate(dec)
    assert np.abs(demodulate(b) - ref_audio).max() < 1e-4


def test_oracle_mixes_a_carrier_to_dc(synth):
    """A station at +f Hz mixed by the increment of +f is the same station generated at 0 Hz, up to the carrier's
    constant phase 2 pi f / fs (s3_fm's phase includes sample 0), the u8 rounding of the two waveforms and synth's
    centre of 127.5 (a DC of -0.5 - 0.5j per sample, which the mixer moves away from 0 Hz)."""
    n, R, f = 40960, 10, 204_800.0
    b0 = mix_boxcar(synth.s3_fm(n, seed=3, sigma=0.0), R, 0)
    bf = mix_boxcar(synth.s3_fm(n, seed=3, sigma=0.0, carrier=f), R, int(round(f / FS * 2**32)))
    assert np.abs(bf - b0 * np.exp(2j * np.pi * f / FS)).max() < np.sqrt(2) * R
    assert np.abs(b0).min() > 900


def test_station_separation_oracle(synth):
    n, R = 4 * 10 * 62 * 40, 10
    iq = three_stations(n)
    rows = [reference_audio(iq, R, int(round(car / FS * 2**32))) for car, _ in STATIONS]
    m = station_margins(rows, FS / (4 * R))
    assert min(m) > STATION_MARGIN_DB + 6.0, m


def test_channel_tune_encoding(pkg):
    tune = pkg.fm_channel_tune
    assert tune(0.0, FS) == 0
    assert tune(FS / 4, FS) == 2**30
    assert tune(-FS / 4, FS) == 2**32 - 2**30                    # two's complement
    assert tune(100_000.0, FS) == round(100_000.0 / FS * 2**32)
    assert tune(-100_000.0, FS) == (2**32 - round(100_000.0 / FS * 2**32))
    assert tune(1.0, FS) == round(2**32 / FS)                     # 2097.152 -> 2097
    assert tune(FS / 2**32 * 2.5, FS) == 3                       # halves round away from zero
    assert tune(FS / 2, FS) == 2**31
    assert tune(-FS / 2, FS) == 2**31                            # -2^31 as uint32
    L = pkg.lib()
    import ctypes
    out = ctypes.c_uint32(12345)
    for off, fs in ((FS / 2 * (1 + 1e-12), FS), (-FS / 2 * (1 + 1e-12), FS), (0.0, 0.0), (0.0, -FS),
                    (float("nan"), FS), (0.0, float("nan")), (1e3, float("inf"))):
        assert L.b200_fm_channel_tune(off, fs, ctypes.byref(out)) == -1, (off, fs)
        assert out.value == 12345
    assert L.b200_fm_channel_tune(0.0, FS, None) == -1


# ------------------------------------------------------------------------------------------------------------------
# GPU
# ------------------------------------------------------------------------------------------------------------------

def batch_len(R, n_audio):
    """n_samples holding at least n_audio audio samples, a multiple of 4R and of 8."""
    q = 4 * R * (2 if R % 2 else 1)
    return ((4 * R * n_audio + q - 1) // q) * q


def incs_tensor(torch, incs):
    a = np.ascontiguousarray(np.asarray(incs, dtype=np.int64) & 0xFFFFFFFF)
    return torch.as_tensor(a.astype(np.uint32).view(np.int32)).cuda()


def load_ring(pkg, iq, R):
    ring = pkg.StreamRing(iq.shape[0], iq.shape[1], R=R)
    ring.load(iq)
    return ring


@pytest.mark.gpu
@pytest.mark.parametrize("R", [10, 5, 12, 16, 1, 7, 64, 3, 256])
def test_zero_offset_is_fm_exec(pkg, synth, cuda, R):
    torch = cuda
    n = batch_len(R, 62 * 3 + 10)
    S, Ch = 3, 2
    iq = np.stack([synth.s3_fm(n, seed=10 + s) if s != 1 else synth.s1_noise(n, seed=10 + s) for s in range(S)])
    ring = load_ring(pkg, iq, R)
    audio, dec = pkg.fm_exec(ring, decimated=True)
    ch_audio, bb = pkg.fm_channels_exec(ring, incs_tensor(torch, np.zeros((S, Ch))), 0, baseband=True)
    torch.cuda.synchronize()
    dec, audio = dec.cpu().numpy(), audio.cpu().numpy()
    bb, ch_audio = bb.cpu().numpy(), ch_audio.cpu().numpy()
    for c in range(Ch):
        assert np.array_equal(bb[:, c], dec.astype(np.float32))
        assert np.abs(ch_audio[:, c] - audio).max() <= 1e-6


def offsets_for(R, S, Ch, rng):
    """Per stream and channel: +-fs/2, multiples of fs/R, small and random offsets."""
    fixed = [FS / 2, -FS / 2, FS / R, -2 * FS / R, 0.0, 123_456.7, -1.0]
    out = np.empty((S, Ch), dtype=np.int64)
    for s in range(S):
        for c in range(Ch):
            k = s * Ch + c
            f = fixed[k % len(fixed)] if k < 2 * len(fixed) else rng.uniform(-FS / 2, FS / 2)
            if abs(f) > FS / 2:
                f = np.sign(f) * FS / 2
            out[s, c] = round(f / FS * 2**32) & 0xFFFFFFFF
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("R,Ch", [(10, 1), (10, 3), (10, 10), (10, 32), (5, 3), (12, 10), (16, 32), (64, 3), (5, 32)])
def test_offsets_against_oracle(pkg, synth, cuda, R, Ch):
    torch = cuda
    rng = np.random.default_rng(R * 100 + Ch)
    S = 3
    n = batch_len(R, 62 * 4 + 6)
    iq = np.stack([synth.s3_fm(n, seed=20 + s, carrier=150_000.0 * (s - 1)) if s != 2 else synth.s1_noise(n, seed=22)
                   for s in range(S)])
    incs = offsets_for(R, S, Ch, rng)
    ring = load_ring(pkg, iq, R)
    audio, bb = pkg.fm_channels_exec(ring, incs_tensor(torch, incs), 0, baseband=True)
    torch.cuda.synchronize()
    audio, bb = audio.cpu().numpy(), bb.cpu().numpy()
    tol_bb = 4e-6 * 128 * R
    for s in range(S):
        for c in range(Ch):
            ref = mix_boxcar(iq[s], R, int(incs[s, c]))
            err = max(np.abs(bb[s, c, :, 0] - ref.real).max(), np.abs(bb[s, c, :, 1] - ref.imag).max())
            assert err <= tol_bb, (s, c, err)
            assert np.abs(audio[s, c] - demodulate(bb[s, c])).max() <= 1e-4, (s, c)


@pytest.mark.gpu
def test_rotation_accuracy_at_r1(pkg, synth, cuda):
    """At R = 1 the baseband IS x[n] exp(-j phi(n)): its error over |x| bounds the per-sample sin / cos error."""
    torch = cuda
    n = 8 * 62 * 4 * 4
    iq = synth.s1_noise(n, seed=5)[None]
    incs = np.array([[round(0.3183 * 2**32), 2**31 + 12345, 977]], dtype=np.int64)
    ring = load_ring(pkg, iq, 1)
    _, bb = pkg.fm_channels_exec(ring, incs_tensor(torch, incs), 4 * 1000, baseband=True)
    bb = bb.cpu().numpy()
    mag = np.abs((iq[0, :, 0] - 128.0) + 1j * (iq[0, :, 1] - 128.0))
    for c in range(3):
        ref = mix_boxcar(iq[0], 1, int(incs[0, c]), 4000)
        err = np.maximum(np.abs(bb[0, c, :, 0] - ref.real), np.abs(bb[0, c, :, 1] - ref.imag))
        ok = mag > 0
        assert (err[ok] / mag[ok]).max() < 2e-6


@pytest.mark.gpu
@pytest.mark.parametrize("R", [10, 7])
def test_batches_equal_one_long_batch(pkg, synth, cuda, R):
    torch = cuda
    n = batch_len(R, 62 * 2 + 20)
    S, Ch = 2, 4
    iq = np.stack([synth.s3_fm(3 * n, seed=30 + s, carrier=-200_000.0) for s in range(S)])
    incs = incs_tensor(torch, [[round(f / FS * 2**32) for f in (-200e3, 0.0, 333e3, 1e6)]] * S)
    long_ring = load_ring(pkg, iq, R)
    a_long, b_long = pkg.fm_channels_exec(long_ring, incs, 0, baseband=True)
    ring = pkg.StreamRing(S, n, R=R)
    parts_a, parts_b = [], []
    for k in range(3):
        ring.load(np.ascontiguousarray(iq[:, k * n:(k + 1) * n]))
        a, b = pkg.fm_channels_exec(ring, incs, k * n, baseband=True)
        parts_a.append(a.clone())
        parts_b.append(b.clone())
        ring.carry()
    torch.cuda.synchronize()
    assert torch.equal(torch.cat(parts_a, dim=2), a_long)
    assert torch.equal(torch.cat(parts_b, dim=2), b_long)


@pytest.mark.gpu
@pytest.mark.parametrize("first", [(2**33 // 40 + 1234) * 40, (2**62 // 40 - 5000) * 40])
def test_far_stream_positions(pkg, synth, cuda, first):
    torch = cuda
    R, n = 10, batch_len(10, 62 * 3)
    iq = synth.s3_fm(n, seed=44, carrier=300e3)[None]
    incs = np.array([[round(300e3 / FS * 2**32), round(-777_777.0 / FS * 2**32) & 0xFFFFFFFF, 2**31 - 1]])
    ring = load_ring(pkg, iq, R)           # history all 128: mixes to zero at any position
    audio, bb = pkg.fm_channels_exec(ring, incs_tensor(torch, incs), first, baseband=True)
    audio, bb = audio.cpu().numpy(), bb.cpu().numpy()
    for c in range(3):
        ref = mix_boxcar(iq[0], R, int(incs[0, c]), first)
        err = max(np.abs(bb[0, c, :, 0] - ref.real).max(), np.abs(bb[0, c, :, 1] - ref.imag).max())
        assert err <= 4e-6 * 128 * R
        assert np.abs(audio[0, c] - demodulate(bb[0, c])).max() <= 1e-4
    # the position matters: the same batch at 0 mixes with other phases
    other, _ = pkg.fm_channels_exec(ring, incs_tensor(torch, incs[:, :1]), 0)
    assert not np.array_equal(other.cpu().numpy()[0, 0], audio[0, 0]) or incs[0, 0] * first % 2**32 == 0


@pytest.mark.gpu
@pytest.mark.parametrize("R", [10, 12])
def test_channels_are_independent(pkg, synth, cuda, R):
    torch = cuda
    n = batch_len(R, 62 * 3)
    S, Ch = 2, 11
    rng = np.random.default_rng(9)
    iq = np.stack([synth.s3_fm(n, seed=50 + s, carrier=90e3) for s in range(S)])
    incs = rng.integers(0, 2**32, size=(S, Ch), dtype=np.int64)
    ring = load_ring(pkg, iq, R)
    a_all, b_all = pkg.fm_channels_exec(ring, incs_tensor(torch, incs), 40 * R, baseband=True)
    for c in range(Ch):
        a1, b1 = pkg.fm_channels_exec(ring, incs_tensor(torch, incs[:, c:c + 1]), 40 * R, baseband=True)
        assert torch.equal(a1[:, 0], a_all[:, c]) and torch.equal(b1[:, 0], b_all[:, c])
    perm = rng.permutation(Ch)
    a_p, b_p = pkg.fm_channels_exec(ring, incs_tensor(torch, incs[:, perm]), 40 * R, baseband=True)
    assert torch.equal(a_p, a_all[:, perm]) and torch.equal(b_p, b_all[:, perm])


@pytest.mark.gpu
def test_stations_separate(pkg, cuda):
    torch = cuda
    n, R = 4 * 10 * 62 * 40, 10
    iq = three_stations(n)[None]
    incs = np.array([[pkg.fm_channel_tune(car, FS) for car, _ in STATIONS]])
    ring = load_ring(pkg, iq, R)
    audio, _ = pkg.fm_channels_exec(ring, incs_tensor(torch, incs), 0)
    m = station_margins(audio.cpu().numpy()[0], FS / (4 * R))
    assert min(m) > STATION_MARGIN_DB, m


@pytest.mark.gpu
def test_arguments_refused_before_launch(pkg, synth, cuda):
    import ctypes as C
    torch = cuda
    R, n, S = 10, 4960, 2
    ring = load_ring(pkg, np.stack([synth.s1_noise(n, seed=s) for s in range(S)]), R)
    incs = incs_tensor(torch, np.zeros((S, 32)))
    audio = torch.empty((S * 33, n // 40 + 8), dtype=torch.float32, device="cuda")
    bb = torch.empty((S * 2, n // R, 2), dtype=torch.float32, device="cuda")
    L = pkg.lib()
    iq = ring.batch.data_ptr()

    def call(iq=iq, stride=ring.stride_bytes, n_samples=n, first=0, inc=incs.data_ptr(), Ch=2, au=audio.data_ptr(), R=R,
             ast=audio.stride(0), bbp=0, bbs=0):
        return L.b200_fm_channels_exec(C.c_void_p(iq), stride, S, n_samples, R, first, C.c_void_p(inc) if inc else None,
                                       Ch, C.c_void_p(au) if au else None, ast, C.c_void_p(bbp) if bbp else None, bbs,
                                       None)

    torch.cuda.synchronize()
    assert call() == 0
    torch.cuda.synchronize()
    before = pkg.launch_count()
    cases = [(dict(Ch=0), -1), (dict(Ch=33), -1), (dict(first=-40), -1), (dict(first=20), -1), (dict(first=41), -1),
             (dict(n_samples=n - 20), -1), (dict(n_samples=-40), -1),
             (dict(R=5, n_samples=60), -1), (dict(R=0), -1), (dict(R=257), -1),
             (dict(inc=0), -1), (dict(au=0), -1), (dict(iq=iq + 2), -4), (dict(stride=ring.stride_bytes + 8), -4),
             # rows closer than a row's length would overlap
             (dict(ast=n // 40 - 1), -1), (dict(bbp=bb.data_ptr(), bbs=n // R - 1), -1)]
    for kw, want in cases:
        assert call(**kw) == want, kw
        assert pkg.last_error() if hasattr(pkg, "last_error") else pkg.binding.last_error()
    assert pkg.launch_count() == before


@pytest.mark.gpu
@pytest.mark.parametrize("R", [10, 5])
def test_session_channels(pkg, synth, cuda, R):
    torch = cuda
    S, Ch = 3, 3
    tile = int(pkg.lib().b200_chain_tile_samples(R))
    n = tile * 2
    iq = np.stack([synth.s3_fm(4 * n, seed=60 + s, carrier=-250e3) for s in range(S)])
    incs = np.array([[pkg.fm_channel_tune(f, FS) for f in (-250e3, 0.0, 410e3)]] * S, dtype=np.int64)
    sess = pkg.Session(S, n, R=R)
    got = [sess.channels(np.ascontiguousarray(iq[:, k * n:(k + 1) * n]), n, incs) for k in range(4)]
    ring = pkg.StreamRing(S, n, R=R)
    for k in range(4):
        ring.load(np.ascontiguousarray(iq[:, k * n:(k + 1) * n]))
        a, _ = pkg.fm_channels_exec(ring, incs_tensor(torch, incs), k * n)
        assert np.array_equal(a.cpu().numpy(), got[k]), k
        ring.carry()

    # interleaved with chain calls: every call advances the position.  Channel calls at inc = 0 match fm_exec at
    # that position, and the chain calls return what a session that only runs chain calls returns
    n_audio = n // (4 * R)
    h_db = np.empty((S, n // 1024, 1024), np.float32)
    plain = pkg.Session(S, n, R=R)
    sess.reset()
    ring.reset()
    for k in range(4):
        part = np.ascontiguousarray(iq[:, k * n:(k + 1) * n])
        ring.load(part)
        ref, _ = pkg.fm_exec(ring)
        ref = ref.cpu().numpy()
        want = np.empty((S, n_audio), np.float32)
        plain.chain(part, n, h_db, want)
        if k % 2 == 0:
            h_au = np.empty((S, n_audio), np.float32)
            sess.chain(part, n, h_db, h_au)
            assert np.array_equal(h_au, want), k
        else:
            a = sess.channels(part, n, np.zeros((S, 1), np.int64))
            assert np.abs(a[:, 0] - ref).max() <= 1e-6, k
        ring.carry()
    # reset returns to position 0: the first batch gives the first result again
    sess.reset()
    assert np.array_equal(sess.channels(np.ascontiguousarray(iq[:, :n]), n, incs), got[0])
    sess.close()
    plain.close()
