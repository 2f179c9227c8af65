"""The FM kernels at down factors other than 10, sized from the machine so that every resident CTA or warp walks
several tiles, and the audio extensions at every rate a chain can produce.

Each FM kernel is persistent: a CTA (or a warp) walks tiles through a TMA ring, refilling a stage with the tile
two steps ahead and flipping the mbarrier parity every pass over the ring.  A test with fewer tiles than resident
workers never reaches the refill, the parity flip or a walk across a stream boundary.  So every case here computes
its size from b200_sm_count() and an UPPER bound on residency, and asserts that the tiles cover every worker at
least WALK times; the tile count per stream is an odd prime, so it is not a multiple of the grid and workers cross
stream boundaries mid-walk.

References: the CPU oracle's cic_decimate / fm_demodulate (the reference's own arithmetic) for b200_fm_exec, the
float64 channel oracle of test_gpu_fm_channels.py for b200_fm_channels_exec, a float64 sequential loop for the
de-emphasis and the oracle's atan2_approx for the device's atan2 forms.
"""
import functools
import math

import numpy as np
import pytest
from scipy.signal import lfilter

from test_gpu_fm import AUDIO_TOL, oracle_stream
from test_gpu_fm_channels import FS, demodulate, incs_tensor, mix_boxcar

WALK = 3                        # tiles every resident worker walks at least
SM_THREADS = 2048               # resident threads per SM (sm_100)
SM_SMEM = 228 * 1024            # shared memory per SM (sm_100); each CTA also reserves 1 KB of it


def sm_count(pkg):
    n = int(pkg.lib().b200_sm_count())
    assert n > 0
    return n


def is_prime(n):
    return n > 1 and all(n % k for k in range(2, math.isqrt(n) + 1))


def tiles_per_stream(workers, n_streams):
    """The least odd prime >= the tiles per stream that give every worker WALK tiles.  A prime is a multiple of
    the grid only if it equals it, and every grid here is a multiple of the SM count."""
    t = max(3, -(-WALK * workers // n_streams))
    while not is_prime(t):
        t += 1
    return t


def short_tile(T):
    """Audio samples in a stream's last tile: even (n_samples = 4 R n_audio must be a multiple of 8 for odd R)
    and less than T."""
    return max(2, (T // 2) & ~1)


# ---- b200_fm_exec ------------------------------------------------------------------------------------------------

def fm_tile_audio(R):
    """Audio samples per tile: 62 for fm_chain_warp_kernel (3 <= R <= 16); for fm_chain_kernel<0> the largest of
    128, 64, 32, 16, 8 whose staged bytes fit 32 KB (fm_tile_audio in fm_chain.cu)."""
    if 3 <= R <= 16:
        return 62
    T = 128
    while T > 8 and (4 * T + 32) * 2 * R > 32768:
        T >>= 1
    return T


def fm_workers(pkg, R):
    """Upper bound on the tiles b200_fm_exec has in flight: 64 warps per SM for the warp-per-tile kernel, 8 CTAs of
    256 threads per SM for fm_chain_kernel."""
    return sm_count(pkg) * (SM_THREADS // 32 if 3 <= R <= 16 else SM_THREADS // 256)


@functools.lru_cache(maxsize=None)
def fm_segment(kind, n_seg, seed):
    from importlib import import_module
    synth = import_module("rtl_ws_b200.synth")
    if kind == "fm":
        return synth.s3_fm(n_seg, seed=seed, deviation=75e3)
    # full scale: the CIC output reaches about 127 R, e.g. +-32512 at R = 256
    return synth.s3_fm(n_seg, seed=seed, deviation=25e3, carrier=3e3, amplitude=127.0, sigma=0.4)


def fm_streams(n, seed):
    """Three different streams of n samples: white bytes, an FM station, a full-scale FM station (the last two
    repeat a segment whose length is not a multiple of any tile)."""
    rng = np.random.default_rng(seed)
    noise = rng.integers(0, 256, size=(n, 2), dtype=np.uint8)
    fm = np.resize(fm_segment("fm", 1_000_003, 1), (n, 2))
    loud = np.resize(fm_segment("loud", 999_983, 2), (n, 2))
    return np.stack([noise, fm, loud])


def fm_size(pkg, R, n_streams):
    """(n_samples, tiles per stream) for a b200_fm_exec batch whose every worker walks >= WALK tiles."""
    T = fm_tile_audio(R)
    tps = tiles_per_stream(fm_workers(pkg, R), n_streams)
    n_audio = (tps - 1) * T + short_tile(T)
    n = 4 * R * n_audio
    assert n % 8 == 0 and -(-n_audio // T) == tps and n_audio % T != 0
    assert n_streams * tps >= WALK * fm_workers(pkg, R)
    return n, tps


@pytest.mark.gpu
@pytest.mark.parametrize("R", [3, 7, 12, 16, 1, 2, 30, 31, 56, 57, 102, 103, 170, 171, 255, 256])
def test_fm_exec_walks_tiles(pkg, cuda, po, R):
    """R = 3..16: fm_chain_warp_kernel (odd and even R); otherwise fm_chain_kernel<0> on both sides of every tile
    size boundary (T = 128 up to R = 30, 64 to 56, 32 to 102, 16 to 170, 8 to 256)."""
    torch = cuda
    S = 3
    n, _ = fm_size(pkg, R, S)
    iqs = fm_streams(n, seed=R)
    ring = pkg.StreamRing(S, n, R=R)
    ring.load(iqs)
    audio, dec = pkg.fm_exec(ring, decimated=True)
    torch.cuda.synchronize()
    audio, dec = audio.cpu().numpy(), dec.cpu().numpy()
    for s in range(S):
        want_dec, want_audio = oracle_stream(po, iqs[s], R)
        assert np.array_equal(dec[s], want_dec), (R, s)
        err = np.abs(audio[s] - want_audio)
        assert err.max() <= AUDIO_TOL, (R, s, int(err.argmax()), len(want_audio))


@pytest.mark.gpu
@pytest.mark.parametrize("R", [171, 256])
def test_fm_exec_two_batches_carry_the_history(pkg, cuda, po, R):
    """At R = 171 and 256 the carried history is 32 R = 5472 / 8192 samples: two batches == one stream."""
    torch = cuda
    S = 3
    n, _ = fm_size(pkg, R, S)
    iqs = fm_streams(2 * n, seed=1000 + R)
    ring = pkg.StreamRing(S, n, R=R)
    audios, decs = [], []
    for b in range(2):
        ring.load(np.ascontiguousarray(iqs[:, b * n:(b + 1) * n]))
        audio, dec = pkg.fm_exec(ring, decimated=True)
        audios.append(audio.cpu().numpy())
        decs.append(dec.cpu().numpy())
        ring.carry()
    torch.cuda.synchronize()
    for s in range(S):
        want_dec, want_audio = oracle_stream(po, iqs[s], R)
        assert np.array_equal(np.concatenate([d[s] for d in decs]), want_dec), s
        assert np.abs(np.concatenate([a[s] for a in audios]) - want_audio).max() <= AUDIO_TOL, s


# ---- b200_fm_channels_exec ---------------------------------------------------------------------------------------

FC_T = 62


def fc_ctas_per_sm(R):
    """Upper bound on resident fm_channels_kernel CTAs per SM: 288 threads each, and the shared memory of launch_fc
    (fm_channels.cu): ring stages of 280 * 2R bytes, two while they fit 120 KB (R <= 109), taps, demod[] and work[]
    of G channels (G = 8 at R = 10, 4 otherwise), barriers."""
    G = 8 if R == 10 else 4
    stage = 280 * 2 * R
    stages = 2 if 2 * stage <= 120 * 1024 else 1
    smem = stages * stage + G * R * 16 + G * (288 + 144) * 4 + 16
    return min(SM_THREADS // 288, SM_SMEM // (smem + 1024))


# offsets on the fs / 64 grid: inc * d == 0 mod 2^32 for every delay d that is a multiple of 64
FC_STEPS = (5, -11, 23)


@pytest.mark.gpu
@pytest.mark.parametrize("R", [10, 7, 109, 110, 256])
def test_fm_channels_walk_tiles(pkg, cuda, synth, R):
    """R = 10: the G = 8 kernel; 7 and 109: the generic kernel with two ring stages; 110 and 256: one stage.
    The first, a middle and the last stream against the float64 oracle; every stream through a bit-exact shift
    property: stream s is stream 0 delayed by d_s samples (silence, bytes of 128, in front), d_s a multiple of
    4R and of 64, so with increments on the fs / 64 grid the integer mixer phases repeat and the baseband and audio
    must be stream 0's, shifted by d_s / R and d_s / (4R) samples."""
    torch = cuda
    S = 5
    workers = sm_count(pkg) * fc_ctas_per_sm(R)
    tps = tiles_per_stream(workers, S)
    n_audio = (tps - 1) * FC_T + short_tile(FC_T)
    n = 4 * R * n_audio
    assert n % 8 == 0 and -(-n_audio // FC_T) == tps and S * tps >= WALK * workers
    D = math.lcm(4 * R, 64)
    delays = [0] + [D * (3 + 17 * (s - 1)) for s in range(1, S)]
    assert delays[-1] < n // 2
    base = synth.s3_fm(n, seed=3 + R, carrier=(FC_STEPS[0] << 26) / 2**32 * FS)       # a station on channel 0
    iq = np.full((S, n, 2), 128, np.uint8)
    for s, d in enumerate(delays):
        iq[s, d:] = base[:n - d]
    incs = np.array([[(k << 26) & 0xFFFFFFFF for k in FC_STEPS]] * S, dtype=np.int64)
    first = 4 * R * 12345
    ring = pkg.StreamRing(S, n, R=R)
    ring.load(iq)
    audio, bb = pkg.fm_channels_exec(ring, incs_tensor(torch, incs), first, baseband=True)
    torch.cuda.synchronize()
    for s, d in enumerate(delays[1:], start=1):
        a, m = d // (4 * R), d // R
        assert torch.equal(audio[s, :, a:], audio[0, :, :n_audio - a]), s
        assert not audio[s, :, :a].any(), s
        assert torch.equal(bb[s, :, m:], bb[0, :, :n // R - m]), s
        assert not bb[s, :, :m].any(), s
    audio, bb = audio.cpu().numpy(), bb.cpu().numpy()
    tol_bb = 4e-6 * 128 * R
    for s in (0, S // 2, S - 1):
        for c in range(len(FC_STEPS)):
            ref = mix_boxcar(iq[s], R, int(incs[s, c]), first)
            err = max(np.abs(bb[s, c, :, 0] - ref.real).max(), np.abs(bb[s, c, :, 1] - ref.imag).max())
            assert err <= tol_bb, (s, c, err)
            assert np.abs(audio[s, c] - demodulate(bb[s, c])).max() <= 1e-4, (s, c)


# ---- outputs written into rows of wider tensors ------------------------------------------------------------------

def nan_rows(torch, shape, width):
    """A view of `shape` whose rows (last dimension) are the first shape[-1] floats of NaN rows `width` long."""
    full = torch.full(tuple(shape[:-1]) + (width,), float("nan"), dtype=torch.float32, device="cuda")
    return full, full[..., :shape[-1]]


@pytest.mark.gpu
@pytest.mark.parametrize("R", [7, 171])
def test_fm_exec_padded_rows(pkg, cuda, po, synth, R):
    """Audio and decimated rows inside wider NaN rows, short last tiles: every padding value stays NaN."""
    torch = cuda
    S = 3
    T = fm_tile_audio(R)
    n_audio = 5 * T + short_tile(T)
    n = 4 * R * n_audio
    iqs = np.stack([synth.s1_noise(n, seed=80 + s) if s % 2 else synth.s3_fm(n, seed=80 + s) for s in range(S)])
    ring = pkg.StreamRing(S, n, R=R)
    ring.load(iqs)
    a_full, audio = nan_rows(torch, (S, n_audio), n_audio + 37)
    d_full = torch.full((S, n // R + 19, 2), float("nan"), dtype=torch.float32, device="cuda")
    pkg.fm_exec(ring, audio=audio, dec=d_full.view(torch.int32)[:, :n // R])
    torch.cuda.synchronize()
    assert torch.isnan(a_full[:, n_audio:]).all() and torch.isnan(d_full[:, n // R:]).all()
    audio, dec = audio.cpu().numpy(), d_full.view(torch.int32)[:, :n // R].cpu().numpy()
    for s in range(S):
        want_dec, want_audio = oracle_stream(po, iqs[s], R)
        assert np.array_equal(dec[s], want_dec)
        assert np.abs(audio[s] - want_audio).max() <= AUDIO_TOL


@pytest.mark.gpu
@pytest.mark.parametrize("R", [10, 7])
def test_fm_channels_padded_rows(pkg, cuda, synth, R):
    """Channel audio rows inside wider NaN rows, a short last tile: the padding stays NaN, the rows hold what a
    call with packed rows returns."""
    torch = cuda
    S, Ch = 2, 3
    n_audio = 5 * FC_T + short_tile(FC_T)
    n = 4 * R * n_audio
    iq = np.stack([synth.s3_fm(n, seed=90 + s, carrier=100e3) for s in range(S)])
    incs = np.array([[pkg.fm_channel_tune(f, FS) for f in (100e3, -300e3, 0.0)]] * S, dtype=np.int64)
    ring = pkg.StreamRing(S, n, R=R)
    ring.load(iq)
    full, audio = nan_rows(torch, (S, Ch, n_audio), n_audio + 29)
    pkg.fm_channels_exec(ring, incs_tensor(torch, incs), 0, audio=audio)
    want, bb = pkg.fm_channels_exec(ring, incs_tensor(torch, incs), 0, baseband=True)
    torch.cuda.synchronize()
    assert torch.isnan(full[..., n_audio:]).all()
    assert torch.equal(audio, want)
    for s in range(S):
        for c in range(Ch):
            assert np.abs(want[s, c].cpu().numpy() - demodulate(bb[s, c].cpu().numpy())).max() <= 1e-4


@pytest.mark.gpu
@pytest.mark.parametrize("flags_name", ["AUDIO_DEEMPH_75US", "AUDIO_RESAMPLE_48K", "both"])
def test_audio_post_padded_rows(pkg, cuda, po, flags_name):
    """Input and output rows inside wider NaN rows, a short last chunk: a read past the input row would put NaN
    into the output, a write past the output row would overwrite the padding."""
    torch = cuda
    flags = pkg.AUDIO_DEEMPH_75US | pkg.AUDIO_RESAMPLE_48K if flags_name == "both" else getattr(pkg, flags_name)
    S, n = 3, 3 * 1024 + 16 * 21
    x = np.random.default_rng(12).uniform(-1, 1, size=(S, n)).astype(np.float32)
    in_full, xin = nan_rows(torch, (S, n), n + 24)
    xin.copy_(torch.as_tensor(x))
    n_out = int(pkg.lib().b200_audio_post_out_samples(n, flags))
    out_full, out = nan_rows(torch, (S, n_out), n_out + 40)
    state = torch.zeros((S, pkg.AUDIO_POST_STATE_FLOATS), dtype=torch.float32, device="cuda")
    pkg.audio_post(xin, state, flags, 51200.0, out=out)
    torch.cuda.synchronize()
    assert torch.isnan(out_full[:, n_out:]).all()
    got = out.cpu().numpy()
    for s in range(S):
        want = x[s]
        if flags & pkg.AUDIO_DEEMPH_75US:
            want, _ = po.deemphasis(want, 51200.0, 75e-6)
        if flags & pkg.AUDIO_RESAMPLE_48K:
            want, _ = po.resample_15_16(want)
        assert np.abs(got[s] - want).max() <= 2e-6


# ---- b200_audio_post at every audio rate fs / (4R) -----------------------------------------------------------------

def deemphasis_f64(x, alpha, y_prev=0.0):
    """y[n] = y[n-1] + alpha (x[n] - y[n-1]) in float64, sequentially from y[-1] = y_prev -> (y, y[-1] for the next
    batch).  alpha is the float32 the library computes (orc_deemphasis_alpha)."""
    a = float(alpha)
    y, _ = lfilter([a], [1.0, a - 1.0], np.asarray(x, np.float64), zi=[(1.0 - a) * y_prev])
    return y, float(y[-1]) if len(y) else y_prev


def test_deemphasis_f64_is_the_definition(po):
    """CPU: the float64 loop above against the oracle's float32 one at the reference's 51.2 kHz, across batches."""
    x = np.random.default_rng(4).uniform(-1, 1, size=20000).astype(np.float32)
    for tau in (50e-6, 75e-6):
        alpha = po.port().orc_deemphasis_alpha(51200.0, tau)
        st, y64 = np.zeros(1, np.float32), 0.0
        for lo, hi in ((0, 7), (7, 12007), (12007, 20000)):
            want, st = po.deemphasis(x[lo:hi], 51200.0, tau, st)
            got, y64 = deemphasis_f64(x[lo:hi], alpha, y64)
            assert np.abs(got - want).max() <= 1e-6


# fs / (4R) at 2.048 MS/s for R = 1, 2, 4, 5, 10, 16, 256, and 3.2 MS/s at R = 1
CHAIN_RATES = [2_048_000.0 / (4 * R) for R in (1, 2, 4, 5, 10, 16, 256)] + [800_000.0]


@pytest.mark.gpu
@pytest.mark.parametrize("resample", [False, True])
@pytest.mark.parametrize("tau", [50e-6, 75e-6])
@pytest.mark.parametrize("rate", CHAIN_RATES)
def test_audio_post_at_chain_rates(pkg, cuda, po, rate, tau, resample):
    """Batches of 2^16 and more samples (64 and more CTAs per stream) and one of 16, state carried across them,
    against the float64 loop within 2e-6.  The resampler's ratio is 15/16 at any rate."""
    torch = cuda
    flags = (pkg.AUDIO_DEEMPH_50US if tau == 50e-6 else pkg.AUDIO_DEEMPH_75US) | (pkg.AUDIO_RESAMPLE_48K if resample else 0)
    alpha = po.port().orc_deemphasis_alpha(rate, tau)
    S = 2
    batches = [65536 + 16 * 37, 16, 2 * 65536 - 16 * 5]
    x = np.random.default_rng(int(rate) + int(tau * 1e6)).uniform(-1, 1, size=(S, sum(batches))).astype(np.float32)
    state = torch.zeros((S, pkg.AUDIO_POST_STATE_FLOATS), dtype=torch.float32, device="cuda")
    y_prev = [0.0] * S
    hist = [np.zeros(15, np.float32) for _ in range(S)]
    pos = 0
    for n in batches:
        got = pkg.audio_post(torch.as_tensor(x[:, pos:pos + n]).cuda(), state, flags, rate).cpu().numpy()
        for s in range(S):
            want, y_prev[s] = deemphasis_f64(x[s, pos:pos + n], alpha, y_prev[s])
            if resample:
                want, hist[s] = po.resample_15_16(want.astype(np.float32), hist[s])
            assert got[s].shape == want.shape
            err = np.abs(got[s] - want)
            assert err.max() <= 2e-6, (s, pos, int(err.argmax()), float(err.max()))
        pos += n


@pytest.mark.gpu
def test_audio_post_refuses_runs_in_over_1024(pkg, cuda):
    """De-emphasis starts each output ceil(ln 1e-7 / ln(1 - alpha)) samples early; above 1024 (about 850 kHz at
    75 us, 1.27 MHz at 50 us) the call is refused before any launch.  The resampler alone takes any rate."""
    torch = cuda
    x = torch.zeros((1, 4096), dtype=torch.float32, device="cuda")
    state = torch.zeros((1, pkg.AUDIO_POST_STATE_FLOATS), dtype=torch.float32, device="cuda")
    torch.cuda.synchronize()
    before = pkg.launch_count()
    for rate, flags in ((900e3, pkg.AUDIO_DEEMPH_75US), (1.3e6, pkg.AUDIO_DEEMPH_50US), (1e30, pkg.AUDIO_DEEMPH_50US),
                        (900e3, pkg.AUDIO_DEEMPH_75US | pkg.AUDIO_RESAMPLE_48K)):
        with pytest.raises(pkg.B200Error):
            pkg.audio_post(x, state, flags, rate)
    assert pkg.launch_count() == before
    for rate, flags in ((900e3, pkg.AUDIO_DEEMPH_50US), (1.2e6, pkg.AUDIO_DEEMPH_50US), (1e9, pkg.AUDIO_RESAMPLE_48K)):
        pkg.audio_post(x, state, flags, rate)
    assert pkg.launch_count() > before


# ---- atan2_approx at the CIC magnitudes of R = 256 ------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("which", [0, 2])
def test_atan2_forms_up_to_r256_magnitudes(pkg, cuda, po, which):
    """Forms 0 (the FM kernels') and 2 (b200_fm_exec_cs32's) on integers in +-32768, the CIC range at R = 256:
    random pairs, both diagonals (the branch at |y| == |x|), one off them on either side, and both axes."""
    rng = np.random.default_rng(256 + which)
    v = np.arange(-32768, 32769, dtype=np.int64)
    w = v[1:-1]                                 # w +- 1 stays inside +-32768
    z = np.zeros_like(v)
    pairs = [("random", rng.integers(-32768, 32769, 100_000), rng.integers(-32768, 32769, 100_000)),
             ("small", rng.integers(-64, 65, 20_000), rng.integers(-32768, 32769, 20_000)),
             ("diag_pp", v, v), ("diag_pm", v, -v), ("diag_y+1", w + 1, w), ("diag_y-1", w - 1, w),
             ("diag_-y+1", -w + 1, w), ("diag_-y-1", -w - 1, w), ("axis_y0", z, v), ("axis_x0", v, z)]
    for name, y, x in pairs:
        got = pkg.debug_atan2(y, x, which)
        want = po.atan2_approx(y.astype(np.float32), x.astype(np.float32))
        err = np.abs(got - want)
        assert err.max() <= 1e-6, (name, int(y[err.argmax()]), int(x[err.argmax()]), float(err.max()))
