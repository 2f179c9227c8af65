"""The general-shape spectrum kernel (spectrum_generic.cu) and the paths that only it serves, against a float64 numpy
reference: u8 frames of 16 to 512 points, every b200_spectrum_exec_cs32 / b200_spectrum_exec_rf32 call (any N, including
the N > 8192 form that works out of the plan's global scratch), plan scratch shared by execs on different CUDA streams,
and the reference-named spectrum_add_* calls at lengths other than 1024.

Tolerances are those of test_gpu_spectrum.py: |dP| <= 1e-4 * P + 1e-4 * mean(P); dB within 0.01 on every bin above
-60 dB of the row mean (for N >= 16384: 0.01 above -40 dB and 0.03 between -60 and -40 dB); payload bytes equal except
where the float64 dB value is within that dB tolerance of an integer, and then off by one at most.  Bytes are compared
on the bins the dB rule covers: at cs32 and rf32 levels a bin 80 dB below its row's mean still has a non-zero byte,
and an f32 transform has no 0.01 dB to give there.

Frame geometries (GEOMETRIES) cover K = 1, K = 3 with Hann frames at 50 % overlap, gaps between rows
(row_hop = 3N + 8) and overlapping rows (row_hop = N/2 + 8).  log2 N is odd for N = 32, 128, 512, 2048, 8192 and 32768:
those sizes run the kernel's radix-2 clean-up pass.
"""
import numpy as np
import pytest

from test_gpu_spectrum import check_db, check_power

# (K, hop, row_hop, hann) as functions of N
GEOMETRIES = {
    "k1": lambda N: (1, N, N, False),
    "k3_hann_half": lambda N: (3, N // 2, 3 * N // 2, True),
    "k2_gaps": lambda N: (2, N, 3 * N + 8, False),
    "k3_hann_overlap": lambda N: (3, N // 2, N // 2 + 8, True),
}


def hann(N):
    return 0.5 - 0.5 * np.cos(2 * np.pi * np.arange(N, dtype=np.float64) / N)


def ref_rows(x, N, hop, K, row_hop, window=None):
    """float64 spectrum rows of one stream x (complex128, already scaled as spectrum.c scales it): row r is
    sum_j fftshift(|fft(x[r*row_hop + j*hop : +N] * w)|^2), j = 0..K-1, with the display position of DC (N/2) replaced by
    the cumulative patch of spectrum.c:30-33, sum_j (K - j) * P_j[N/2 - 1]."""
    x = np.asarray(x, dtype=np.complex128)
    span = (K - 1) * hop + N
    n_rows = 0 if len(x) < span else (len(x) - span) // row_hop + 1
    out = np.zeros((n_rows, N))
    step = max(1, (1 << 21) // (K * N))
    for r0 in range(0, n_rows, step):
        r = np.arange(r0, min(n_rows, r0 + step))
        starts = r[:, None] * row_hop + np.arange(K)[None, :] * hop                   # [rows, K]
        frames = x[starts[:, :, None] + np.arange(N)]                                   # [rows, K, N]
        if window is not None:
            frames = frames * window
        P = np.fft.fftshift(np.abs(np.fft.fft(frames, axis=-1)) ** 2, axes=-1)
        out[r] = P.sum(axis=1)
        out[r, N // 2] = ((K - np.arange(K)) * P[:, :, N // 2 - 1]).sum(axis=1)
    return out


def scale_u8(v):
    v = np.asarray(v, dtype=np.float64)
    return ((v[..., 0] - 128) + 1j * (v[..., 1] - 128)) / 128


def scale_cs32(v):
    v = np.asarray(v, dtype=np.float64)
    return (v[..., 0] + 1j * v[..., 1]) / 128


def scale_rf32(v):
    return np.asarray(v, dtype=np.float64) + 0j


def n_samples(N, K, hop, row_hop, rows):
    return (rows - 1) * row_hop + (K - 1) * hop + N


def cic_like(n, R, seed):
    """cmplx_s32 [n, 2] in the range of a CIC decimator's output at down factor R (sums of R offset bytes,
    -128 R .. 127 R): two tones at 0.45 of full scale each, plus noise."""
    rng = np.random.default_rng(seed)
    t = np.arange(n)
    x = 0.45 * 128 * R * (np.exp(2j * np.pi * 0.123 * t) + np.exp(-2j * np.pi * 0.31 * t))
    x += 2.0 * R * (rng.standard_normal(n) + 1j * rng.standard_normal(n))
    v = np.stack([np.rint(x.real), np.rint(x.imag)], axis=-1)
    return np.clip(v, -128 * R, 127 * R).astype(np.int32)


def audio_like(n, kind, seed):
    """rf32 [n]: unit-variance noise, or two audio-range tones within +-1."""
    if kind == "noise":
        return np.random.default_rng(seed).standard_normal(n).astype(np.float32)
    t = np.arange(n) / 51200.0
    return (0.6 * np.sin(2 * np.pi * 1000.3 * t + seed) + 0.4 * np.cos(2 * np.pi * 7919.0 * t)).astype(np.float32)


def padded(torch, arr, pad):
    """arr [S, n, ...] as a cuda view whose stream rows sit `pad` samples further apart than n (a slice of a wider
    tensor: the stream stride is not n samples)."""
    t = torch.as_tensor(np.ascontiguousarray(arr))
    wide = torch.full((t.shape[0], t.shape[1] + pad) + tuple(t.shape[2:]), 99, dtype=t.dtype, device="cuda")
    wide[:, :t.shape[1]] = t.cuda()
    return wide[:, :t.shape[1]]


def run(plan, kind, x, **kw):
    fn = {"u8": plan.exec, "cs32": plan.exec_cs32, "rf32": plan.exec_rf32}[kind]
    return fn(x, **kw)


def all_outputs(torch, plan, kind, x, n_rows=None):
    out = run(plan, kind, x, n_rows=n_rows, db=True, power=True, db_u8=True)
    torch.cuda.synchronize()
    return {k: v.cpu().numpy() for k, v in out.items()}


def low_tol(N):
    """dB tolerance between -60 and -40 dB of the row mean (0.01 dB holds above -40 dB at every N)."""
    return 0.03 if N >= 16384 else 0.01


def check_bytes(po, got_u8, want, K, gain_db=0, low=0.01):
    """Payload bytes on the bins the dB rule covers: equal, except where the float64 dB value is within the dB
    tolerance of an integer, and then off by one at most."""
    for r in range(want.shape[0]):
        ref, dbf = po.db_payload(want[r], K, gain_db)
        mean = want[r].mean()
        covered = want[r] > 1e-6 * mean
        tol = np.where(want[r] > 1e-4 * mean, 0.01, low)
        diff = (got_u8[r] != ref) & covered
        if diff.any():
            frac = np.abs(dbf - np.rint(dbf))
            assert (frac[diff] <= np.broadcast_to(tol, frac.shape)[diff]).all()
            assert (np.abs(got_u8[r][diff].astype(int) - ref[diff].astype(int)) <= 1).all()
        assert diff.sum() < 0.01 * max(covered.sum(), 1)


def check_rows(po, got, want, K, gain_db=0, low=0.01):
    """got: dict of one stream's [rows, N] outputs; want: float64 reference rows (linear power); low: the dB tolerance
    between -60 and -40 dB of the row mean."""
    check_power(got["power"], want)
    gain = 10.0 ** int(gain_db / 10)                  # cbb_main.c:112, C integer division truncates toward zero
    check_db(got["db"], want, K=K, gain=gain, floor=1e-4)
    check_db(got["db"], want, K=K, gain=gain, floor=1e-6, tol=low)
    check_bytes(po, got["db_u8"], want, K, gain_db, low)


# ---- the reference itself, against the C oracle (no GPU) --------------------------------------------------------

@pytest.mark.parametrize("N", [16, 32, 128, 512, 2048])
def test_reference_matches_c_oracle(po, synth, N):
    for gi, (name, geo) in enumerate(GEOMETRIES.items()):
        K, hop, row_hop, use_hann = geo(N)
        w = hann(N) if use_hann else None
        iq = synth.s2_tones(n_samples(N, K, hop, row_hop, 5), N=N, seed=N + gi)
        want = po.Spectrum(N, window=w).rows(iq, hop=hop, K=K, row_hop=row_hop)
        got = ref_rows(scale_u8(iq), N, hop, K, row_hop, w)
        assert got.shape == want.shape == (5, N), name
        assert (np.abs(got - want) <= 1e-12 * want.mean(axis=1, keepdims=True)).all(), name
    # the other two input types, frame by frame through spectrum_add_cmplx_s32 / spectrum_add_real_f32
    for use_hann in (False, True):
        w = hann(N) if use_hann else None
        K, hop = 3, N // 2
        xs = cic_like(n_samples(N, K, hop, K * hop, 2), 256, seed=N)
        xs[::7] = np.random.default_rng(N).integers(-2 ** 31, 2 ** 31, size=xs[::7].shape, dtype=np.int64)
        xr = audio_like(len(xs), "noise", seed=N)
        for src, add, scale in ((xs, "add_cmplx_s32", scale_cs32), (xr, "add_real_f32", scale_rf32)):
            want = np.zeros((2, N))
            sp = po.Spectrum(N, window=w)
            for r in range(2):
                for j in range(K):
                    start = r * K * hop + j * hop
                    assert getattr(sp, add)(src[start:start + N], want[r]) == 0
            got = ref_rows(scale(src), N, hop, K, K * hop, w)
            assert (np.abs(got - want) <= 1e-12 * want.mean(axis=1, keepdims=True)).all(), (add, use_hann)


# ---- u8 frames on the generic kernel ------------------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("N", [16, 32, 64, 128, 256, 512])
def test_u8_small_frames(pkg, cuda, po, synth, N):
    """Three streams that are slices of a wider tensor, all three outputs, every geometry.  The K = 1 run has
    more (stream, row) items than the kernel's grid (3 CTAs per SM at these sizes), so every CTA walks several items
    and re-zeroes its accumulator between them.  Asking for dB only gives the same bits as asking for everything."""
    torch = cuda
    sm = int(pkg.lib().b200_sm_count())
    for gi, (name, geo) in enumerate(GEOMETRIES.items()):
        K, hop, row_hop, use_hann = geo(N)
        rows = sm + 5 if K == 1 else 9
        n = n_samples(N, K, hop, row_hop, rows)
        iqs = np.stack([synth.s2_tones(n, N=N, seed=10 * N + 3 * gi + s) for s in range(3)])
        x = padded(torch, iqs, 24)
        plan = pkg.SpectrumPlan(N, hop=hop, K=K, row_hop=row_hop, window=pkg.WINDOW_HANN if use_hann else pkg.WINDOW_RECT)
        got = all_outputs(torch, plan, "u8", x)
        assert got["power"].shape == (3, rows, N), name
        if K == 1:
            assert 3 * rows > 3 * sm
        w = hann(N) if use_hann else None
        for s in range(3):
            want = ref_rows(scale_u8(iqs[s]), N, hop, K, row_hop, w)
            check_rows(po, {k: v[s] for k, v in got.items()}, want, K)
        db_only = plan.exec(x, db=True)["db"]
        torch.cuda.synchronize()
        assert np.array_equal(db_only.cpu().numpy(), got["db"], equal_nan=True), name


# ---- cs32 and rf32 at every length --------------------------------------------------------------------------------

ALL_N = [16, 32, 128, 1024, 2048, 8192, 16384, 32768, 65536]
TONE_LOW_TOL = 0.06          # noiseless rf32 tones, between -60 and -40 dB of the row mean (see below)


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["cs32", "rf32"])
@pytest.mark.parametrize("N", ALL_N)
def test_cs32_rf32_every_length(pkg, cuda, po, N, kind):
    """Two strided streams, all three outputs, every geometry.  cs32 stream 0 holds CIC-range values at R = 4, stream
    1 at R = 256 (+-32768); rf32 stream 0 is unit-variance noise, stream 1 two noiseless tones within +-1.  N > 8192
    runs the form that keeps its work arrays in the plan's global scratch.

    The noiseless tones are the one input held to a wider bound, between -60 and -40 dB of the row mean only: with no
    noise floor the rectangular window's leakage skirt reaches bins 50-60 dB below the mean, where the rounding of an
    f32 transform (about 1e-8 of the tone's peak) is no longer small.  That is the limit of f32, not of this kernel:
    scipy.fft in complex64 on the same frames is 0.016 dB off at N = 8192 and 0.025 dB at N = 65536 there.  Measured
    worst case of this kernel on a B200 (1000 W limit), over every geometry: 0.014 dB at N = 8192, 0.020 dB at N = 32768
    and 0.038 dB at N = 65536, all on rectangular K = 1 rows.  Above -40 dB the tones hold 0.01 dB like every other
    input."""
    torch = cuda
    for gi, (name, geo) in enumerate(GEOMETRIES.items()):
        K, hop, row_hop, use_hann = geo(N)
        rows = 2 if N >= 16384 else 5
        n = n_samples(N, K, hop, row_hop, rows)
        plan = pkg.SpectrumPlan(N, hop=hop, K=K, row_hop=row_hop, window=pkg.WINDOW_HANN if use_hann else pkg.WINDOW_RECT)
        if kind == "cs32":
            xs = np.stack([cic_like(n, R, seed=N + gi) for R in (4, 256)])
            out = plan.exec_cs32(padded(torch, xs, 8), db=True, power=True, db_u8=True)
            scale = scale_cs32
        else:
            xs = np.stack([audio_like(n, "noise", seed=N + gi), audio_like(n, "tones", seed=gi)])
            out = plan.exec_rf32(padded(torch, xs, 8), db=True, power=True, db_u8=True)
            scale = scale_rf32
        torch.cuda.synchronize()
        got = {k: v.cpu().numpy() for k, v in out.items()}
        assert got["power"].shape == (2, rows, N), name
        w = hann(N) if use_hann else None
        for s in range(2):
            want = ref_rows(scale(xs[s]), N, hop, K, row_hop, w)
            low = max(low_tol(N), TONE_LOW_TOL) if (kind, s) == ("rf32", 1) else low_tol(N)
            check_rows(po, {k: v[s] for k, v in got.items()}, want, K, low=low)


@pytest.mark.gpu
@pytest.mark.parametrize("N", [32, 2048, 65536])
def test_cs32_full_range_int32(pkg, cuda, po, N):
    """Random int32 over the whole range: the conversion to f32 rounds each sample (2^-24 relative), well inside the
    tolerance; the powers (up to ~2^78) stay far from f32 overflow."""
    torch = cuda
    for name in ("k1", "k3_hann_half"):
        K, hop, row_hop, use_hann = GEOMETRIES[name](N)
        n = n_samples(N, K, hop, row_hop, 3)
        xs = np.random.default_rng(N).integers(-2 ** 31, 2 ** 31, size=(1, n, 2), dtype=np.int64).astype(np.int32)
        plan = pkg.SpectrumPlan(N, hop=hop, K=K, row_hop=row_hop, window=pkg.WINDOW_HANN if use_hann else pkg.WINDOW_RECT)
        got = all_outputs(torch, plan, "cs32", torch.as_tensor(xs).cuda())
        want = ref_rows(scale_cs32(xs[0]), N, hop, K, row_hop, hann(N) if use_hann else None)
        check_rows(po, {k: v[0] for k, v in got.items()}, want, K, low=low_tol(N))


@pytest.mark.gpu
def test_cs32_16384_more_rows_than_scratch(pkg, cuda, po):
    """N = 16384 from cs32 input with more rows than the plan has per-CTA work arrays (2 per SM): CTAs re-use their
    global scratch and accumulator for a second and third row."""
    torch = cuda
    N = 16384
    rows = 2 * int(pkg.lib().b200_sm_count()) + 9
    xs = cic_like(N * rows, 64, seed=5)[None]
    plan = pkg.SpectrumPlan(N)
    got = all_outputs(torch, plan, "cs32", torch.as_tensor(xs).cuda())
    assert got["power"].shape == (1, rows, N)
    want = ref_rows(scale_cs32(xs[0]), N, N, 1, N)
    check_power(got["power"][0], want)
    check_db(got["db"][0], want, floor=1e-4)
    check_db(got["db"][0], want, floor=1e-6, tol=0.03)
    check_bytes(po, got["db_u8"][0][::23], want[::23], 1, 0, low_tol(N))


# ---- edges ------------------------------------------------------------------------------------------------------------

def _input(kind, n, fill=None, seed=0, synth=None, N=1024):
    if kind == "u8":
        return synth.s2_tones(n, N=N, seed=seed) if fill is None else np.full((n, 2), fill, np.uint8)
    if kind == "cs32":
        return cic_like(n, 10, seed) if fill is None else np.full((n, 2), fill, np.int32)
    return audio_like(n, "noise", seed) if fill is None else np.full(n, fill, np.float32)


SCALE = {"u8": scale_u8, "cs32": scale_cs32, "rf32": scale_rf32}


@pytest.mark.gpu
@pytest.mark.parametrize("kind,N", [("u8", 32), ("u8", 512), ("cs32", 128), ("cs32", 32768), ("rf32", 16), ("rf32", 65536)])
def test_all_zero_input(pkg, cuda, kind, N):
    """Zero signal (u8 bytes of 128): power 0, dB -inf, payload byte 0 in every bin, rectangular and Hann."""
    torch = cuda
    for name in ("k1", "k3_hann_overlap"):
        K, hop, row_hop, use_hann = GEOMETRIES[name](N)
        x = _input(kind, n_samples(N, K, hop, row_hop, 3), fill=128 if kind == "u8" else 0)
        plan = pkg.SpectrumPlan(N, hop=hop, K=K, row_hop=row_hop, window=pkg.WINDOW_HANN if use_hann else pkg.WINDOW_RECT)
        got = all_outputs(torch, plan, kind, torch.as_tensor(x[None]).cuda())
        assert got["power"].shape == (1, 3, N)
        assert not got["power"].any() and np.isneginf(got["db"]).all() and not got["db_u8"].any(), (kind, N, name)


@pytest.mark.gpu
@pytest.mark.parametrize("kind,N", [("u8", 128), ("cs32", 16384), ("rf32", 2048)])
def test_gain_saturation_and_negative_decade(pkg, cuda, po, synth, kind, N):
    """gain_db = 300 lifts every bin past 255 dB: the payload byte saturates at 255.  gain_db = -15 is ONE decade down
    (cbb_main.c:112 divides integers: -15 / 10 == -1 in C), not 1.5 and not two."""
    torch = cuda
    K, hop, row_hop, _ = GEOMETRIES["k2_gaps"](N)
    x = _input(kind, n_samples(N, K, hop, row_hop, 3), seed=N, synth=synth, N=N)
    want = ref_rows(SCALE[kind](x), N, hop, K, row_hop)
    for gain_db, gain in ((300, 1e30), (-15, 0.1)):
        plan = pkg.SpectrumPlan(N, hop=hop, K=K, row_hop=row_hop, gain_db=gain_db)
        got = {k: v[0] for k, v in all_outputs(torch, plan, kind, torch.as_tensor(x[None]).cuda()).items()}
        check_power(got["power"], want)
        check_db(got["db"], want, K=K, gain=gain, floor=1e-4 if N >= 16384 else 1e-6)
        check_bytes(po, got["db_u8"], want, K, gain_db, low_tol(N))
        if gain_db == 300:
            loud = 10 * np.log10(gain * want / K) >= 256
            assert loud.mean() > 0.9 and (got["db_u8"][loud] == 255).all()


@pytest.mark.gpu
@pytest.mark.parametrize("kind,N", [("u8", 64), ("cs32", 32768), ("rf32", 8192)])
def test_single_row_and_no_rows(pkg, cuda, po, synth, kind, N):
    """Exactly one row's worth of samples, one sample short of it (no rows), and an explicit n_rows = 0."""
    torch = cuda
    K, hop, row_hop, _ = GEOMETRIES["k3_hann_half"](N)
    plan = pkg.SpectrumPlan(N, hop=hop, K=K, row_hop=row_hop, window=pkg.WINDOW_HANN)
    n = n_samples(N, K, hop, row_hop, 1)
    x = _input(kind, n, seed=3, synth=synth, N=N)
    got = {k: v[0] for k, v in all_outputs(torch, plan, kind, torch.as_tensor(x[None]).cuda()).items()}
    assert got["power"].shape == (1, N)
    check_rows(po, got, ref_rows(SCALE[kind](x), N, hop, K, row_hop, hann(N)), K, low=low_tol(N))
    assert plan.rows(n - 1) == 0
    short = all_outputs(torch, plan, kind, torch.as_tensor(x[None, :n - 1]).cuda())
    assert all(v.shape == (1, 0, N) for v in short.values())
    none = all_outputs(torch, plan, kind, torch.as_tensor(np.stack([x, x])).cuda(), n_rows=0)
    assert all(v.shape == (2, 0, N) for v in none.values())


@pytest.mark.gpu
@pytest.mark.parametrize("kind,N", [("u8", 16), ("u8", 128), ("u8", 512), ("cs32", 1024), ("cs32", 32768), ("cs32", 65536),
                                    ("rf32", 32), ("rf32", 16384)])
def test_tone_on_last_bin_drives_dc_patch(pkg, cuda, po, synth, kind, N):
    """One tone per frame exactly on bin N-1 (display index N/2 - 1; a real cosine on bin 1 has its mirror there): the
    cumulative DC-position patch then carries most of the row's power, so a patch written by the wrong thread, or
    with the wrong weights, fails the power check at display index N/2."""
    torch = cuda
    for K in (1, 3):
        hop = N
        n = n_samples(N, K, hop, K * hop, 2)
        t = np.arange(n)
        if kind == "u8":
            x = synth.tone(n, N - 1, N)
        elif kind == "cs32":
            z = 30000 * np.exp(2j * np.pi * (N - 1) * t / N)
            x = np.stack([np.rint(z.real), np.rint(z.imag)], axis=-1).astype(np.int32)
        else:
            x = np.cos(2 * np.pi * t / N).astype(np.float32)
        plan = pkg.SpectrumPlan(N, hop=hop, K=K)
        got = {k: v[0] for k, v in all_outputs(torch, plan, kind, torch.as_tensor(x[None]).cuda()).items()}
        want = ref_rows(SCALE[kind](x), N, hop, K, K * hop)
        assert (want[:, N // 2] > 0.2 * want.sum(axis=1)).all()
        check_rows(po, got, want, K, low=low_tol(N))
        if K == 1:
            assert np.array_equal(got["power"][:, N // 2], got["power"][:, N // 2 - 1])


# ---- plan scratch shared across CUDA streams ----------------------------------------------------------------------

def _hold_streams(torch, *streams):
    """Make `streams` wait for a few milliseconds of work on the current stream, so that the host has enqueued every
    exec before any of them can start: execs that nothing orders would then run at the same time."""
    a = torch.randn(4096, 4096, device="cuda")
    for _ in range(3):
        torch.mm(a, a)
    ev = torch.cuda.Event()
    ev.record()
    for s in streams:
        s.wait_event(ev)


@pytest.mark.gpu
def test_plan_scratch_shared_across_cuda_streams(pkg, cuda, synth):
    """Execs of one plan on two CUDA streams, enqueued back to back with no host synchronisation, share the plan's
    scratch (the four-step kernel's work arrays for u8 N = 65536 and 16384, the generic kernel's for cs32 N = 16384):
    each result must equal its serial run bit for bit.  Each exec has fewer items than the kernel's grid could hold
    twice over, so two unordered execs would be resident together and write the same scratch slots.  The last case
    alternates u8 and cs32 execs of one N = 16384 plan: one ordering event, one scratch that both kernels use."""
    torch = cuda
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
    u8_65536 = pkg.SpectrumPlan(65536, hop=32768, window=pkg.WINDOW_HANN)
    n = 32768 * 31                                                   # 30 rows per stream, 60 items per exec
    u8_in = [torch.as_tensor(np.stack([synth.s2_tones(n, N=65536, seed=50 + 2 * i + s) for s in range(2)])).cuda()
             for i in range(2)]
    cs32_16384 = pkg.SpectrumPlan(16384)
    cs32_in = [torch.as_tensor(np.stack([cic_like(16384 * 30, 256, seed=60 + 2 * i + s) for s in range(2)])).cuda()
               for i in range(2)]
    u8_16384_in = [torch.as_tensor(np.stack([synth.s2_tones(16384 * 30, N=16384, seed=70 + 2 * i + s) for s in range(2)])).cuda()
                   for i in range(2)]

    def exec_(plan, kind, x, out=None, stream=None):
        return run(plan, kind, x, db=True, power=True, db_u8=True, out=out, stream=stream)

    cases = [[(u8_65536, "u8", u8_in[0]), (u8_65536, "u8", u8_in[1]), (u8_65536, "u8", u8_in[1]), (u8_65536, "u8", u8_in[0])],
             [(cs32_16384, "cs32", cs32_in[0]), (cs32_16384, "cs32", cs32_in[1]), (cs32_16384, "cs32", cs32_in[1]),
              (cs32_16384, "cs32", cs32_in[0])],
             [(cs32_16384, "u8", u8_16384_in[0]), (cs32_16384, "cs32", cs32_in[1]), (cs32_16384, "u8", u8_16384_in[1]),
              (cs32_16384, "cs32", cs32_in[0])]]
    for case in cases:
        serial = [exec_(plan, kind, x) for plan, kind, x in case]
        torch.cuda.synchronize()
        outs = [{k: torch.empty_like(v) for k, v in ref.items()} for ref in serial]
        _hold_streams(torch, s1, s2)
        for i, (plan, kind, x) in enumerate(case):
            exec_(plan, kind, x, out=outs[i], stream=(s1, s2)[i % 2])
        torch.cuda.synchronize()
        for i, (plan, kind, x) in enumerate(case):
            for k in serial[i]:
                assert torch.equal(outs[i][k], serial[i][k]), (plan.N, kind, i, k)


# ---- the reference-named interface at other lengths ---------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("N", [16, 128, 8192, 65536])
def test_compat_spectrum_add_other_lengths(pkg, cuda, po, synth, N):
    """spectrum_add_cmplx_u8 / _cmplx_s32 / _real_f32 accumulate into a dirty caller buffer as spectrum.c does: every
    bin adds its power, the DC position adds its (already updated) left neighbour."""
    rng = np.random.default_rng(N)
    inputs = {"add_cmplx_u8": synth.s2_tones(N, N=N, seed=N),
              "add_cmplx_s32": cic_like(N, 256, seed=N),
              "add_real_f32": audio_like(N, "noise", seed=N)}
    s = pkg.spectrum_alloc(N)
    try:
        for name, x in inputs.items():
            init = rng.uniform(0, 50, N)
            got = init.copy()
            assert getattr(pkg, "spectrum_" + name)(s, x, got, N) == 0
            want = init.copy()
            assert getattr(po.Spectrum(N), name)(x, want) == 0
            np.testing.assert_allclose(got, want, rtol=1e-4, atol=1e-4 * want.mean(), err_msg=name)
            assert got[N // 2] == init[N // 2] + got[N // 2 - 1], name
    finally:
        pkg.spectrum_free(s)
    with pytest.raises(pkg.B200Error):
        pkg.spectrum_alloc(1000)             # powers of two only (spectrum.c plans any N with FFTW)
