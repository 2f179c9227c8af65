"""GPU parity: the batched spectrum kernels (through the C ABI) against the CPU oracle, the
golden vectors of the unmodified reference, and size-independent properties at full size.

Tolerances (BASELINE.json north_star): bin indexing exact; linear power within 1e-4
relative, stated as |dP| <= 1e-4 * P + 1e-4 * mean(P) (the reference transforms in f64, the
GPU in f32: a bin far below the frame's mean power cannot hold 1e-4 of ITSELF);
log spectra within 0.01 dB on every bin whose power is above 1e-6 (-60 dB) of the frame's mean
(an f32 transform leaves ~5e-7 of the frame's rms amplitude as error in every bin);
payload bytes equal except where the f64 dB value sits within 0.01 of an integer.
"""
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def check_power(got, want):
    got = np.asarray(got, dtype=np.float64)
    mean = want.mean(axis=-1, keepdims=True)
    err = np.abs(got - want)
    bound = 1e-4 * want + 1e-4 * mean
    assert (err <= bound).all(), f"linear power: worst err/bound = {(err / np.maximum(bound, 1e-300)).max():.3g}"


def check_db(got_db, want_power, K=1, gain=1.0, floor=1e-6, tol=0.01):
    want_power = np.asarray(want_power, dtype=np.float64)
    with np.errstate(divide="ignore"):
        want_db = 10 * np.log10(gain * want_power / K)
    mean = want_power.mean(axis=-1, keepdims=True)
    ok = want_power > floor * mean
    assert np.abs(got_db[ok] - want_db[ok]).max() <= tol
    zero = want_power == 0
    assert np.all(np.isneginf(got_db[zero]))


def check_payload(got_u8, want_power, K, gain_db, po):
    for r in range(want_power.shape[0]):
        want, dbf = po.db_payload(want_power[r], K, gain_db)
        diff = got_u8[r] != want
        if diff.any():
            frac = np.abs(dbf[diff] - np.rint(dbf[diff]))
            assert (frac <= 0.01).all() and (np.abs(got_u8[r][diff].astype(int) - want[diff].astype(int)) <= 1).all()
        assert diff.mean() < 0.01


def run_plan(pkg, torch, iq_np, **kw):
    iq = torch.as_tensor(np.ascontiguousarray(iq_np)).cuda()
    if iq.dim() == 2:
        iq = iq[None]
    plan = pkg.SpectrumPlan(**kw)
    out = plan.exec(iq, db=True, power=True, db_u8=True)
    torch.cuda.synchronize()
    return {k: v.cpu().numpy() for k, v in out.items()}


@pytest.mark.parametrize("gen", ["s1", "s2", "s3"])
def test_n1024_per_frame(pkg, cuda, po, synth, gen):
    iq = {"s1": synth.s1_noise, "s2": synth.s2_tones, "s3": synth.s3_fm}[gen](1024 * 37)
    out = run_plan(pkg, cuda, iq, N=1024)
    want = po.Spectrum(1024).rows(iq)
    assert out["power"].shape == (1, 37, 1024)
    check_power(out["power"][0], want)
    check_db(out["db"][0], want)
    check_payload(out["db_u8"][0], want, 1, 0, po)
    # bin indexing: the strongest bin is the same in every frame
    assert np.array_equal(out["power"][0].argmax(axis=1), want.argmax(axis=1))
    # DC-position patch (spectrum.c:30-33): display index 512 repeats index 511 bit for bit
    assert np.array_equal(out["power"][0][:, 512], out["power"][0][:, 511])


@pytest.mark.parametrize("K,gain", [(2, 0), (6, 0), (6, 17), (6, 30), (5, -10)])
def test_n1024_accumulated_rows_and_gain(pkg, cuda, po, synth, K, gain):
    iq = synth.s2_tones(1024 * (4 * K + 1), seed=K)
    out = run_plan(pkg, cuda, iq, N=1024, K=K, gain_db=gain)
    want = po.Spectrum(1024).rows(iq, K=K)
    assert out["power"].shape[1] == 4
    check_power(out["power"][0], want)
    # cumulative DC patch: sum_j (K - j) * P_j[N-1]
    frames = po.Spectrum(1024).rows(iq)
    for r in range(4):
        w = sum((K - j) * frames[r * K + j, 511] for j in range(K))
        assert abs(out["power"][0][r, 512] / w - 1) < 1e-4
    check_db(out["db"][0], want, K=K, gain=10.0 ** (int(gain / 10)))     # C integer division truncates
    check_payload(out["db_u8"][0], want, K, gain, po)


def test_n1024_reference_cadence_and_goldens(pkg, cuda, po, synth):
    # the cadence the reference's driver produces: 6 frames every 4th 131072-sample buffer
    g = np.load(os.path.join(GOLD, "cbb_gain17.npz"))
    iq = synth.s2_tones(int(g["n"]), N=1024, seed=int(g["seed"]))
    out = run_plan(pkg, cuda, iq, N=1024, K=6, row_hop=4 * 131072, gain_db=17)
    assert out["power"].shape[1] == len(g["power"])
    check_power(out["power"][0], g["power"])
    check_payload(out["db_u8"][0], g["power"], 6, 17, po)
    exact = (out["db_u8"][0] == g["payload"]).mean()
    assert exact > 0.995
    g = np.load(os.path.join(GOLD, "spectrum_n1024.npz"))
    out = run_plan(pkg, cuda, g["iq"], N=1024, K=6)
    check_power(out["power"][0], g["rows_k6"])
    g = np.load(os.path.join(GOLD, "spectrum_kat.npz"))
    out = run_plan(pkg, cuda, g["iq_dc"], N=1024)
    assert not out["power"].any() and np.isneginf(out["db"]).all() and not out["db_u8"].any()
    out = run_plan(pkg, cuda, g["iq_tone"], N=1024, K=2)
    check_power(out["power"][0], g["rows_tone_k2"])
    assert out["power"][0, 0].argmax() == 612


def test_n1024_overlap_window_and_streams(pkg, cuda, po, synth):
    # 50% overlap + Hann (extension; the reference is rectangular, hop = N), 5 independent streams
    n = 1024 * 9
    iqs = np.stack([synth.s2_tones(n, seed=40 + s) for s in range(5)])
    out = run_plan(pkg, cuda, iqs, N=1024, hop=512, window=pkg.WINDOW_HANN)
    assert out["power"].shape == (5, 17, 1024)
    for s in range(5):
        want = po.Spectrum(1024, window=synth.hann(1024)).rows(iqs[s], hop=512)
        check_power(out["power"][s], want)
        check_db(out["db"][s], want)
    out = run_plan(pkg, cuda, iqs, N=1024, K=3, hop=512, window=pkg.WINDOW_HANN)
    for s in range(5):
        want = po.Spectrum(1024, window=synth.hann(1024)).rows(iqs[s], hop=512, K=3)
        check_power(out["power"][s], want)


def test_strided_stream_rows_and_empty(pkg, cuda, po, synth):
    torch = cuda
    ring = pkg.StreamRing(3, 1024 * 8)
    iqs = np.stack([synth.s1_noise(1024 * 8, seed=s) for s in range(3)])
    ring.load(iqs)
    plan = pkg.SpectrumPlan(1024)
    out = plan.exec(ring.batch, power=True)
    torch.cuda.synchronize()
    for s in range(3):
        check_power(out["power"][s].cpu().numpy(), po.Spectrum(1024).rows(iqs[s]))
    empty = plan.exec(ring.batch[:, :512], power=True)
    assert empty["power"].shape == (3, 0, 1024)
    with pytest.raises(pkg.B200Error):
        pkg.SpectrumPlan(1000)
    with pytest.raises(pkg.B200Error):
        pkg.SpectrumPlan(1024, hop=100)


@pytest.mark.parametrize("N,K", [(16, 1), (256, 2), (2048, 1), (4096, 1), (4096, 3), (8192, 1), (16384, 1), (16384, 3), (32768, 1),
                                 (32768, 2), (65536, 1)])
def test_other_frame_lengths(pkg, cuda, po, synth, N, K):
    iq = synth.s2_tones(N * K * 2 + 8, N=N, seed=N % 97)
    out = run_plan(pkg, cuda, iq, N=N, K=K)
    want = po.Spectrum(N).rows(iq, K=K)
    check_power(out["power"][0], want)
    check_db(out["db"][0], want, K=K)
    assert np.array_equal(out["power"][0].argmax(axis=1), want.argmax(axis=1))


@pytest.mark.parametrize("N,rows", [(2048, 1300), (4096, 1300), (8192, 330)])
def test_persistent_loop_many_rows(pkg, cuda, po, synth, N, rows):
    """More rows than resident CTAs: every CTA walks several frames (TMA ring wrap-around, mbarrier phase
    flips), K = 1 and K = 2, rectangular and Hann at 50 % overlap; u8 payload bytes included."""
    torch = cuda
    iq = synth.s2_tones(N * rows, N=N, seed=N % 89)
    out = run_plan(pkg, cuda, iq, N=N)
    want = po.Spectrum(N).rows(iq)
    assert out["power"].shape == (1, rows, N)
    check_power(out["power"][0], want)
    check_db(out["db"][0], want)
    check_payload(out["db_u8"][0][::97], want[::97], 1, 0, po)
    out = run_plan(pkg, cuda, iq[:N * 200], N=N, K=2, hop=N // 2, window=pkg.WINDOW_HANN)
    want = po.Spectrum(N, window=synth.hann(N)).rows(iq[:N * 200], hop=N // 2, K=2)
    check_power(out["power"][0], want)
    check_db(out["db"][0], want, K=2)


@pytest.mark.parametrize("N,rows", [(16384, 400), (32768, 210)])
def test_four_step_kernel_16384_32768(pkg, cuda, po, synth, N, rows):
    """N = 16384 and 32768 run the 65536-point kernel's four-step form with 16 / 32 polyphase branches: more rows than
    CTAs (each CTA walks a run of frames), rectangular with hop = N, Hann at 50 % overlap (half-frame re-use and the
    row swizzle of the narrower rows), K = 2 accumulation, two streams, u8 payload bytes.  dB tolerance as for the
    65536-point frames (BASELINE.md section 4): millions of bins through 14-15 f32 stages hold 0.01 dB above -40 dB of
    the frame mean and 0.03 dB between -60 and -40 dB."""
    def check_db_long(got, want, K=1):
        check_db(got, want, K=K, floor=1e-4)
        check_db(got, want, K=K, floor=1e-6, tol=0.03)

    iq = np.stack([synth.s2_tones(N * rows // 2, N=N, seed=N % 83 + s) for s in range(2)])
    out = run_plan(pkg, cuda, iq, N=N)
    for s in range(2):
        want = po.Spectrum(N).rows(iq[s])
        assert out["power"].shape == (2, rows // 2, N)
        check_power(out["power"][s], want)
        check_db_long(out["db"][s], want)
        check_payload(out["db_u8"][s][::37], want[::37], 1, 0, po)
    out = run_plan(pkg, cuda, iq, N=N, hop=N // 2, window=pkg.WINDOW_HANN)
    for s in range(2):
        want = po.Spectrum(N, window=synth.hann(N)).rows(iq[s], hop=N // 2)
        check_power(out["power"][s], want)
        check_db_long(out["db"][s], want)
    out = run_plan(pkg, cuda, iq[0], N=N, K=2, hop=N // 2, window=pkg.WINDOW_HANN)
    want = po.Spectrum(N, window=synth.hann(N)).rows(iq[0], hop=N // 2, K=2)
    check_power(out["power"][0], want)
    check_db_long(out["db"][0], want, K=2)


def test_goldens_n4096_n65536(pkg, cuda, synth):
    g = np.load(os.path.join(GOLD, "spectrum_n4096.npz"))
    out = run_plan(pkg, cuda, g["iq"], N=4096, K=3)
    check_power(out["power"][0], g["rows_k3"])
    g = np.load(os.path.join(GOLD, "spectrum_n65536.npz"))
    iq = synth.s2_tones(65536, N=65536, seed=int(g["seed"]))
    out = run_plan(pkg, cuda, iq, N=65536)
    check_power(out["power"][0], g["rows_k1"])


def test_wideband_spectrogram_65536_hann_overlap(pkg, cuda, po, synth):
    """BASELINE config 4: 65536-point Hann frames at 50 % overlap, two streams; plus K = 2 rows."""
    iqs = np.stack([synth.s2_tones(65536 * 3, N=65536, seed=5 + s) for s in range(2)])
    out = run_plan(pkg, cuda, iqs, N=65536, hop=32768, window=pkg.WINDOW_HANN)
    assert out["power"].shape == (2, 5, 65536)
    for s in range(2):
        want = po.Spectrum(65536, window=synth.hann(65536)).rows(iqs[s], hop=32768)
        check_power(out["power"][s], want)
        check_db(out["db"][s], want)
        assert np.array_equal(out["power"][s].argmax(axis=1), want.argmax(axis=1))
    out = run_plan(pkg, cuda, iqs, N=65536, hop=32768, K=2, window=pkg.WINDOW_HANN)
    for s in range(2):
        want = po.Spectrum(65536, window=synth.hann(65536)).rows(iqs[s], hop=32768, K=2)
        check_power(out["power"][s], want)
    out = run_plan(pkg, cuda, iqs[0], N=65536, K=3)
    check_power(out["power"][0], po.Spectrum(65536).rows(iqs[0], K=3))


def test_spectrogram_65536_long_capture(pkg, cuda, po, synth):
    """One long capture, more rows than CTAs: every CTA walks a contiguous run of overlapping frames and
    re-uses the resident half of the previous one (rows alternate between the two halves of its buffer);
    the rectangular hop = N case next to it fetches whole frames."""
    n_rows = 450
    iq = synth.s2_tones(32768 * (n_rows + 1), N=65536, seed=11)
    out = run_plan(pkg, cuda, iq, N=65536, hop=32768, window=pkg.WINDOW_HANN)
    assert out["power"].shape == (1, n_rows, 65536)
    want = po.Spectrum(65536, window=synth.hann(65536)).rows(iq, hop=32768)
    check_power(out["power"][0], want)
    # 29 M bins through 16 f32 butterfly stages: the worst bin between -60 and -40 dB of its frame's mean is
    # 0.02 dB off (rectangular and Hann alike); above -40 dB everything is within 0.01 dB
    check_db(out["db"][0], want, floor=1e-4)
    check_db(out["db"][0], want, floor=1e-6, tol=0.03)
    out = run_plan(pkg, cuda, iq, N=65536)
    check_power(out["power"][0], po.Spectrum(65536).rows(iq))


def test_cs32_and_rf32_inputs(pkg, cuda, po):
    torch = cuda
    rng = np.random.default_rng(2)
    x = rng.integers(-1280, 1271, size=(2, 2048, 2), dtype=np.int32)
    plan = pkg.SpectrumPlan(1024)
    got = plan.exec_cs32(torch.as_tensor(x).cuda())["power"].cpu().numpy()
    for s in range(2):
        want = np.zeros((2, 1024))
        sp = po.Spectrum(1024)
        for r in range(2):
            sp.add_cmplx_s32(x[s, 1024 * r:1024 * (r + 1)], want[r])
        check_power(got[s], want)
    xr = rng.standard_normal((2, 2048)).astype(np.float32)
    got = plan.exec_rf32(torch.as_tensor(xr).cuda())["power"].cpu().numpy()
    for s in range(2):
        want = np.zeros((2, 1024))
        sp = po.Spectrum(1024)
        for r in range(2):
            sp.add_real_f32(xr[s, 1024 * r:1024 * (r + 1)], want[r])
        check_power(got[s], want)


@pytest.mark.parametrize("N,n_frames", [(1024, 1 << 20), (4096, 1 << 20), (16384, 1 << 14), (32768, 1 << 13), (65536, 1 << 12)])
def test_full_size_parseval_checksum(pkg, cuda, N, n_frames):
    """BASELINE config 2 at its full size (2^20 frames of 1024 and of 4096 points), and 2^28 samples through each of the
    four-step sizes, through a size-independent property: sum over bins of |X|^2 = N * sum |x|^2 (Parseval).  With the DC
    position replaced by bin N-1's value, sum_i P[i] = N * sum|x|^2 - |sum x|^2 + P[N/2 - 1], all
    exact integers on the input side."""
    torch = cuda
    g = torch.Generator(device="cuda").manual_seed(0)
    iq = torch.randint(0, 256, (1, n_frames * N, 2), dtype=torch.uint8, device="cuda", generator=g)
    plan = pkg.SpectrumPlan(N)
    power = plan.exec(iq, db=False, power=True)["power"][0]           # [n_frames, N] f32 (4 / 16 GiB)
    energy = torch.empty(n_frames, dtype=torch.int64, device="cuda")
    dc_pow = torch.empty(n_frames, dtype=torch.int64, device="cuda")
    step = (1 << 25) // N
    for f0 in range(0, n_frames, step):                                # exact integer side, in chunks
        x = iq[0, f0 * N:(f0 + step) * N].view(step, N, 2).to(torch.int32) - 128
        energy[f0:f0 + step] = (x * x).sum(dim=(1, 2), dtype=torch.int64)   # sum |x|^2 * 128^2
        dc = x.sum(dim=1, dtype=torch.int64)
        dc_pow[f0:f0 + step] = (dc * dc).sum(dim=1)
        del x, dc
    want = (N * energy - dc_pow).to(torch.float64) / 16384.0
    got = torch.empty(n_frames, dtype=torch.float64, device="cuda")
    for f0 in range(0, n_frames, step):
        got[f0:f0 + step] = power[f0:f0 + step].to(torch.float64).sum(dim=1)
    got -= power[:, N // 2].to(torch.float64)
    rel = ((got - want).abs() / want).max().item()
    assert rel < 2e-6, rel
    assert torch.equal(power[:, N // 2], power[:, N // 2 - 1])
    # a checksum of checksums over all frames, in float64: what is left is the systematic part of the f32
    # rounding (twiddles whose |w|^2 is 1 +- 6e-8), which grows with the number of stages
    assert abs(got.sum().item() / want.sum().item() - 1) < (1e-7 if N == 1024 else 2e-7 if N == 4096 else 4e-7)


@pytest.mark.parametrize("hop,window", [(1024, 0), (512, 1), (256, 1), (1016, 0)])
def test_n1024_db_only_tiled_path(pkg, cuda, po, synth, hop, window):
    """dB rows only, K = 1, frames hop <= N apart: the tiled kernel (five frames per TMA copy).  Row counts
    that are not a multiple of five, several streams, overlap with and without the Hann window."""
    torch = cuda
    n_streams, n_rows = 3, 53
    n = hop * (n_rows - 1) + 1024
    iqs = np.stack([synth.s2_tones(n, seed=400 + s) for s in range(n_streams)])
    d = torch.as_tensor(iqs).cuda()
    plan = pkg.SpectrumPlan(1024, hop=hop, window=window)
    db = plan.exec(d, db=True)["db"]
    torch.cuda.synchronize()
    assert db.shape == (n_streams, n_rows, 1024)
    db = db.cpu().numpy()
    for s in range(n_streams):
        want = po.Spectrum(1024, window=synth.hann(1024) if window else None).rows(iqs[s], hop=hop)
        check_db(db[s], want)


def test_db_only_matches_all_outputs(pkg, cuda, po, synth):
    """Requesting only the dB output must give the same bits as requesting everything, for odd
    row counts and several streams (the outputs are written by separate store loops)."""
    torch = cuda
    for n_streams, n_frames in ((1, 1), (1, 7), (3, 5), (4, 16), (5, 333)):
        ring = pkg.StreamRing(n_streams, 1024 * n_frames + 8)
        iqs = np.stack([synth.s2_tones(1024 * n_frames + 8, seed=200 + s) for s in range(n_streams)])
        ring.load(iqs)
        plan = pkg.SpectrumPlan(1024)
        fast = plan.exec(ring.batch, db=True)["db"]
        both = plan.exec(ring.batch, db=True, power=True)
        torch.cuda.synchronize()
        assert fast.shape == (n_streams, n_frames, 1024)
        assert torch.equal(fast, both["db"])
        for s in range(min(n_streams, 2)):
            check_db(fast[s].cpu().numpy(), po.Spectrum(1024).rows(iqs[s]))


def test_spectrogram_full_size_shift_property(pkg, cuda):
    """BASELINE config 4 scale (a 2^27-sample capture, 65536-point Hann frames at 50 % overlap)
    through a size-independent property: delaying the capture by one hop shifts the spectrogram
    by exactly one row, bit for bit (frames are computed independently from the same bytes)."""
    torch = cuda
    n = 1 << 27
    hop = 32768
    g = torch.Generator(device="cuda").manual_seed(11)
    iq = torch.randint(0, 256, (2, n, 2), dtype=torch.uint8, device="cuda", generator=g)
    iq[1, hop:] = iq[0, :n - hop]
    plan = pkg.SpectrumPlan(65536, hop=hop, window=pkg.WINDOW_HANN)
    db = plan.exec(iq, db=True)["db"]
    torch.cuda.synchronize()
    rows = plan.rows(n)
    assert db.shape == (2, rows, 65536) and rows == (n - 65536) // hop + 1
    assert torch.equal(db[1, 1:], db[0, :rows - 1])
    assert torch.isfinite(db[0]).all()
    # white bytes: every row's mean power sits at the analytic level
    #   E|X|^2 = sum(w^2) * E|x|^2,  E|x|^2 = 2 * (256^2 - 1) / 12 / 128^2
    lin = torch.pow(10.0, db[0, ::64].double() / 10).mean().item()
    want = 0.375 * 65536 * 2 * (256 ** 2 - 1) / 12 / 128 ** 2
    assert abs(lin / want - 1) < 0.01
