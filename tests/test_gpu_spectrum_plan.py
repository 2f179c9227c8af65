"""The spectrum plan's host path: what b200_spectrum_plan_create and the three spectrum execs refuse, and that every
refusal returns before anything is launched; one launch per accepted exec at every N that has its own kernel; and one
plan's scratch shared by the four-step kernel (u8, N >= 16384) and the generic kernel (cs32 / rf32, N > 8192).

Return codes are those of include/b200sdr.h: B200_OK 0, B200_ERR_ARG -1, B200_ERR_ALIGN -4.
"""
import ctypes as C

import numpy as np
import pytest

OK, ERR_ARG, ERR_ALIGN = 0, -1, -4
SPECIALISED_U8_N = [1024, 2048, 4096, 8192, 16384, 65536]      # u8 kernels that read 16-byte words
ROW_LIMIT_N = [1024, 2048, 4096, 8192]                          # u8 kernels that index rows in 32 bits
EVERY_KERNEL_N = [16, 512, 1024, 2048, 4096, 8192, 16384, 65536]


@pytest.fixture
def L(pkg, cuda):
    return pkg.lib()


def exec_fn(L, kind):
    return {"u8": L.b200_spectrum_exec, "cs32": L.b200_spectrum_exec_cs32, "rf32": L.b200_spectrum_exec_rf32}[kind]


def raw_exec(L, kind, plan_h, iq_ptr, stride, n_streams, n_rows, db=None, power=None, db_u8=None):
    """The C exec with raw pointers (None = NULL) on the default stream."""
    vp = lambda t: None if t is None else C.c_void_p(t if isinstance(t, int) else t.data_ptr())
    return exec_fn(L, kind)(plan_h, vp(iq_ptr), stride, n_streams, n_rows, vp(db), vp(power), vp(db_u8), None)


def clear_error(pkg, L):
    """Leave an error text that no spectrum call writes, so that the next check sees the text that call set."""
    assert L.b200_fm_channel_tune(C.c_double(1.0), C.c_double(0.0), None) == ERR_ARG
    assert pkg.binding.last_error().startswith("fm channel tune")


def u8_input(torch, n_streams, n, seed, pad=0):
    """cuda uint8 [n_streams, n + pad, 2] of random bytes."""
    rng = np.random.default_rng(seed)
    return torch.as_tensor(rng.integers(0, 256, size=(n_streams, n + pad, 2), dtype=np.uint8)).cuda()


def kind_input(torch, kind, n, seed):
    rng = np.random.default_rng(seed)
    if kind == "u8":
        return u8_input(torch, 1, n, seed)
    if kind == "cs32":
        return torch.as_tensor(rng.integers(-30000, 30000, size=(1, n, 2), dtype=np.int32)).cuda()
    return torch.as_tensor(rng.standard_normal((1, n)).astype(np.float32)).cuda()


def run(plan, kind, x):
    fn = {"u8": plan.exec, "cs32": plan.exec_cs32, "rf32": plan.exec_rf32}[kind]
    return fn(x, db=True, power=True, db_u8=True)


@pytest.mark.gpu
def test_plan_create_refused(pkg, L):
    cases = [dict(N=8), dict(N=1000), dict(N=131072), dict(K=0), dict(hop=1028), dict(row_hop=1028), dict(window=2)]
    before = pkg.launch_count()
    for kw in cases:
        a = dict(N=1024, hop=1024, K=1, row_hop=0, window=pkg.WINDOW_RECT, gain_db=0)
        a.update(kw)
        clear_error(pkg, L)
        assert not L.b200_spectrum_plan_create(a["N"], a["hop"], a["K"], a["row_hop"], a["window"], a["gain_db"]), kw
        assert pkg.binding.last_error().startswith("spectrum plan"), (kw, pkg.binding.last_error())
    assert pkg.launch_count() == before


@pytest.mark.gpu
@pytest.mark.parametrize("N", SPECIALISED_U8_N)
def test_u8_alignment_refused(pkg, cuda, L, N):
    """A pointer 2 bytes past a 16-byte boundary, or a stream stride 8 bytes off a multiple of 16: B200_ERR_ALIGN with
    no launch, from a real tensor that holds both streams either way."""
    torch = cuda
    plan = pkg.SpectrumPlan(N)
    buf = u8_input(torch, 2, N, seed=N, pad=16)                  # each stream N + 16 samples: 2N + 32 bytes
    db = torch.empty((2, 1, N), dtype=torch.float32, device="cuda")
    base = buf.data_ptr()
    assert base % 16 == 0 and (2 * N) % 16 == 0
    torch.cuda.synchronize()
    before = pkg.launch_count()
    for ptr, stride in ((base + 2, 2 * N + 16), (base, 2 * N + 8)):
        clear_error(pkg, L)
        assert raw_exec(L, "u8", plan.h, ptr, stride, 2, 1, db=db) == ERR_ALIGN, (ptr - base, stride)
        assert pkg.binding.last_error().startswith("spectrum exec"), pkg.binding.last_error()
    assert pkg.launch_count() == before


@pytest.mark.gpu
def test_u8_unaligned_accepted_on_generic_kernel(pkg, cuda, L):
    """At N = 512 (the generic kernel reads 2-byte samples) a pointer 2 bytes past a 16-byte boundary is accepted, and
    gives the bits the same samples give from an aligned tensor."""
    torch = cuda
    N, rows = 512, 7
    buf = u8_input(torch, 1, N * rows, seed=1, pad=8)
    shifted = buf[:, 1:1 + N * rows]
    aligned = shifted.clone()
    assert shifted.data_ptr() % 16 == 2 and aligned.data_ptr() % 16 == 0
    plan = pkg.SpectrumPlan(N)
    outs = []
    for x in (shifted, aligned):
        out = {k: torch.empty((1, rows, N), dtype=dt, device="cuda")
               for k, dt in (("db", torch.float32), ("power", torch.float32), ("db_u8", torch.uint8))}
        before = pkg.launch_count()
        assert raw_exec(L, "u8", plan.h, x.data_ptr(), 0, 1, rows, **out) == OK, pkg.binding.last_error()
        assert pkg.launch_count() == before + 1
        outs.append(out)
    torch.cuda.synchronize()
    for k in outs[0]:
        assert torch.equal(outs[0][k], outs[1][k]), k


@pytest.mark.gpu
@pytest.mark.parametrize("N", ROW_LIMIT_N)
def test_u8_row_limit_refused(pkg, cuda, L, N):
    """n_streams * n_rows >= 2^31 is refused with B200_ERR_ARG before anything is launched, so an aligned fake pointer
    is never read."""
    plan = pkg.SpectrumPlan(N)
    before = pkg.launch_count()
    for n_streams, n_rows in ((2, 1 << 30), (1, 1 << 31), (1 << 20, 1 << 11)):
        clear_error(pkg, L)
        assert raw_exec(L, "u8", plan.h, 1 << 20, 0, n_streams, n_rows, db=1 << 20) == ERR_ARG, (n_streams, n_rows)
        assert "2^31" in pkg.binding.last_error(), pkg.binding.last_error()
    assert pkg.launch_count() == before


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["u8", "cs32", "rf32"])
def test_exec_arguments(pkg, cuda, L, kind):
    """A NULL plan, negative counts and a NULL input with rows to compute are B200_ERR_ARG; no streams or no rows is
    B200_OK with nothing launched, with a NULL input too."""
    torch = cuda
    N = 1024
    plan = pkg.SpectrumPlan(N)
    x = kind_input(torch, kind, N, seed=2)
    db = torch.empty((1, 1, N), dtype=torch.float32, device="cuda")
    torch.cuda.synchronize()
    before = pkg.launch_count()
    for h, ptr, n_streams, n_rows in ((None, x.data_ptr(), 1, 1), (plan.h, x.data_ptr(), -1, 1),
                                      (plan.h, x.data_ptr(), 1, -1), (plan.h, None, 1, 1)):
        clear_error(pkg, L)
        assert raw_exec(L, kind, h, ptr, 0, n_streams, n_rows, db=db) == ERR_ARG, (h, ptr, n_streams, n_rows)
        assert pkg.binding.last_error().startswith("spectrum exec"), pkg.binding.last_error()
    for ptr in (x.data_ptr(), None):
        for n_streams, n_rows in ((0, 1), (1, 0), (0, 0)):
            assert raw_exec(L, kind, plan.h, ptr, 0, n_streams, n_rows, db=db) == OK, (ptr, n_streams, n_rows)
    assert pkg.launch_count() == before


@pytest.mark.gpu
@pytest.mark.parametrize("N", EVERY_KERNEL_N)
def test_one_launch_per_exec(pkg, cuda, N):
    """Every accepted exec adds exactly one launch: u8 on its kernel for N (at N = 1024 also the tiled form, which takes
    dB rows only from 12 rows up), cs32 and rf32 on the generic kernel, shared-memory form up to 8192 and global-scratch
    form above.  The second exec of a plan has its scratch and ordering event already."""
    torch = cuda
    rows = 12 if N <= 8192 else 2
    for kind in ("u8", "cs32", "rf32"):
        plan = pkg.SpectrumPlan(N)
        x = kind_input(torch, kind, N * rows, seed=N)
        for db_only in ((False, True) if (kind, N) == ("u8", 1024) else (False, False)):
            before = pkg.launch_count()
            fn = {"u8": plan.exec, "cs32": plan.exec_cs32, "rf32": plan.exec_rf32}[kind]
            out = fn(x, db=True, power=not db_only, db_u8=not db_only)
            assert pkg.launch_count() == before + 1, (kind, db_only)
            assert out["db"].shape == (1, rows, N)
    torch.cuda.synchronize()


@pytest.mark.gpu
@pytest.mark.parametrize("N,K,hop", [(16384, 1, 16384), (65536, 2, 32768)])
def test_scratch_shared_by_four_step_and_generic(pkg, cuda, N, K, hop):
    """One plan executed u8 -> cs32 -> rf32 -> u8: the generic kernel's first exec grows the scratch the four-step
    kernel got at creation (from none at K = 1, from a smaller one at K = 2), and the four-step kernel then runs out of
    the grown one.  Each result equals, bit for bit, the same exec on a fresh plan."""
    torch = cuda
    window = pkg.WINDOW_HANN if K > 1 else pkg.WINDOW_RECT
    rows = 3
    n = (rows - 1) * K * hop + (K - 1) * hop + N
    inputs = {kind: kind_input(torch, kind, n, seed=N + i) for i, kind in enumerate(("u8", "cs32", "rf32"))}
    shared = pkg.SpectrumPlan(N, hop=hop, K=K, window=window)
    got = [(kind, run(shared, kind, inputs[kind])) for kind in ("u8", "cs32", "rf32", "u8")]
    torch.cuda.synchronize()
    for i, (kind, out) in enumerate(got):
        fresh = pkg.SpectrumPlan(N, hop=hop, K=K, window=window)
        want = run(fresh, kind, inputs[kind])
        torch.cuda.synchronize()
        assert out["power"].shape == (1, rows, N)
        for k in want:
            assert torch.equal(out[k], want[k]), (i, kind, k)
        fresh.close()
