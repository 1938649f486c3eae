"""GPU parity tests (run with -m gpu on a B200): the CUDA path, called through the C ABI, against the CPU
oracle, the committed golden fixtures (reference numba outputs) and the stored outputs of the reference's own CUDA
kernels (src/core/kernels.cu compiled unmodified, tests/golden/ref_cuda_kernels.npz).

Tolerance (north_star): <= 1e-12 relative FP64, measured as max|du|/max|u| and ||du||_2/||u||_2."""
import os

import numpy as np
import pytest

import oracle as orc
import skellysim_b200 as skb
from conftest import GOLDEN_DIR, rel_l2, rel_max

pytestmark = pytest.mark.gpu
TOL = 1e-12
SL, DL = skb.KERNEL_STOKESLET, skb.KERNEL_STRESSLET


def _rand(seed, ns, nt, coincident=0, scale=1.0):
    rng = np.random.default_rng(seed)
    rs = rng.uniform(-1, 1, (ns, 3)) * scale
    rt = rng.uniform(-1, 1, (nt, 3)) * scale
    if coincident:
        rt[:coincident] = rs[:coincident]
    return rs, rt, rng.uniform(-1, 1, (ns, 3)), rng.uniform(-1, 1, (ns, 9))


@pytest.fixture(scope="module")
def ctx():
    c = skb.Context(1)
    yield c
    c.close()


def _check(u, ref, tol=TOL):
    assert np.isfinite(u).all()
    assert rel_max(u, ref) < tol, rel_max(u, ref)
    assert rel_l2(u, ref) < tol, rel_l2(u, ref)


def test_kernel_test_shape_stateless_entry_points():
    # tests/core/kernel_test.cpp:25-37: n_src=1229, n_trg=743, eta=1.3, U[-1,1]; reference gate 5e-9 on ||.||_2
    rs, rt, f3, f9 = _rand(1, 1229, 743)
    eta = 1.3
    u = skb.stokeslet_direct(rs, f3, rt) / eta
    ref = orc.stokeslet_direct(rs, f3, rt) / eta
    _check(u, ref)
    assert np.linalg.norm(u - ref) < 5e-9
    d = skb.stresslet_direct(rs, f9, rt) / eta
    refd = orc.stresslet_direct(rs, f9, rt) / eta
    _check(d, refd)
    assert np.linalg.norm(d - refd) < 5e-9


@pytest.mark.parametrize("case", ["kernel_test", "ragged", "single", "fibers16x32", "wide_range"])
def test_golden_reference_outputs(golden_cases, case):
    g = golden_cases[case]
    eta = float(g["eta"])
    u = skb.stokeslet_direct(g["r_src"], g["f_sl"], g["r_trg"]) / eta
    _check(u, g["u_stokeslet"])
    f_dl = orc.form_double_layer(g["normals"], g["density"], eta)
    d = skb.stresslet_direct(g["r_src"], f_dl, g["r_trg"]) / eta
    _check(d, g["u_stresslet"])


def test_against_reference_cuda_kernels():
    # the UNMODIFIED reference kernels.cu, run on a B200 (stored by tests/golden/make_golden.py --cuda), vs the oracle
    # and vs the new path
    g = np.load(os.path.join(GOLDEN_DIR, "ref_cuda_kernels.npz"))
    rs, rt, f3, f9 = g["r_src"], g["r_trg"], g["f_sl"], g["f_dl"]
    ref_u, ref_d = g["u_stokeslet"], g["u_stresslet"]
    # oracle pinned by the reference itself
    _check(orc.stokeslet_direct(rs, f3, rt), ref_u)
    _check(orc.stresslet_direct(rs, f9, rt), ref_d)
    # new path vs reference
    _check(skb.stokeslet_direct(rs, f3, rt), ref_u)
    _check(skb.stresslet_direct(rs, f9, rt), ref_d)


@pytest.mark.parametrize("ns,nt", [(1, 1), (1, 1000), (2, 3), (127, 129), (128, 128), (129, 511), (1000, 1),
                                   (257, 2049), (4097, 777)])
def test_ragged_sizes(ctx, ns, nt):
    rs, rt, f3, f9 = _rand(100 + ns + nt, ns, nt)
    ctx.set_targets(rt)
    ctx.set_sources(SL, rs)
    ctx.set_sources(DL, rs)
    _check(ctx.eval(SL, f3), orc.stokeslet_direct(rs, f3, rt))
    _check(ctx.eval(DL, f9), orc.stresslet_direct(rs, f9, rt))


def test_empty_inputs(ctx):
    rs, rt, f3, f9 = _rand(5, 10, 7)
    e3, e9 = np.zeros((0, 3)), np.zeros((0, 9))
    ctx.set_targets(rt)
    ctx.set_sources(SL, e3)
    ctx.set_sources(DL, e3)
    assert np.array_equal(ctx.eval(SL, e3), np.zeros((7, 3)))
    assert np.array_equal(ctx.eval(DL, e9), np.zeros((7, 3)))
    ctx.set_targets(e3)
    ctx.set_sources(SL, rs)
    assert ctx.eval(SL, f3).shape == (0, 3)
    assert skb.stokeslet_direct(e3, e3, rt).shape == (7, 3)


def test_coincident_points_targets_equal_sources(ctx):
    # apply_matvec: the first N_f targets ARE the fiber sources (system.cpp:287-299); r == 0 pairs give exactly 0
    rs, _, f3, f9 = _rand(9, 2000, 1)
    ctx.set_targets(rs)
    ctx.set_sources(SL, rs)
    ctx.set_sources(DL, rs)
    u = ctx.eval(SL, f3)
    d = ctx.eval(DL, f9)
    _check(u, orc.stokeslet_direct(rs, f3, rs))
    _check(d, orc.stresslet_direct(rs, f9, rs))


def test_duplicate_sources_and_zero_strength(ctx):
    rng = np.random.default_rng(2)
    rs = np.repeat(rng.uniform(-1, 1, (50, 3)), 4, axis=0)  # every source position 4x
    f3 = rng.uniform(-1, 1, (200, 3))
    f3[::3] = 0.0
    rt = np.concatenate([rs[::7], rng.uniform(-1, 1, (33, 3))])
    ctx.set_targets(rt)
    ctx.set_sources(SL, rs)
    _check(ctx.eval(SL, f3), orc.stokeslet_direct(rs, f3, rt))


@pytest.mark.parametrize("T", [1, 2, 4, 8])
@pytest.mark.parametrize("S", [1, 3, 16])
def test_all_kernel_variants(T, S):
    rs, rt, f3, f9 = _rand(40 + T + S, 3001, 2500, coincident=100)
    with skb.Context(1) as c:
        c.set_tuning(T, S)
        c.set_targets(rt)
        c.set_sources(SL, rs)
        c.set_sources(DL, rs)
        u = c.eval(SL, f3)
        st = c.stats()
        assert st["targets_per_thread"] == T
        d = c.eval(DL, f9)
    _check(u, orc.stokeslet_direct(rs, f3, rt))
    _check(d, orc.stresslet_direct(rs, f9, rt))


def test_position_caching_and_repeated_evals(ctx):
    # GMRES: positions fixed, strengths change every iteration (system.cpp:486-489)
    rs, rt, f3, _ = _rand(77, 1500, 900)
    ctx.set_targets(rt)
    ctx.set_sources(SL, rs)
    rng = np.random.default_rng(0)
    for _ in range(3):
        f = rng.normal(size=f3.shape)
        _check(ctx.eval(SL, f), orc.stokeslet_direct(rs, f, rt))
    # bitwise run-to-run reproducibility (fixed-order split reduction, no atomics)
    a = ctx.eval(SL, f3)
    b = ctx.eval(SL, f3)
    assert np.array_equal(a, b)


def test_accumulate_and_fused(ctx):
    rs, rt, f3, f9 = _rand(31, 700, 450)
    rs2 = rs[:300] + 0.01
    ctx.set_targets(rt)
    ctx.set_sources(SL, rs)
    ctx.set_sources(DL, rs2)
    ref = orc.stokeslet_direct(rs, f3, rt) + orc.stresslet_direct(rs2, f9[:300], rt)
    out = ctx.eval(SL, f3)
    ctx.eval(DL, f9[:300], out=out, accumulate=True)
    _check(out, ref)
    _check(ctx.eval_fused(f3, f9[:300]), ref)
    _check(ctx.eval_fused(f3, None), orc.stokeslet_direct(rs, f3, rt))


def test_double_layer_formed_on_device(ctx):
    # Periphery::flow: f_dl = 2 eta n (x) rho (periphery.cpp:68-71) then stresslet / eta
    rng = np.random.default_rng(8)
    pos, nrm, dens = rng.uniform(-2, 2, (1300, 3)), rng.normal(size=(1300, 3)), rng.normal(size=(1300, 3))
    rt = rng.uniform(-1, 1, (999, 3))
    eta = 0.7
    ctx.set_targets(rt)
    ctx.set_sources(DL, pos)
    ctx.set_source_normals(nrm)
    u = ctx.eval_double_layer(dens, eta) / eta
    _check(u, orc.periphery_flow(rt, pos, nrm, dens, eta))
    # identical (bitwise) to shipping the host-formed 9-component strength
    u9 = ctx.eval(DL, orc.form_double_layer(nrm, dens, eta)) / eta
    assert np.array_equal(u, u9)


def test_analytic_identities_on_gpu():
    f = np.array([[0.0, 0.0, 2.0]])
    src = np.zeros((1, 3))
    r = 1.7
    u = skb.stokeslet_direct(src, f, np.array([[0, 0, r], [r, 0, 0]]))
    assert abs(u[0, 2] - 2.0 / (4 * np.pi * r)) < 1e-15
    assert abs(u[1, 2] - 2.0 / (8 * np.pi * r)) < 1e-15


def test_scale_extremes(ctx):
    # coordinates ~1e-6 and ~1e+6: the rsqrt seed/Newton path must hold relative accuracy across exponents
    for scale in (1e-6, 1e6):
        rs, rt, f3, f9 = _rand(3, 500, 300, scale=scale)
        ctx.set_targets(rt)
        ctx.set_sources(SL, rs)
        ctx.set_sources(DL, rs)
        _check(ctx.eval(SL, f3), orc.stokeslet_direct(rs, f3, rt))
        _check(ctx.eval(DL, f9), orc.stresslet_direct(rs, f9, rt))


def test_true_error_vs_long_double(ctx):
    # both the FP64 oracle and the CUDA path against 80-bit arithmetic: the CUDA path is not worse than 10x oracle
    rs, rt, f3, f9 = _rand(13, 4000, 512)
    ld = orc.stokeslet_direct_ld(rs, f3, rt)
    ctx.set_targets(rt)
    ctx.set_sources(SL, rs)
    e_gpu = rel_max(ctx.eval(SL, f3), ld)
    e_cpu = rel_max(orc.stokeslet_direct(rs, f3, rt), ld)
    assert e_gpu < 1e-13 and e_gpu < 10 * e_cpu + 1e-15


def test_full_size_properties_c2():
    # BASELINE C2-sized call (SL 32 000 -> 40 000) checked through size-independent properties + a subset oracle
    rng = np.random.default_rng(1)
    ns, nt = 32000, 40000
    rs = rng.uniform(-4, 4, (ns, 3))
    rt = np.concatenate([rs, rng.uniform(-4, 4, (nt - ns, 3))])
    f1, f2 = rng.uniform(-1, 1, (ns, 3)), rng.uniform(-1, 1, (ns, 3))
    with skb.Context(1) as c:
        c.set_targets(rt)
        c.set_sources(SL, rs)
        u1, u2 = c.eval(SL, f1), c.eval(SL, f2)
        u12 = c.eval(SL, 2.0 * f1 - 0.5 * f2)
        # linearity in the strengths
        assert rel_max(u12, 2.0 * u1 - 0.5 * u2) < 1e-12
        # permutation invariance of the sources (summation order changes, value must not beyond rounding)
        perm = rng.permutation(ns)
        c.set_sources(SL, rs[perm])
        assert rel_max(c.eval(SL, f1[perm]), u1) < 1e-12
        st = c.stats()
        assert st["n_pairs"] == ns * nt
    sub = rng.choice(nt, 256, replace=False)
    _check(u1[sub], orc.stokeslet_direct_cpu(rs, f1, rt[sub], 1.0))


def test_device_pointer_api_with_torch():
    import torch
    rs, rt, f3, _ = _rand(55, 3000, 2000)
    dev = torch.device("cuda:0")
    d_rs, d_rt, d_f = (torch.from_numpy(x).to(dev) for x in (rs, rt, f3))
    d_u = torch.empty((2000, 3), dtype=torch.float64, device=dev)
    torch.cuda.synchronize()
    with skb.Context(1) as c:
        stream = torch.cuda.current_stream().cuda_stream
        c.set_targets_device(d_rt.data_ptr(), 2000, stream)
        c.set_sources_device(SL, d_rs.data_ptr(), 3000, stream)
        c.eval_device(SL, d_f.data_ptr(), d_u.data_ptr(), False, stream)
        torch.cuda.synchronize()
        _check(d_u.cpu().numpy(), orc.stokeslet_direct(rs, f3, rt))


def test_error_paths(ctx):
    with pytest.raises(skb.SkbError):
        skb.Context(1).eval(SL, np.zeros((0, 3)))  # nothing set
    with pytest.raises(skb.SkbError):
        skb.Context(64)
    with pytest.raises(ValueError):
        ctx.set_targets(np.zeros((3, 2)))


def test_launches_are_counted(ctx):
    from skellysim_b200 import capi
    rs, rt, f3, _ = _rand(1, 300, 200)
    ctx.set_targets(rt)
    ctx.set_sources(SL, rs)
    n0 = capi.launch_count()
    ctx.eval(SL, f3)
    assert capi.launch_count() - n0 == 3  # pack + pair sums + split reduction


@pytest.mark.parametrize("kernel", ["stokeslet", "stresslet"])
@pytest.mark.parametrize("driver", ["gpu", "gpu_cached", "impl"])
def test_cpp_kernel_test_clone(kernel, driver):
    # tests/cpp/kernel_test.cpp == SkellySim tests/core/kernel_test.cpp re-created against the drop-in library:
    # C++ host code -> skelly_b200/kernels.hpp -> C ABI, plus the reference-named kernels::*_gpu_impl symbols
    import os
    import subprocess
    exe = os.path.join(os.path.dirname(os.path.abspath(__file__)), "cpp", "kernel_test")
    assert os.path.exists(exe), "tests/cpp/kernel_test not built (run __graft_entry__.build())"
    r = subprocess.run([exe, f"--kernel={kernel}", f"--driver={driver}"], capture_output=True, text=True, timeout=120)
    assert r.returncode == 0, r.stdout + r.stderr


def test_c4_scale_one_million_nodes_single_gpu():
    # BASELINE C4 size on ONE GPU: 1e6 x 1e6 = 1e12 Stokeslet pairs (~1.2-1.4 s).  Checked on a target subset against
    # the CPU port; exercises the 64-bit index paths at large n, with the symmetric kernel (47 GB of reverse partials,
    # inside the 30 %-of-HBM budget of a 180 GB B200) and with the plain kernel.
    rng = np.random.default_rng(12)
    n = 1_000_000
    rs = rng.uniform(-10, 10, (n, 3))
    f = rng.uniform(-1, 1, (n, 3))
    with skb.Context(1) as c:
        c.set_targets(rs)
        c.set_sources(SL, rs)
        u = c.eval(SL, f)
        st = c.stats()
        assert st["n_pairs"] == n * n
        used_sym = c.last_eval_was_symmetric()
        c.set_symmetric(0)
        u_plain = c.eval(SL, f)
        assert not c.last_eval_was_symmetric()
    assert np.isfinite(u).all() and np.isfinite(u_plain).all()
    sub = rng.choice(n, 64, replace=False)
    ref = orc.stokeslet_direct_cpu(rs, f, rs[sub], 1.0)
    assert rel_max(u[sub], ref) < 1e-12 and rel_max(u_plain[sub], ref) < 1e-12
    print("1e6 nodes: symmetric kernel used:", used_sym)
