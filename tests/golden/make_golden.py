#!/usr/bin/env python
"""Generate golden vectors for the pair-kernel hot path FROM THE REFERENCE ITSELF.

Run inside the build container only (needs /root/reference and numba):

    python tests/golden/make_golden.py

Imports the reference's own Green's-function kernels, `src/skelly_sim/kernels.py`
(`oseen_kernel_source_target_numba` :271-321, `stresslet_kernel_source_target_numba` :660-692,
`rotlet_kernel_source_target_numba` :335-384), evaluates them on seeded inputs and stores
inputs + outputs as small .npz fixtures next to this script.  The numba kernels regularise
r < 1e-5 instead of skipping r == 0, so every case keeps sources and targets non-coincident
(min separation asserted below); coincident-point semantics are pinned by a fourth fixture,
the outputs of the reference's CUDA kernels (oracle/_ref/libskelly_ref_kernels_cu.so, built by
`make -C oracle` from the reference tree), generated on a GPU with

    python tests/golden/make_golden.py --cuda

The fixtures are the reference's outputs: tests compare the oracle (and through it the CUDA path)
against them; nothing at test time reads the reference tree or its build.
"""
import importlib.util
import os
import sys

import numpy as np

REF = "/root/reference/src/skelly_sim/kernels.py"
HERE = os.path.dirname(os.path.abspath(__file__))


def load_ref():
    spec = importlib.util.spec_from_file_location("ref_kernels", REF)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def min_sep(a, b):
    d = a[:, None, :] - b[None, :, :]
    return np.sqrt((d * d).sum(-1)).min()


def straight_fibers(rng, n_fibers, n_nodes, length, box):
    """x0 + L*linspace(0, nhat, n) (skelly_config.py:306-308), random centre/orientation."""
    pos = []
    for _ in range(n_fibers):
        x0 = rng.uniform(-box, box, 3)
        nh = rng.normal(size=3)
        nh /= np.linalg.norm(nh)
        s = np.linspace(0.0, length, n_nodes)
        pos.append(x0[None, :] + s[:, None] * nh[None, :])
    return np.concatenate(pos)


def main():
    K = load_ref()
    cases = {}

    # S1: kernel_test.cpp clone -- n_src=1229, n_trg=743, eta=1.3, U[-1,1] (kernel_test.cpp:25-37), seeded
    rng = np.random.default_rng(1)
    r_src = rng.uniform(-1, 1, (1229, 3))
    r_trg = rng.uniform(-1, 1, (743, 3))
    cases["kernel_test"] = dict(r_src=r_src, r_trg=r_trg, eta=1.3, f_sl=rng.uniform(-1, 1, (1229, 3)),
                                normals=rng.uniform(-1, 1, (1229, 3)), density=rng.uniform(-1, 1, (1229, 3)),
                                torque=rng.uniform(-1, 1, (1229, 3)))

    # small ragged case (sizes not multiples of anything)
    rng = np.random.default_rng(2)
    cases["ragged"] = dict(r_src=rng.uniform(-2, 2, (37, 3)), r_trg=rng.uniform(-2, 2, (5, 3)), eta=0.7,
                           f_sl=rng.normal(size=(37, 3)), normals=rng.normal(size=(37, 3)),
                           density=rng.normal(size=(37, 3)), torque=rng.normal(size=(37, 3)))

    # single source / single target
    rng = np.random.default_rng(3)
    cases["single"] = dict(r_src=rng.uniform(-1, 1, (1, 3)), r_trg=rng.uniform(2, 3, (1, 3)), eta=1.0,
                           f_sl=rng.normal(size=(1, 3)), normals=rng.normal(size=(1, 3)),
                           density=rng.normal(size=(1, 3)), torque=rng.normal(size=(1, 3)))

    # C1-like: 16 fibers x 32 nodes as sources; targets = a shifted copy (non-coincident) + shell-like ring
    rng = np.random.default_rng(4)
    fib = straight_fibers(rng, 16, 32, 1.0, 2.0)
    trg = fib + rng.uniform(0.01, 0.02, fib.shape)
    cases["fibers16x32"] = dict(r_src=fib, r_trg=trg, eta=1.0, f_sl=rng.uniform(-1, 1, fib.shape),
                                normals=rng.normal(size=fib.shape), density=rng.uniform(-1, 1, fib.shape),
                                torque=rng.uniform(-1, 1, fib.shape))

    # wide dynamic range of separations (near-singular pairs at 1e-4 .. far pairs at 1e2)
    rng = np.random.default_rng(5)
    r_src = rng.uniform(-1, 1, (300, 3)) * np.logspace(-2, 2, 300)[:, None]
    r_trg = r_src[:200] + rng.normal(size=(200, 3)) * 1e-4
    cases["wide_range"] = dict(r_src=r_src, r_trg=r_trg, eta=2.5, f_sl=rng.normal(size=(300, 3)),
                               normals=rng.normal(size=(300, 3)), density=rng.normal(size=(300, 3)),
                               torque=rng.normal(size=(300, 3)))

    for name, c in cases.items():
        sep = min_sep(c["r_trg"], c["r_src"])
        assert sep > 2e-5, (name, sep)  # stay clear of the python kernels' regularisation branch
        eta = c["eta"]
        nt = c["r_trg"].shape[0]
        u_sl = K.oseen_kernel_source_target_numba(c["r_src"].ravel(), c["r_trg"].ravel(), c["f_sl"].ravel(),
                                                  eta=eta).reshape(nt, 3)
        u_dl = K.stresslet_kernel_source_target_numba(c["r_src"].ravel(), c["r_trg"].ravel(), c["normals"].ravel(),
                                                      c["density"].ravel(), eta=eta).reshape(nt, 3)
        u_rot = K.rotlet_kernel_source_target_numba(c["r_src"].ravel(), c["r_trg"].ravel(), c["torque"].ravel(),
                                                    eta=eta).reshape(nt, 3)
        out = os.path.join(HERE, f"ref_numba_{name}.npz")
        np.savez_compressed(out, u_stokeslet=u_sl, u_stresslet=u_dl, u_rotlet=u_rot, min_sep=sep, **c)
        print(f"{name}: n_src={c['r_src'].shape[0]} n_trg={nt} min_sep={sep:.3e} -> {os.path.basename(out)} "
              f"({os.path.getsize(out)} B)")


def regularised():
    """Second fixture: the regularised branch (0 < r < epsilon_distance = 1e-5 -> r := sqrt(r^2 + reg^2), reg = 5e-3) of
    the helpers the flow layer uses next to the big sums -- `oseen_kernel_source_target_numba` (:271-321, the same rule
    as kernels::oseen_tensor_contract_direct, kernels.cpp:146-195, for every r > 0), `rotlet_kernel_source_target_numba`
    (:335-384 == kernels::rotlet, kernels.cpp:206-242, including r == 0) and the self form
    `oseen_kernel_times_density_numba` (:196-268, diagonal skipped like `dr2 == 0 -> continue` in the C++)."""
    K = load_ref()
    rng = np.random.default_rng(11)
    src = straight_fibers(rng, 2, 16, 1.0, 1.0)
    n = src.shape[0]
    dirs = rng.normal(size=(n, 3))
    dirs /= np.linalg.norm(dirs, axis=1)[:, None]
    # one target per source at a controlled distance: inside the regularised ball, just outside, far
    dist = np.concatenate([np.full(10, 3e-6), np.full(6, 8e-6), np.full(6, 1.5e-5), np.full(n - 22, 2e-2)])
    trg = src + dirs * dist[:, None]
    # rotlet only: two targets exactly ON sources (contribution 0 in both implementations)
    trg_rot = np.concatenate([trg, src[:2]])
    f, t = rng.uniform(-1, 1, (n, 3)), rng.uniform(-1, 1, (n, 3))
    eta = 0.8
    u_oseen = K.oseen_kernel_source_target_numba(src.ravel(), trg.ravel(), f.ravel(), eta=eta).reshape(-1, 3)
    u_rot = K.rotlet_kernel_source_target_numba(src.ravel(), trg_rot.ravel(), t.ravel(), eta=eta).reshape(-1, 3)
    # self form: a fiber whose nodes 3/4 and 9/10 are closer than epsilon_distance
    x = straight_fibers(rng, 1, 12, 1.0, 0.5)
    x[4] = x[3] + 4e-6 * dirs[0]
    x[10] = x[9] + 9e-6 * dirs[1]
    fs = rng.uniform(-1, 1, x.shape)
    u_self = K.oseen_kernel_times_density_numba(x.ravel(), fs.ravel(), eta=eta).reshape(-1, 3)
    out = os.path.join(HERE, "ref_numba_regularised.npz")
    np.savez_compressed(out, r_src=src, r_trg=trg, r_trg_rotlet=trg_rot, f=f, torque=t, eta=eta, u_oseen=u_oseen,
                        u_rotlet=u_rot, x_self=x, f_self=fs, u_self=u_self, dist=dist)
    print(f"regularised: {n} sources, {int((dist < 1e-5).sum())} pairs inside the regularised ball -> "
          f"{os.path.basename(out)} ({os.path.getsize(out)} B)")


def shell_double_layer():
    """Third fixture: the periphery's double layer as the reference's precompute builds it --
    `stresslet_kernel_times_normal_numba` (:535-590), the matrix precompute.py:113 starts
    `stresslet_plus_complementary` from -- contracted with a density.  Its off-diagonal blocks are the kernel
    Periphery::flow evaluates (periphery.cpp:55-79: f_dl = 2 eta n (x) rho, stresslet, / eta), so
    S @ density == Periphery::flow at the shell's own nodes with the r = 0 pairs skipped; this pins the normal /
    density index convention and the -3/(4 pi) normalisation on a second, independent reference function."""
    K = load_ref()
    rng = np.random.default_rng(21)
    n = 60
    d = rng.normal(size=(n, 3))
    d /= np.linalg.norm(d, axis=1)[:, None]
    nodes = d * np.array([3.0, 2.0, 2.0])
    normals = -d / np.array([3.0, 2.0, 2.0])
    normals /= np.linalg.norm(normals, axis=1)[:, None]     # inward normals of the ellipsoid
    density = rng.uniform(-1, 1, (n, 3))
    S = K.stresslet_kernel_times_normal_numba(nodes.ravel(), normals.ravel(), eta=1.0)
    u = (S @ density.ravel()).reshape(n, 3)
    out = os.path.join(HERE, "ref_numba_shell_double_layer.npz")
    np.savez_compressed(out, nodes=nodes, normals=normals, density=density, u=u,
                        S_block_0_1=S[0:3, 3:6], S_diag_max=np.abs(np.stack([S[3 * i:3 * i + 3, 3 * i:3 * i + 3]
                                                                            for i in range(n)])).max())
    print(f"shell_double_layer: {n} nodes -> {os.path.basename(out)} ({os.path.getsize(out)} B)")


def reference_cuda():
    """Fourth fixture: kernels::stokeslet_direct_gpu_impl / stresslet_direct_gpu_impl of the reference's kernels.cu,
    compiled unmodified, on the kernel_test.cpp shape (1229 sources, 743 targets) with 17 targets ON sources: the
    r == 0 pairs the numba kernels cannot pin (they regularise) contribute exactly 0 here."""
    sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
    import oracle as orc
    if not orc.refgpu_available():
        sys.exit("oracle/_ref/libskelly_ref_kernels_cu.so not built: run `make -C oracle` with the reference tree")
    rng = np.random.default_rng(21)
    r_src = rng.uniform(-1, 1, (1229, 3))
    r_trg = rng.uniform(-1, 1, (743, 3))
    r_trg[:17] = r_src[:17]
    f_sl, f_dl = rng.uniform(-1, 1, (1229, 3)), rng.uniform(-1, 1, (1229, 9))
    u_sl = orc.ref_stokeslet_direct_gpu_impl(r_src, f_sl, r_trg)
    u_dl = orc.ref_stresslet_direct_gpu_impl(r_src, f_dl, r_trg)
    out = os.path.join(HERE, "ref_cuda_kernels.npz")
    np.savez_compressed(out, r_src=r_src, r_trg=r_trg, f_sl=f_sl, f_dl=f_dl, u_stokeslet=u_sl, u_stresslet=u_dl)
    print(f"reference_cuda: n_src={r_src.shape[0]} n_trg={r_trg.shape[0]} -> {os.path.basename(out)} "
          f"({os.path.getsize(out)} B)")


if __name__ == "__main__":
    if sys.argv[1:] == ["--cuda"]:
        reference_cuda()
        sys.exit(0)
    if not os.path.exists(REF):
        sys.exit("reference tree not present: golden vectors can only be regenerated in the build container")
    main()
    regularised()
    shell_double_layer()
