"""Host-side facts of bench.py (no GPU): the workloads are the ones BASELINE.json names, both arms describe them with the
same config, and the CPU arm of the C3 matvec (the `--impl reference` / `cpu_baseline` leg) agrees with the plain-numpy
oracle on a small system."""
import json
import math

import numpy as np
import pytest

import bench
import oracle as orc


def test_c3_is_the_contract_configuration():
    nf, ns, nb, n_bodies, scaling = bench.system_sizes("c3", 1)
    assert (nf, ns, nb, n_bodies, scaling) == (3000, 6000, 400, 1, "weak")
    assert nf * 32 + ns + nb == 102400  # SURVEY.md 8d S4 / BASELINE configs[2]
    # weak scaling: nodes grow like sqrt(N) so that the pairs per GPU stay fixed
    for n, nodes in ((2, 144661), (4, 204400), (8, 288891)):
        f, s, b, _, _ = bench.system_sizes("c3", n)
        assert f * 32 + s + b == nodes
        assert abs((f * 32 + s + b) / 102400 - math.sqrt(n)) < 0.01
    assert bench.system_sizes("c4", 8)[:2] == (31250, 0) and bench.system_sizes("c4", 8)[4] == "strong"


def test_pair_count_and_config_are_facts_of_the_workload_only():
    g = bench.make_system("c3", 1, sizes=(40, 90, 30, 1, "weak"))
    nf, ns, nb = 40 * 32, 90, 30
    n_all = nf + ns + nb
    # SL fibers->all, DL periphery->fibers+bodies, DL bodies->all, SL + rotlet of the body centre -> all (system.cpp:298-316)
    assert bench.pairs_per_matvec(g) == nf * n_all + ns * (nf + nb) + (nb + 2) * n_all
    c1, c2 = bench.config_for(g, 1), bench.config_for(g, 1)
    assert c1 == c2 and json.dumps(c1)  # serialisable, deterministic
    assert c1["n_nodes"] == n_all and "system.cpp:269-324" in c1["workload"]
    assert not any(k in c1 for k in ("model", "seq_len", "global_batch"))


def test_reference_kernel_only_figure_is_read_from_the_committed_launch_list(tmp_path):
    ms = bench.ref_kernel_only_ms()
    assert ms is not None and 5.0 < ms < 100.0
    assert bench.ref_kernel_only_ms(str(tmp_path / "missing.csv")) is None
    p = tmp_path / "junk.csv"
    p.write_text('==PROF== Connected\n"ID","x"\n"0","1"\n')
    assert bench.ref_kernel_only_ms(str(p)) is None


def test_dump_outputs_writes_the_result_buffers_as_float64_npy(tmp_path):
    """--dump-outputs on one rank: each result buffer trimmed to the rows the rank owns, one .npy per array."""
    import types

    import torch
    g = bench.make_system("c3", 1, sizes=(3, 20, 5, 1, "weak"))
    nf, ns, nb = g["fib"].shape[0], g["shell"].shape[0], g["body"].shape[0]
    rng = np.random.default_rng(0)
    res, outs, vb = rng.normal(size=4 * nf + 1), rng.normal(size=(ns + 1, 3)), rng.normal(size=(nb + 1, 3))
    rs = types.SimpleNamespace(torch=types.SimpleNamespace(cuda=types.SimpleNamespace(synchronize=lambda: None)),
                               g=g, world=1, rank=0, ranges=(0, 3, 0, ns, 0, nb), nf=nf, ns=ns, nb=nb, n_fw=nf, n_sw=ns,
                               n_bw=nb, dn=object(), d_res=torch.from_numpy(res), d_outs=torch.from_numpy(outs),
                               d_vb=torch.from_numpy(vb))
    bench.dump_outputs(rs, str(tmp_path / "out"))
    got = {p.name: np.load(p) for p in (tmp_path / "out").iterdir()}
    assert sorted(got) == ["res_fibers.npy", "res_shell.npy", "v_bodies.npy"]
    assert all(a.dtype == np.float64 for a in got.values())
    assert np.array_equal(got["res_fibers.npy"], res[:4 * nf])
    assert np.array_equal(got["res_shell.npy"], outs[:ns])
    assert np.array_equal(got["v_bodies.npy"], vb[:nb])


def test_cpu_arm_matches_the_plain_oracle_on_a_small_system():
    """CpuMatvec (what `--impl reference`, `cpu_baseline` and the in-run accuracy gate use: threaded C kernels + batched
    numpy) == the loop-form oracle composition of System::apply_matvec (oracle.apply_matvec_fibers, system.cpp:298-319),
    whole matvec and row-subset form."""
    g = bench.make_system("c3", 1, sizes=(12, 150, 40, 1, "weak"))
    n, nfib = g["n"], g["n_fibers"]
    ops = bench.Ops(g, 0, nfib)
    ns = g["shell"].shape[0]
    M = bench.dense_rows(3 * ns, 3 * ns, 0)
    cpu = bench.CpuMatvec(g, ops, M)
    cpu.threads = 2
    inp = bench.make_inputs(g, 0)
    out = cpu.apply(inp)
    fib = dict(pos=g["fib"], n_nodes=g["n_nodes"], lengths=g["lengths"])
    shell = dict(pos=g["shell"], normals=g["shell_n"], density=inp["xs"])
    body = dict(pos=g["body"], normals=g["body_n"], density=inp["bd"], centers=g["centers"], forces=inp["ft"][:, :3],
                torques=inp["ft"][:, 3:])
    o = dict(n_nodes=g["n_nodes"], A=list(ops.A), force=list(ops.F), D_1_0={n: ops.D}, P={n: ops.P}, xs=ops.xs,
             length_prev=ops.lprev, plus=ops.plus)
    res, v_all = orc.apply_matvec_fibers(fib, shell, body, o, inp["x"], bench.ETA, inp["link"])
    nf = g["fib"].shape[0]
    res_shell = orc.periphery_dense_apply(M, inp["xs"].reshape(-1), v_all[nf:nf + ns].reshape(-1))

    def close(a, b):
        a, b = np.asarray(a).ravel(), np.asarray(b).ravel()
        assert a.shape == b.shape
        assert np.abs(a - b).max() <= 1e-11 * np.abs(b).max()

    close(out["res_fib"], res)
    close(out["out_shell"], res_shell)
    close(out["v_body"], v_all[nf + ns:])
    # the row-subset form the accuracy gate uses: two whole fibers + some periphery and body rows
    fsel = np.array([3, 7])
    rows = np.concatenate([np.arange(3 * n, 4 * n), np.arange(7 * n, 8 * n), nf + np.arange(0, ns, 7),
                           nf + ns + np.arange(0, 40, 3)])
    sub = cpu.apply(inp, rows=rows, fibers=fsel)
    close(sub["v_rows"], v_all[rows])
    close(sub["res_fib"], res.reshape(nfib, 4 * n)[fsel])
