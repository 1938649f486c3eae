#!/usr/bin/env python
"""bench.py -- headline benchmark of the SkellySim hydrodynamic hot path on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--workload c3|c2|c4] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W

Metric (BASELINE.json): "Stokeslet pair-interactions/s; GMRES matvec ms at N=1e5 nodes, 1/2/4/8 GPU".  One matvec =
one System::apply_matvec (src/core/system.cpp:269-324): apply_fiber_force, the four evaluator calls (Stokeslet
fibers -> all, stresslet periphery -> fibers+bodies, stresslet + Stokeslet + rotlet bodies -> all), the fiber self
term, fc.matvec and the periphery's dense operator -- on the BASELINE C3 system (3000 fibers x 32 nodes + 6000
periphery nodes + 1 body x 400 nodes = 102 400 nodes), geometry and operators resident on the device(s) exactly as
between the GMRES iterations of one timestep, the solution vector changing every matvec.  One timed STEP = 8 consecutive
matvecs (a slice of one GMRES solve), so that the driver's 20 steps time ~2 s of GPU work.

  value : whole-job pair interactions per second = (source x target pairs of one matvec) x matvecs / time, operands
          already in HBM (device-pointer C ABI, skb_flow_apply_matvec_device).  ms_per_matvec is printed next to it.
  e2e   : the same matvecs through the reference-facing call with HOST buffers (N = 1: skb_flow_apply_matvec_dense, the
          C ABI call a SkellySim integration makes; H2D of the solution vector and D2H of the result inside every call).
  N > 1 : one rank per GPU, weak scaling (node counts ~ sqrt(N): pairs per GPU stay fixed).  Every rank owns whole
          fibers, periphery rows and body rows; strengths and partial velocities travel through peer memory inside the
          library's own kernels (group_kernels.cuh) -- no collective call per matvec.  --exchange nccl: the round-1
          path (torch.distributed all-gather, plain kernel on own rows) for A/B.
  extras: roofline of the dominant kernel (symmetric fiber-fiber block) measured live with CUDA events inside the timed
          steps; cpu_baseline = the CPU port of the same matvec on all host cores (N = 1); stokeslet_call, solve
          (K GMRES-shaped iterations P^-1 then A, device resident), periphery_dense, fiber_operators, ref_gpu_baseline
          (the reference's kernels.cu on this GPU), strong scaling of the fixed C3 system and the in-process
          multi-device flow (skb_mflow) at N > 1.

Prints ONE JSON line (rank 0).  `--impl reference` times the CPU port of the reference's OpenMP direct path for the
same matvec (oracle/, all host threads; PVFMM/STKFMM/Eigen are not installable here); ranks > 0 exit at once.
`--dump-outputs DIR` writes the result of the last timed matvec (res_fibers, res_shell, v_bodies; float64 .npy) so that
two builds can be compared output for output on the same seeded inputs.
"""
from __future__ import annotations

import argparse
import json
import math
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")
os.environ.setdefault("NCCL_DEBUG", "WARN")  # (no "NCCL version ..." line on stdout next to the JSON line)

SL_FLOP_PER_PAIR = 28  # SURVEY.md 8d / BASELINE.md 2.1 (kernels.cu:65-75)
DL_FLOP_PER_PAIR = 40
NOMINAL_FP64_TFLOPS = 148 * 64 * 2 * 1.965e9 / 1e12  # 148 SMs x 64 DFMA/clk x 2 flop x max SM clock = 37.2
UBENCH_FP64_TFLOPS = 36.1  # 2-register DFMA micro-benchmark on this GPU model, profiles/r1_fp64_ubench.md
INNER = 8  # matvecs per timed step
ETA = 1.0


# ------------------------------------------------------------------------------------------------
# synthetic system (SURVEY.md 8d S3/S4, Appendix C)
# ------------------------------------------------------------------------------------------------
def make_suspension(n_fibers: int, n_shell: int, seed: int = 1, n_nodes: int = 32, length: float = 1.0):
    """Straight fibers x0 + L*linspace(0,1,n)*nhat (skelly_config.py:306-308) with random centres inside the
    ellipsoid a,b,c = 7.8,4.16,4.16 (skelly_config.py:548-550) scaled with the fiber count; shell nodes on the
    1.04x surface (precompute.py:34) with inward normals (precompute.py:78-80)."""
    rng = np.random.default_rng(seed)
    scale = max(1.0, (n_fibers / 1000.0) ** (1.0 / 3.0))
    abc = np.array([7.8, 4.16, 4.16]) * scale
    c = rng.normal(size=(n_fibers, 3))
    c /= np.linalg.norm(c, axis=1)[:, None]
    c *= (rng.uniform(0, 1, n_fibers) ** (1 / 3))[:, None] * 0.85
    centres = c * abc
    nh = rng.normal(size=(n_fibers, 3))
    nh /= np.linalg.norm(nh, axis=1)[:, None]
    s = np.linspace(-0.5 * length, 0.5 * length, n_nodes)
    fib = (centres[:, None, :] + s[None, :, None] * nh[:, None, :]).reshape(-1, 3)
    d = rng.normal(size=(max(n_shell, 1), 3))[:n_shell]
    d /= np.linalg.norm(d, axis=1)[:, None] if n_shell else 1.0
    shell = d * abc * 1.04
    nrm = -(shell / (abc * 1.04) ** 2)
    if n_shell:
        nrm /= np.linalg.norm(nrm, axis=1)[:, None]
    return np.ascontiguousarray(fib), np.ascontiguousarray(shell), np.ascontiguousarray(nrm), nh


def system_sizes(workload: str, n_gpus: int):
    """(n_fibers, n_shell, n_body_nodes, n_bodies, scaling).  c3/c2 grow like sqrt(N) (pairs per GPU fixed: weak);
    c4 is the fixed 1e6-node free-fiber suspension (strong)."""
    g = math.sqrt(n_gpus)
    if workload == "c3":   # configs[2]-like, SURVEY.md 8d S4: 3000 x 32 + 6000 + 1 x 400 = 102 400 nodes at N = 1
        return int(round(3000 * g)), int(round(6000 * g)), 400, 1, "weak"
    if workload == "c2":   # configs[1]: 1000 fibers x 32 + 8000-node ellipsoid periphery
        return int(round(1000 * g)), int(round(8000 * g)), 0, 0, "weak"
    if workload == "c4":   # configs[3]: 31 250 x 32 = 1e6 free-fiber nodes, target-partitioned over the GPUs
        return 31250, 0, 0, 0, "strong"
    raise SystemExit(f"unknown workload {workload}")


def make_system(workload: str, n_gpus: int, seed: int = 2, sizes=None):
    n_fibers, n_shell, n_body, n_bodies, scaling = sizes or system_sizes(workload, n_gpus)
    fib, shell, nrm, nh = make_suspension(n_fibers, n_shell, seed=seed)
    rng = np.random.default_rng(seed)
    e = rng.normal(size=(max(n_body, 1), 3))[:n_body]
    if n_body:
        e /= np.linalg.norm(e, axis=1)[:, None]
    centers = np.zeros((n_bodies, 3))
    body = (centers[0] + 0.5 * e) if n_bodies else np.zeros((0, 3))
    return dict(workload=workload, scaling=scaling, n_fibers=n_fibers, n=32, fib=fib, nh=nh,
                n_nodes=np.full(n_fibers, 32, dtype=np.int32), lengths=np.ones(n_fibers), shell=shell, shell_n=nrm,
                body=np.ascontiguousarray(body), body_n=np.ascontiguousarray(e), centers=centers, n_bodies=n_bodies)


def pairs_per_matvec(g) -> float:
    nf, ns, nb = g["fib"].shape[0], g["shell"].shape[0], g["body"].shape[0]
    n_all = nf + ns + nb
    return float(nf) * n_all + float(ns) * (nf + nb) + float(nb + 2 * g["n_bodies"]) * n_all


def flop_per_matvec(g) -> float:
    nf, ns, nb = g["fib"].shape[0], g["shell"].shape[0], g["body"].shape[0]
    n_all = nf + ns + nb
    return (SL_FLOP_PER_PAIR * (float(nf) + g["n_bodies"]) * n_all
            + DL_FLOP_PER_PAIR * (float(ns) * (nf + nb) + float(nb) * n_all))


def config_for(g, n_gpus: int) -> dict:
    """Facts of the workload only -- identical in the GPU arm and the reference arm."""
    nf, ns, nb = g["fib"].shape[0], g["shell"].shape[0], g["body"].shape[0]
    return {"workload": (f"{g['workload']}: System::apply_matvec (system.cpp:269-324) on {g['n_fibers']} fibers x 32 nodes "
                         f"+ {ns} periphery nodes + {g['n_bodies']} body x {nb} nodes = {nf + ns + nb} nodes; FP64 direct "
                         "kernels; SL fibers->all, DL periphery->fibers+bodies, DL+SL+rotlet bodies->all, fiber self "
                         "term, per-fiber operators, periphery dense operator"),
            "n_fiber_nodes": nf, "n_shell_nodes": ns, "n_body_nodes": nb, "n_nodes": nf + ns + nb,
            "pairs_per_matvec": pairs_per_matvec(g), "n_gpus_sized_for": n_gpus, "eta": ETA}


class Ops:
    """Per-fiber operators of fibers [f0, f1) with the reference's shapes and sparsity (fiber_finite_difference.cpp:
    97-187, 317-335, 519-558): A_ 4n x 4n and force_operator_ 3n x 4n dense per fiber; D_1_0 n x n banded (5-point
    stencils); P_downsample_bc (4n-14) x 4n block diagonal (three (n-4) x n blocks and one (n-2) x n).  Entries are
    random: the kernels treat them as dense GEMV operands, only the block structure of P is exploited.  Generated in
    blocks of 256 fibers with their own seeds, so any rank (and the checker) can rebuild any fiber's operators."""
    BLOCK = 256

    @staticmethod
    def _range(kind: int, rows: int, n: int, f0: int, f1: int, seed: int):
        """Storage array (fibers, 4n columns, rows): every fiber's matrix COLUMN-major, as Eigen's .data() -- what the C
        ABI takes.  The matrix itself is the transposed view."""
        out = np.empty((f1 - f0, 4 * n, rows))
        for blk in range(f0 // Ops.BLOCK, (max(f1, 1) - 1) // Ops.BLOCK + 1):
            lo, hi = blk * Ops.BLOCK, (blk + 1) * Ops.BLOCK
            a, b = max(lo, f0), min(hi, f1)
            if b <= a:
                continue
            rng = np.random.default_rng([seed, kind, blk])
            m = rng.standard_normal((Ops.BLOCK, 4 * n, rows))
            out[a - f0:b - f0] = m[a - lo:b - lo]
        out /= np.sqrt(4 * n)
        return out

    @staticmethod
    def A_range(g, f0, f1, seed=6):
        return Ops._range(0, 4 * g["n"], g["n"], f0, f1, seed).transpose(0, 2, 1)

    @staticmethod
    def F_range(g, f0, f1, seed=6):
        return Ops._range(1, 3 * g["n"], g["n"], f0, f1, seed).transpose(0, 2, 1)

    def __init__(self, g, f0: int, f1: int, seed: int = 6, with_A=True):
        n = g["n"]
        self.n, self.f0, self.f1 = n, f0, f1
        self.A = Ops.A_range(g, f0, f1, seed) if with_A else None   # (k, 4n, 4n) views of column-major storage
        self.F = Ops.F_range(g, f0, f1, seed)                       # (k, 3n, 4n)
        self.xs = np.repeat(g["nh"][f0:f1], n, axis=0)              # straight fibers: the tangent is nhat everywhere
        self.lprev = np.ones(f1 - f0)
        self.plus = (np.random.default_rng([seed, 2]).integers(0, 2, g["n_fibers"]).astype(np.int32))[f0:f1]
        crng = np.random.default_rng([seed, 3])                      # class matrices: the same on every rank
        D = np.zeros((n, n))
        for i in range(n):
            lo = min(max(i - 2, 0), n - 5)
            D[lo:lo + 5, i] = crng.standard_normal(5)               # stored pre-transposed (ffd.cpp:537)
        P = np.zeros((4 * n - 14, 4 * n))
        for b in range(3):
            P[b * (n - 4):(b + 1) * (n - 4), b * n:(b + 1) * n] = crng.standard_normal((n - 4, n)) / np.sqrt(n)
        P[3 * (n - 4):, 3 * n:] = crng.standard_normal((n - 2, n)) / np.sqrt(n)
        self.D, self.P = D, P


def make_inputs(g, k: int):
    """Solution-sized inputs of matvec number k: x_fibers (4 N_f), x_shell, body densities, forces|torques, link."""
    rng = np.random.default_rng(1000 + k)
    nf, ns, nb = g["fib"].shape[0], g["shell"].shape[0], g["body"].shape[0]
    return dict(x=rng.standard_normal(4 * nf), xs=rng.uniform(-1, 1, (ns, 3)), bd=rng.uniform(-1, 1, (nb, 3)),
                ft=rng.uniform(-1, 1, (g["n_bodies"], 6)), link=rng.standard_normal((g["n_fibers"], 7)))


def dense_rows(n_rows: int, n_cols: int, row0: int, seed: int = 4):
    """Rows [row0, row0 + n_rows) of the periphery's dense operator (stresslet_plus_complementary_), reproducible per
    row block."""
    rng = np.random.default_rng(seed + 104729 * (row0 + 1))
    A = rng.random((n_rows, n_cols))
    A -= 0.5
    A *= 2.0 / max(n_cols, 1)
    return A


# ------------------------------------------------------------------------------------------------
# clocks / throttle sampling during the timed region (pynvml, no subprocess)
# ------------------------------------------------------------------------------------------------
class ClockSampler:
    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap",
               0x80: "hw_power_brake_slowdown", 0x2: "applications_clocks_setting", 0x100: "display_clock_setting"}

    def __init__(self, index: int, period_s: float = 0.02):
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop = threading.Event()
        self._thr = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self._nv = pynvml
            self._h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self._h, pynvml.NVML_CLOCK_SM)
        except Exception as e:  # pragma: no cover
            self._nv = None
            self.err = str(e)
        self.period = period_s

    def _run(self):
        nv = self._nv
        while not self._stop.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self._h, nv.NVML_CLOCK_SM))
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(self._h)
                except Exception:
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self._h)
                for bit, name in self.REASONS.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            self._stop.wait(self.period)

    def __enter__(self):
        if self._nv:
            self._thr = threading.Thread(target=self._run, daemon=True)
            self._thr.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        if self._thr:
            self._thr.join()

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": 0}
        return {"sm_mhz": float(np.median(self.samples)), "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(self.samples)}


# ------------------------------------------------------------------------------------------------
# CPU arm: the same System::apply_matvec on the host cores (oracle port of kernels::*_direct_cpu with the reference's
# OpenMP target chunking, kernels.cpp:42-83, + BLAS for the dense algebra the reference does with Eigen)
# ------------------------------------------------------------------------------------------------
def host_thread_candidates():
    try:
        full = max(1, len(os.sched_getaffinity(0)))
    except AttributeError:
        full = max(1, os.cpu_count() or 1)
    return sorted({full, max(1, full // 2)}, reverse=True)


class CpuMatvec:
    """Times / evaluates the matvec on the CPU.  rows: optional subset of v_all rows [fibers | shell | bodies] to
    evaluate the pair sums at (bounded sample / accuracy gate); None = all."""

    def __init__(self, g, ops: "Ops", M, F_all=None):
        """ops: operators of fibers [ops.f0, ops.f1) (the fibers whose res_fibers may be asked for); F_all: the
        force operators of ALL fibers (defaults to ops.F when ops covers the container)."""
        import oracle as orc
        self.orc, self.g, self.ops, self.M = orc, g, ops, M
        self.F_all = F_all if F_all is not None else ops.F
        assert self.F_all.shape[0] == g["n_fibers"]
        self.threads = None
        self.thread_probe = {}
        n, nfib = g["n"], g["n_fibers"]
        self.w = np.tile(orc.trapezoid_weights(n, 1.0), nfib)
        self.r_all = np.concatenate([g["fib"], g["shell"], g["body"]])

    def pick_threads(self):
        """All logical CPUs or one per physical core (SMT off), whichever is faster on a probe; both are reported."""
        if self.threads is not None:
            return self.threads
        g, orc = self.g, self.orc
        f = np.random.default_rng(0).uniform(-1, 1, g["fib"].shape)
        probe = self.r_all[:max(2048, 64 * host_thread_candidates()[0])]
        for th in host_thread_candidates():
            orc.stokeslet_direct_cpu(g["fib"], f, probe, 1.0, th)
            t0 = time.perf_counter()
            for _ in range(2):
                orc.stokeslet_direct_cpu(g["fib"], f, probe, 1.0, th)
            self.thread_probe[th] = 2 * g["fib"].shape[0] * probe.shape[0] / (time.perf_counter() - t0)
        self.threads = max(self.thread_probe, key=self.thread_probe.get)
        return self.threads

    def apply(self, inp, rows=None, fibers=None):
        """Returns dict(res_fib, out_shell, v_body, v_rows).  rows = None: whole matvec.  rows given: pair sums only at
        those rows of v_all; res_fib then only for the listed `fibers` (whose nodes must be in rows)."""
        g, ops, orc, th = self.g, self.ops, self.orc, self.pick_threads()
        n, nfib = g["n"], g["n_fibers"]
        nf, ns, nb = g["fib"].shape[0], g["shell"].shape[0], g["body"].shape[0]
        x = inp["x"].reshape(nfib, 4 * n)
        # fw = fc.apply_fiber_force(x_fibers)            system.cpp:298, fcfd.cpp:272-287
        ff = np.matmul(self.F_all, x[:, :, None])[:, :, 0]                # (nfib, 3n): rows k*n + i
        fw = ff.reshape(nfib, 3, n).transpose(0, 2, 1).reshape(nf, 3)
        wf = fw * self.w[:, None]
        r_t = self.r_all if rows is None else self.r_all[rows]
        # v_all = fc.flow(r_all, fw, eta)               system.cpp:299
        v = orc.stokeslet_direct_cpu(g["fib"], wf, r_t, ETA, th)
        # v_fibers, v_bodies += shell.flow(r_fibbody)     system.cpp:301-315
        if ns:
            f_dl = orc.form_double_layer(g["shell_n"], inp["xs"], ETA)
            not_shell = np.ones(r_t.shape[0], dtype=bool)
            idx = np.arange(nf + ns + nb) if rows is None else np.asarray(rows)
            not_shell = (idx < nf) | (idx >= nf + ns)
            if not_shell.any():
                v[not_shell] += orc.stresslet_direct_cpu(g["shell"], f_dl, r_t[not_shell], ETA, th)
        # v_all += bc.flow(r_all, x_bodies, links)       system.cpp:316
        if nb:
            f_b = orc.form_double_layer(g["body_n"], inp["bd"], ETA)
            v += orc.stresslet_direct_cpu(g["body"], f_b, r_t, ETA, th)
            v += orc.stokeslet_direct_cpu(g["centers"], inp["ft"][:, :3], r_t, ETA, th)
            v += orc.rotlet(g["centers"], r_t, inp["ft"][:, 3:], ETA)
        # self term of every fiber (fcfd.cpp:203-210), batched over equal-size fibers
        idx = np.arange(nf + ns + nb) if rows is None else np.asarray(rows)
        fsel = np.arange(nfib) if fibers is None else np.asarray(fibers)
        if rows is None or fibers is not None:
            X = g["fib"].reshape(nfib, n, 3)[fsel]
            W = wf.reshape(nfib, n, 3)[fsel]
            d = X[:, :, None, :] - X[:, None, :, :]
            r2 = np.einsum("fijk,fijk->fij", d, d)
            with np.errstate(divide="ignore"):
                ri = np.where(r2 > 0, 1.0 / np.sqrt(r2), 0.0)
            dw = np.einsum("fijk,fjk->fij", d, W)
            self_v = (np.einsum("fij,fjk->fik", ri, W) + np.einsum("fij,fijk->fik", dw * ri ** 3, d)) / (8 * np.pi * ETA)
            pos = {int(r): i for i, r in enumerate(idx)} if rows is not None else None
            for k, f in enumerate(fsel):
                sl = slice(f * n, (f + 1) * n)
                if rows is None:
                    v[sl] -= self_v[k]
                else:
                    where = [pos[j] for j in range(f * n, (f + 1) * n)]
                    v[where] -= self_v[k]
        out = {"v_rows": v}
        # res_fibers = fc.matvec(x_fibers, v_fibers, links)   system.cpp:318, ffd.cpp:276-312
        if rows is None or fibers is not None:
            bc = 4 * n - 14
            if rows is None:
                vf = v[:nf].reshape(nfib, n, 3)
            else:
                vf = np.stack([v[[pos[j] for j in range(f * n, (f + 1) * n)]] for f in fsel])
            fo = fsel - ops.f0                                            # index into the operators held by `ops`
            xs = ops.xs.reshape(-1, n, 3)[fo]
            D1 = ops.D[None] * (2.0 / ops.lprev[fo])[:, None, None]
            s = np.einsum("fik,fik->fi", xs, vf)
            vT = np.concatenate([vf[:, :, 0], vf[:, :, 1], vf[:, :, 2], np.einsum("fij,fi->fj", D1, s)], axis=1)
            res = np.matmul(ops.A[fo], x[fsel][:, :, None])[:, :, 0]
            res[:, :bc] -= vT @ ops.P.T
            res[:, bc + 3] += np.einsum("fk,fk->f", vf[:, 0], xs[:, 0])
            res[:, bc:bc + 7] += inp["link"][fsel]
            pl = ops.plus[fo].astype(bool)
            res[pl, bc + 10] += np.einsum("fk,fk->f", vf[pl, n - 1], xs[pl, n - 1])
            out["res_fib"] = res
        if rows is None:
            if ns:  # res_shell = stresslet_plus_complementary_ * x_shell + v_shell     periphery.cpp:38-47
                out["out_shell"] = (self.M @ inp["xs"].reshape(-1)).reshape(ns, 3) + v[nf:nf + ns] if self.M is not None \
                    else v[nf:nf + ns]
            out["v_body"] = v[nf + ns:]
        return out


def cpu_timed(cpu: CpuMatvec, inputs, budget_s: float):
    """Repeat whole matvecs for ~budget_s; returns (pairs/s, calls, seconds)."""
    cpu.apply(inputs[0])  # warm-up (page faults, thread pool)
    calls, t0 = 0, time.perf_counter()
    while True:
        cpu.apply(inputs[calls % len(inputs)])
        calls += 1
        dt = time.perf_counter() - t0
        if dt >= budget_s or calls >= 1000:
            break
    return calls * pairs_per_matvec(cpu.g) / dt, calls, dt


def cpu_baseline_dict(cpu: CpuMatvec, val, calls, dt, orc):
    return {"value": val, "unit": "pairs/s", "cores": cpu.threads, "kind": "port",
            "simd": {0: "scalar", 1: "avx2+fma", 2: "avx512"}[orc.simd_level()],
            "threads_tried": {str(k): v for k, v in cpu.thread_probe.items()},
            "ms_per_matvec": 1e3 * dt / calls,
            "sample": f"{calls} whole matvecs of the workload in {dt:.2f} s; pair kernels = CPU port of "
                      "kernels::stokeslet/stresslet_direct_cpu with the reference's OpenMP static target chunks "
                      "(kernels.cpp:42-83), AVX-512; dense algebra = multithreaded BLAS (the reference uses Eigen); the "
                      "reference's own CPU path needs PVFMM/STKFMM: unbuildable here"}


def run_reference_arm(args, rank):
    """--impl reference: the CPU implementation of the same matvec on the host cores, all threads.  Each step is a
    bounded sample of the workload: the whole matvec when it has <= 1.3e10 pairs (C3 at N = 1), else the leading 1/k
    of the fibers, periphery rows and body rows as targets against ALL sources (value = pairs evaluated / time)."""
    if rank != 0:
        return
    import oracle as orc
    g = make_system(args.workload, args.gpus)
    nfib, n = g["n_fibers"], g["n"]
    nf, ns, nb = g["fib"].shape[0], g["shell"].shape[0], g["body"].shape[0]
    k = max(1, int(math.ceil(pairs_per_matvec(g) / 1.3e10)))
    inputs = [make_inputs(g, i) for i in range(2)]
    if k == 1:
        ops = Ops(g, 0, nfib)
        M = dense_rows(3 * ns, 3 * ns, 0) if ns else None
        cpu = CpuMatvec(g, ops, M)
        step = lambda i: cpu.apply(inputs[i % 2])
        pairs_step = pairs_per_matvec(g)
        sample = "each step = ONE whole matvec of the workload (the GPU arm's step is 8 matvecs)"
    else:
        fsel = np.arange(max(1, nfib // k))
        s_sel, b_sel = np.arange(ns // k), np.arange(nb // k)
        rows = np.concatenate([np.arange(len(fsel) * n), nf + s_sel, nf + ns + b_sel]).astype(int)
        ops = Ops(g, 0, len(fsel))
        cpu = CpuMatvec(g, ops, None, F_all=Ops.F_range(g, 0, nfib))
        M_sub = dense_rows(3 * len(s_sel), 3 * ns, 0) if len(s_sel) else None

        def step(i):
            out = cpu.apply(inputs[i % 2], rows=rows, fibers=fsel)
            if M_sub is not None:
                out["out_shell"] = (M_sub @ inputs[i % 2]["xs"].reshape(-1))
            return out
        n_rows = len(rows)
        pairs_step = (float(nf) * n_rows + float(ns) * (n_rows - len(s_sel)) + float(nb + 2 * g["n_bodies"]) * n_rows)
        sample = (f"each step = the leading 1/{k} of the fibers, periphery rows and body rows ({n_rows} target rows, their "
                  f"res_fibers and dense-operator rows) against ALL {nf + ns + nb} sources: {pairs_step:.3e} of "
                  f"{pairs_per_matvec(g):.3e} pairs of one matvec")
    for i in range(max(1, min(args.warmup, 2))):
        step(i)
    t0 = time.perf_counter()
    for i in range(args.steps):
        step(i)
    dt = time.perf_counter() - t0
    val = args.steps * pairs_step / dt
    cb = cpu_baseline_dict(cpu, val, args.steps, dt, orc)
    cb["sample"] = sample + "; " + cb["sample"]
    cb["ms_per_matvec"] = 1e3 * dt / args.steps * pairs_per_matvec(g) / pairs_step
    print(json.dumps({
        "impl": "reference", "metric": "pair_interactions_per_s", "value": val, "unit": "pairs/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps,
        "ms_per_matvec": cb["ms_per_matvec"], "higher_is_better": True, "scaling": g["scaling"], "vs_baseline": None,
        "dtype": "f64", "data": "synthetic", "config": config_for(g, args.gpus), "cpu_baseline": cb,
        "e2e": {"value": val, "unit": "pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0}))


_T0 = time.perf_counter()


def _log(msg):
    if os.environ.get("BENCH_VERBOSE"):
        print(f"[bench +{time.perf_counter() - _T0:7.1f}s] {msg}", file=sys.stderr, flush=True)


# ------------------------------------------------------------------------------------------------
# one rank's device state for a system
# ------------------------------------------------------------------------------------------------
class RankSystem:
    """Flow + dense handle of one rank (whole system at world == 1), inputs resident on the device and in pinned host
    memory, and the step functions."""

    def __init__(self, torch, skb, g, rank, world, local_rank, exchange="peer", with_dense=True, n_inputs=2):
        from skellysim_b200 import capi
        from skellysim_b200.distributed import connect_group
        self.torch, self.skb, self.g, self.rank, self.world = torch, skb, g, rank, world
        self.dev = torch.device("cuda", local_rank)
        nfib, n = g["n_fibers"], g["n"]
        nf, ns, nb = g["fib"].shape[0], g["shell"].shape[0], g["body"].shape[0]
        self.nf, self.ns, self.nb = nf, ns, nb
        if world > 1 and exchange == "nccl":  # round-1 path for A/B: the reference's own decomposition, no dense leg
            from skellysim_b200.distributed import reference_rank_ranges
            self.ranges = reference_rank_ranges(nfib, ns, nb, rank, world)
            with_dense = False
        else:
            self.ranges = capi.partition_query(g["n_nodes"], ns, nb, world, rank)
        f0, f1, s0, s1, b0, b1 = self.ranges
        self.f0, self.f1, self.s0, self.s1, self.b0, self.b1 = f0, f1, s0, s1, b0, b1
        self.n_fw, self.n_sw, self.n_bw = (f1 - f0) * n, s1 - s0, b1 - b0
        fl = skb.Flow(local_rank)
        fl.set_fibers(g["fib"], g["n_nodes"], g["lengths"])
        fl.set_periphery(g["shell"], g["shell_n"])
        fl.set_bodies(g["body"], g["body_n"], g["centers"])
        self.exchange = exchange
        if world > 1:
            fl.set_target_ranges(*self.ranges)
            if exchange == "peer":
                connect_group(fl, rank, world)
        self.fl = fl
        _log("geometry set")
        self.ops = Ops(g, f0, f1)
        fl.set_fiber_class(n, self.ops.D, self.ops.P)
        t0 = time.perf_counter()
        # (.base of the transposed views = the column-major storage the C ABI takes: no host-side reshuffle is timed)
        fl.set_fiber_operators(self.ops.A.base, self.ops.F.base, self.ops.xs, self.ops.lprev, self.ops.plus,
                               colmajor=True)
        self.set_operators_ms = 1e3 * (time.perf_counter() - t0)
        _log("fiber operators uploaded")
        self.dn = None
        self.M_rows = None
        if with_dense and ns:
            self.dn = skb.Dense(device_ids=[local_rank])
            self.M_rows = dense_rows(3 * self.n_sw, 3 * ns, 3 * s0)
            self.dn.set_matrix(skb.DENSE_STRESSLET_PLUS_COMPLEMENTARY, self.M_rows)
            _log("dense operator uploaded")
        # inputs: own slices, device resident + pinned host copies
        t = lambda a: torch.from_numpy(np.ascontiguousarray(a))
        self.inputs_full = [make_inputs(g, k) for k in range(n_inputs)]
        self.h_in, self.d_in = [], []
        for inp in self.inputs_full:
            own = dict(x=inp["x"][4 * f0 * n:4 * f1 * n], xs=inp["xs"][s0:s1], bd=inp["bd"], f=inp["ft"][:, :3],
                       t=inp["ft"][:, 3:], link=inp["link"][f0:f1])
            h = {k: t(v).pin_memory() for k, v in own.items()}
            self.h_in.append(h)
            self.d_in.append({k: v.to(self.dev) for k, v in h.items()})
        kw = dict(dtype=torch.float64, device=self.dev)
        self.d_res = torch.zeros(max(4 * self.n_fw, 1), **kw)
        self.d_outs = torch.zeros((max(self.n_sw, 1), 3), **kw)
        self.d_vb = torch.zeros((max(self.n_bw, 1), 3), **kw)
        self.h_res = torch.zeros(max(4 * self.n_fw, 1), dtype=torch.float64).pin_memory()
        self.h_outs = torch.zeros((max(self.n_sw, 1), 3), dtype=torch.float64).pin_memory()
        self.h_vb = torch.zeros((max(self.n_bw, 1), 3), dtype=torch.float64).pin_memory()
        self.d_e2e = {k: torch.zeros_like(v) for k, v in self.d_in[0].items()}
        if world > 1 and exchange == "nccl":
            from skellysim_b200.distributed import RankApplyMatvec
            self.nccl = RankApplyMatvec(fl, g["n_nodes"], ns, nb, g["n_bodies"], rank, world, device=self.dev)
        torch.cuda.synchronize()

    def p(self, t):
        return t.data_ptr() if t.numel() else 0

    def matvec_device(self, k, src=None):
        """One apply_matvec with operands in HBM (device-pointer C ABI)."""
        d = src or self.d_in[k % len(self.d_in)]
        st = self.torch.cuda.current_stream().cuda_stream
        self.fl.apply_matvec_device(self.dn, self.p(d["x"]), self.p(d["xs"]), self.p(d["bd"]), self.p(d["f"]),
                                    self.p(d["t"]), self.p(d["link"]), ETA, self.d_res.data_ptr(),
                                    self.d_outs.data_ptr(), self.d_vb.data_ptr(), st)

    def matvec_e2e(self, k):
        """The same from HOST buffers: H2D of the solution vector and D2H of the result inside."""
        h = self.h_in[k % len(self.h_in)]
        if self.world == 1:  # the reference-facing C ABI call with host pointers
            ft = np.concatenate([h["f"].numpy(), h["t"].numpy()], axis=1)
            self.fl.apply_matvec(h["x"].numpy(), h["xs"].numpy(), h["bd"].numpy(), ft, ETA,
                                 fiber_link_conditions=h["link"].numpy(), dense=self.dn,
                                 out=(self.h_res.numpy()[:4 * self.nf], self.h_outs.numpy()[:self.ns],
                                      self.h_vb.numpy()[:self.nb]))
            return
        for key, v in h.items():
            self.d_e2e[key].copy_(v, non_blocking=True)
        self.matvec_device(k, src=self.d_e2e)
        self.h_res.copy_(self.d_res, non_blocking=True)
        self.h_outs.copy_(self.d_outs, non_blocking=True)
        self.h_vb.copy_(self.d_vb, non_blocking=True)

    def io_bytes(self):
        h = self.h_in[0]
        return (int(sum(v.numel() for v in h.values()) * 8),
                int((4 * self.n_fw + 3 * self.n_sw + 3 * self.n_bw) * 8))

    def close(self):
        if self.dn is not None:
            self.dn.close()
        self.fl.close()


def accuracy_gate(rs: RankSystem, n_fibers_checked=48, n_shell_checked=1536, n_body_checked=400):
    """GPU result of matvec 0 against the CPU oracle on a sample of rows: every node of `n_fibers_checked` fibers (so
    that fc.matvec's res_fibers can be checked too), shell rows, body rows (>= 4096 target rows in total at C3)."""
    g, n = rs.g, rs.g["n"]
    import oracle as orc  # checker only
    rng = np.random.default_rng(3)
    rs.matvec_device(0)
    rs.torch.cuda.synchronize()
    res = rs.d_res.cpu().numpy()[:4 * rs.n_fw]
    outs = rs.d_outs.cpu().numpy()[:rs.n_sw]
    vb = rs.d_vb.cpu().numpy()[:rs.n_bw]
    fib_sel = np.sort(rng.choice(np.arange(rs.f0, rs.f1), size=min(n_fibers_checked, rs.f1 - rs.f0), replace=False))
    sh_sel = np.sort(rng.choice(np.arange(rs.s0, rs.s1), size=min(n_shell_checked, rs.n_sw), replace=False)) \
        if rs.n_sw else np.zeros(0, dtype=int)
    bo_sel = np.arange(rs.b0, rs.b1)[:n_body_checked]
    rows = np.concatenate([(f * n + np.arange(n)) for f in fib_sel] + [rs.nf + sh_sel, rs.nf + rs.ns + bo_sel]).astype(int)
    F_all = rs.ops.F if rs.world == 1 else Ops.F_range(g, 0, g["n_fibers"])
    errs = {}
    if True:
        cpu = CpuMatvec(g, rs.ops, None, F_all=F_all)
        ref = cpu.apply(rs.inputs_full[0], rows=rows, fibers=fib_sel)
        got_res = np.stack([res[4 * n * (f - rs.f0):4 * n * (f - rs.f0 + 1)] for f in fib_sel])
        errs["res_fibers"] = float(np.abs(got_res - ref["res_fib"]).max() / np.abs(ref["res_fib"]).max())
        v_ref = ref["v_rows"]
        k0 = len(fib_sel) * n
        if len(sh_sel):
            v_sh = v_ref[k0:k0 + len(sh_sel)]
            if rs.dn is not None:
                xs_full = rs.inputs_full[0]["xs"].reshape(-1)
                for i, r in enumerate(sh_sel):
                    v_sh[i] += rs.M_rows[3 * (r - rs.s0):3 * (r - rs.s0) + 3] @ xs_full
            errs["shell_rows"] = float(np.abs(outs[sh_sel - rs.s0] - v_sh).max() / np.abs(v_sh).max())
        if len(bo_sel):
            v_bo = v_ref[k0 + len(sh_sel):]
            errs["body_rows"] = float(np.abs(vb[bo_sel - rs.b0] - v_bo).max() / np.abs(v_bo).max())
    return {"max_rel_err_vs_oracle": max(errs.values()) if errs else None, "by_block": errs,
            "targets_checked": int(rows.shape[0]), "fibers_checked": int(len(fib_sel)), "gate": 1e-12}


def dump_outputs(rs: RankSystem, out_dir: str):
    """--dump-outputs: the result of the last matvec of the timed device path, i.e. what skb_flow_apply_matvec_device
    hands its caller (res_fibers (4 N_f,), res_shell (N_s, 3) -- v_shell without the dense operator -- and v_bodies
    (N_b, 3)), assembled over the ranks, written by rank 0 as out_dir/<name>.npy in float64.  Geometry, operators and
    inputs are seeded, so two builds can be compared file by file.  Whole arrays: the largest workload (c4) writes 32 MB.
    Rows no rank owns would stay NaN."""
    rs.torch.cuda.synchronize()
    parts = [(rs.ranges, rs.d_res.cpu().numpy()[:4 * rs.n_fw], rs.d_outs.cpu().numpy()[:rs.n_sw],
              rs.d_vb.cpu().numpy()[:rs.n_bw])]
    if rs.world > 1:
        import torch.distributed as dist
        mine, parts = parts[0], [None] * rs.world
        dist.all_gather_object(parts, mine)
    if rs.rank != 0:
        return
    n = rs.g["n"]
    res, shell, body = np.full(4 * rs.nf, np.nan), np.full((rs.ns, 3), np.nan), np.full((rs.nb, 3), np.nan)
    for (f0, f1, s0, s1, b0, b1), r, s, b in parts:
        res[4 * n * f0:4 * n * f1], shell[s0:s1], body[b0:b1] = r, s, b
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "res_fibers.npy"), res)
    np.save(os.path.join(out_dir, "res_shell.npy" if rs.dn is not None else "v_shell.npy"), shell)
    np.save(os.path.join(out_dir, "v_bodies.npy"), body)


# ------------------------------------------------------------------------------------------------
# extra legs (N = 1)
# ------------------------------------------------------------------------------------------------
def stokeslet_call_leg(torch, skb, g, dev, local_rank, reps=10):
    """The C3 Stokeslet evaluator call alone (fiber nodes -> all nodes), kernel-only and through skb_eval with host
    buffers: the 'Stokeslet pair-interactions/s' half of the metric."""
    r_src = g["fib"]
    r_trg = np.concatenate([g["fib"], g["shell"], g["body"]])
    f = np.random.default_rng(7).uniform(-1, 1, r_src.shape)
    with skb.Context(1, device_ids=[local_rank]) as ctx:
        ctx.set_targets(r_trg)
        ctx.set_sources(skb.KERNEL_STOKESLET, r_src)
        u = np.empty((r_trg.shape[0], 3))
        ctx.eval(skb.KERNEL_STOKESLET, f, out=u)
        ks, ws = [], []
        for _ in range(reps):
            t0 = time.perf_counter()
            ctx.eval(skb.KERNEL_STOKESLET, f, out=u)
            ws.append(time.perf_counter() - t0)
            ks.append(ctx.stats()["kernel_ms"])
        sym_ms, sym_pairs = ctx.last_sym_kernel()
    pairs = float(r_src.shape[0]) * r_trg.shape[0]
    k = float(np.median(ks))
    return {"n_src": int(r_src.shape[0]), "n_trg": int(r_trg.shape[0]), "kernel_ms": k,
            "pairs_per_s_kernel": pairs / (k * 1e-3), "e2e_ms": 1e3 * float(np.median(ws)),
            "pairs_per_s_e2e": pairs / float(np.median(ws)),
            "frac_of_nominal_fp64": SL_FLOP_PER_PAIR * pairs / (k * 1e-3) / 1e12 / NOMINAL_FP64_TFLOPS,
            "sym_kernel_ms": sym_ms, "sym_kernel_pairs_per_s": (sym_pairs / (sym_ms * 1e-3)) if sym_ms else None}


def ref_kernel_only_ms(path=None):
    """Median duration (ms) of the reference's tiled_driver kernel in the committed ncu launch list, or None."""
    import csv
    path = path or os.path.join(os.path.dirname(os.path.abspath(__file__)), "profiles", "r2_ref_gpu_kernel.csv")
    try:
        ns = [float(r[-1].replace(",", "")) for r in csv.reader(open(path))
              if len(r) > 5 and r[0].isdigit() and "tiled_driver" in r[4] and r[-2] == "ns"]
    except (OSError, ValueError):
        return None
    return float(np.median(ns)) * 1e-6 if ns else None


def ref_gpu_leg(g, reps=5):
    """The reference's own CUDA path (src/core/kernels.cu compiled unmodified for sm_100 into oracle/_ref) on the same
    GPU, same C3 Stokeslet call: end to end (its cudaMalloc + copies + kernel + free, kernels.cu:148-178)."""
    import oracle as orc
    if not orc.refgpu_available():
        return {"unavailable": "oracle/_ref/libskelly_ref_kernels_cu.so not built"}
    r_src = g["fib"]
    r_trg = np.concatenate([g["fib"], g["shell"], g["body"]])
    f = np.random.default_rng(7).uniform(-1, 1, r_src.shape)
    orc.ref_stokeslet_direct_gpu_impl(r_src, f, r_trg)
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        orc.ref_stokeslet_direct_gpu_impl(r_src, f, r_trg)
        ts.append(time.perf_counter() - t0)
    pairs = float(r_src.shape[0]) * r_trg.shape[0]
    out = {"what": "kernels::stokeslet_direct_gpu_impl of the reference (kernels.cu, nvcc -arch=sm_100, unmodified)",
           "e2e_ms": 1e3 * float(np.median(ts)), "pairs_per_s_e2e": pairs / float(np.median(ts)),
           "note": "wall clock of the reference's entry point: 4 cudaMalloc + 3 H2D + kernel + D2H + 4 cudaFree"}
    # its kernel alone cannot be timed from outside the entry point; the committed ncu launch list of this very leg
    # (profiles/r2_ref_gpu_kernel.csv, `ncu --metrics gpu__time_duration.sum -k regex:driver`) is quoted instead
    k_ms = ref_kernel_only_ms() if g["workload"] == "c3" else None
    if k_ms:
        out["kernel_only_ms_ncu"] = k_ms
        out["pairs_per_s_kernel_ncu"] = pairs / (k_ms * 1e-3)
        out["kernel_only_source"] = "profiles/r2_ref_gpu_kernel.csv (recorded on a B200 of this pool, not in this run)"
    return out


def solve_leg(torch, skb, rs: RankSystem, k_iter=30):
    """K GMRES-shaped iterations (P_inv_hydro::apply then A_fiber_hydro::apply, solver_hydro.cpp:23-48), everything
    device resident; per-iteration time, launches and PCIe bytes."""
    from skellysim_b200 import capi
    from skellysim_b200.solver_hydro import HydroOperator, iterate
    g = rs.g
    ns = rs.ns
    # explicit inverses of the fiber blocks and M_inv: stand-ins of the right shapes (timing and launch counts)
    rs.fl.set_fiber_preconditioner(rs.ops.A)
    if rs.dn is not None:
        rs.dn.set_matrix(skb.DENSE_M_INV, dense_rows(3 * ns, 3 * ns, 0, seed=11))
    op = HydroOperator(rs.fl, rs.dn, rs.nf, ns, rs.nb, ETA, rs.dev)
    d = rs.d_in[0]
    x_f, x_s = d["x"].clone(), d["xs"].clone()
    iterate(op, x_f, x_s, d["bd"], d["f"], d["t"], d["link"], 3)
    torch.cuda.synchronize()
    n0 = capi.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    iterate(op, x_f, x_s, d["bd"], d["f"], d["t"], d["link"], k_iter)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    launches = capi.launch_count() - n0
    return {"iterations": k_iter, "ms_per_iteration": ms / k_iter, "launches_per_iteration": launches / k_iter,
            "pcie_bytes_per_iteration": 0,
            "note": "fiber + periphery blocks of P^-1 and A on the device; x never leaves HBM; the body block "
                    f"({rs.nb} nodes) is host glue in the reference too and is passed through as device tensors here",
            "hbm_bytes_per_iteration": int(2 * rs.ops.A.nbytes + rs.ops.F.nbytes + (2 * (3 * ns) ** 2 * 8 if rs.dn else 0))}


def dense_leg(skb, hbm_peak_gbs, local_rank, n_nodes=6000, reps=10):
    n = 3 * n_nodes
    A = dense_rows(n, n, 0)
    rng = np.random.default_rng(4)
    x, v = rng.random(n), rng.random(n)
    with skb.Dense(device_ids=[local_rank]) as dn:
        dn.set_matrix(skb.DENSE_STRESSLET_PLUS_COMPLEMENTARY, A)
        y = dn.apply(skb.DENSE_STRESSLET_PLUS_COMPLEMENTARY, x, v)
        ks, ts = [], []
        for _ in range(reps):
            t0 = time.perf_counter()
            y = dn.apply(skb.DENSE_STRESSLET_PLUS_COMPLEMENTARY, x, v)
            ts.append(1e3 * (time.perf_counter() - t0))
            ks.append(dn.stats()["kernel_ms"])
        bytes_ = dn.stats()["bytes"]
        # the same product with the background row streamer, alone on the GPU (its job is to run BESIDE the pair kernels,
        # see the `overlap` leg; alone, one small CTA per SM does not reach the copy peak)
        import torch
        dev = torch.device("cuda", local_rank)
        d_x = torch.from_numpy(x).to(dev)
        d_y = torch.zeros(n, dtype=torch.float64, device=dev)
        st = torch.cuda.current_stream(dev).cuda_stream
        bs = []
        for _ in range(reps + 2):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            dn.apply_background_device(skb.DENSE_STRESSLET_PLUS_COMPLEMENTARY, d_x.data_ptr(), d_y.data_ptr(), st)
            e1.record()
            torch.cuda.synchronize()
            bs.append(e0.elapsed_time(e1))
        kb = float(np.median(bs[2:]))
        yb = d_y.cpu().numpy()
    rows = np.random.default_rng(0).choice(n, 32, replace=False)
    ref = A[rows] @ x + v[rows]
    err = float(np.max(np.abs(y[rows] - ref) / (np.abs(A[rows]) @ np.abs(x) + np.abs(v[rows]))))
    k = float(np.median(ks))
    return {"workload": f"Periphery::matvec dense operator, {n_nodes} nodes: {n} x {n} FP64 row-major GEMV (+v)",
            "kernel_ms": k, "e2e_ms": float(np.median(ts)), "bytes": int(bytes_),
            "roofline": {"bound": "hbm", "achieved": bytes_ / (k * 1e-3) / 1e9, "peak": hbm_peak_gbs, "unit": "GB/s",
                         "frac": bytes_ / (k * 1e-3) / 1e9 / hbm_peak_gbs},
            "max_backward_err": err,
            "background_streamer": {"kernel_ms_alone": kb, "gbs_alone": bytes_ / (kb * 1e-3) / 1e9,
                                    "max_backward_err": float(np.max(np.abs(yb[rows] - A[rows] @ x) /
                                                                     (np.abs(A[rows]) @ np.abs(x))))}}


def fiber_ops_leg(rs: RankSystem, hbm_peak_gbs, reps=10):
    """The per-fiber operator kernels alone (row N2): apply_fiber_force and fc.matvec over resident operators."""
    torch, fl = rs.torch, rs.fl
    st = torch.cuda.current_stream().cuda_stream
    d = rs.d_in[0]
    fw = torch.zeros((max(rs.n_fw, 1), 3), dtype=torch.float64, device=rs.dev)
    v = torch.randn((max(rs.n_fw, 1), 3), dtype=torch.float64, device=rs.dev)
    ev = lambda: torch.cuda.Event(enable_timing=True)
    kf, km = [], []
    for _ in range(reps + 2):
        a, b, c = ev(), ev(), ev()
        a.record()
        fl.apply_fiber_force_device(d["x"].data_ptr(), fw.data_ptr(), st)
        b.record()
        fl.fiber_matvec_device(d["x"].data_ptr(), v.data_ptr(), d["link"].data_ptr(), rs.d_res.data_ptr(), st)
        c.record()
        torch.cuda.synchronize()
        kf.append(a.elapsed_time(b))
        km.append(b.elapsed_time(c))
    kf, km = float(np.median(kf[2:])), float(np.median(km[2:]))
    mat_bytes = rs.ops.A.nbytes + rs.ops.F.nbytes
    gbs = mat_bytes / ((kf + km) * 1e-3) / 1e9
    return {"fiber_force_ms": kf, "fiber_matvec_ms": km, "operator_bytes": int(mat_bytes),
            "set_operators_ms": rs.set_operators_ms,
            "roofline": {"bound": "hbm", "achieved": gbs, "peak": hbm_peak_gbs, "unit": "GB/s",
                         "frac": gbs / hbm_peak_gbs}}


def overlap_leg(rs: RankSystem, reps=10):
    """A/B of skb_flow_set_overlap on the headline workload: the periphery's dense operator beside the pair kernels
    (background row streamer on a side stream, csrc/stream_kernels.cuh) against one GEMV kernel at the end of the stream."""
    torch = rs.torch

    def run():
        for k in range(3):
            rs.matvec_device(k)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for k in range(reps):
            rs.matvec_device(k)
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / reps

    on = run()
    rs.fl.set_overlap(False)
    off = run()
    rs.fl.set_overlap(True)
    return {"ms_per_matvec_overlap_on": on, "ms_per_matvec_overlap_off": off,
            "what": "stresslet_plus_complementary * x_shell (periphery.cpp:38-47, HBM-bound) streamed by a 3-warp CTA per "
                    "SM beside pair_sym_kernel (FP64-bound) vs. run after the pair kernels; back-to-back matvecs, no L2 "
                    "flush"}


def inprocess_leg(skb, n_devices: int):
    """ONE process driving all GPUs of the box (skb_mflow): the shape the reference's one-rank rule for direct
    evaluators admits.  A C2-sized system through skb_mflow_apply_matvec against the CPU oracle on sampled rows."""
    g = make_system("c2", 1, seed=5, sizes=(1000, 4000, 400, 1, "weak"))
    ops = Ops(g, 0, g["n_fibers"])
    ns = g["shell"].shape[0]
    M = dense_rows(3 * ns, 3 * ns, 0)
    inp = make_inputs(g, 0)
    out = {"n_devices": n_devices}
    with skb.MultiFlow(list(range(n_devices))) as mf:
        mf.set_fibers(g["fib"], g["n_nodes"], g["lengths"])
        mf.set_periphery(g["shell"], g["shell_n"])
        mf.set_bodies(g["body"], g["body_n"], g["centers"])
        mf.set_fiber_class(g["n"], ops.D, ops.P)
        mf.set_fiber_operators(ops.A.base, ops.F.base, ops.xs, ops.lprev, ops.plus, colmajor=True)
        mf.set_dense(skb.DENSE_STRESSLET_PLUS_COMPLEMENTARY, M)
        res, outs, vb = mf.apply_matvec(inp["x"], inp["xs"], inp["bd"], inp["ft"], ETA, inp["link"])
        ts = []
        for _ in range(5):
            t0 = time.perf_counter()
            mf.apply_matvec(inp["x"], inp["xs"], inp["bd"], inp["ft"], ETA, inp["link"])
            ts.append(1e3 * (time.perf_counter() - t0))
        out["device_ms"] = mf.stats()["device_ms"]
    out["e2e_ms"] = float(np.median(ts))
    cpu = CpuMatvec(g, ops, M)
    ref = cpu.apply(inp)
    out["max_rel_err_res_fibers"] = float(np.abs(res.reshape(-1, 4 * g["n"]) - ref["res_fib"]).max()
                                          / np.abs(ref["res_fib"]).max())
    out["max_rel_err_res_shell"] = float(np.abs(outs - ref["out_shell"]).max() / np.abs(ref["out_shell"]).max())
    out["max_rel_err_v_bodies"] = float(np.abs(vb - ref["v_body"]).max() / np.abs(ref["v_body"]).max())
    out["n_nodes"] = int(g["fib"].shape[0] + ns + g["body"].shape[0])
    return out


# ------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="c3", choices=["c2", "c3", "c4"])
    ap.add_argument("--exchange", default="peer", choices=["peer", "nccl"], help="N > 1: peer-memory kernels / NCCL (A/B)")
    ap.add_argument("--inner", type=int, default=0, help="matvecs per timed step (default 8; 1 for c4)")
    ap.add_argument("--no-extras", action="store_true", help="headline only")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-dense-leg", action="store_true")
    ap.add_argument("--no-inprocess", action="store_true")
    ap.add_argument("--no-strong", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the last step's matvec result as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be >= 1")
    if args.dump_outputs and args.exchange == "nccl":
        ap.error("--dump-outputs: the --exchange nccl A/B path keeps no result buffers")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        return run_reference_arm(args, rank)
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("--gpus N > 1 must be launched with torch.distributed.run --nproc-per-node N")
        args.gpus = world
    args.warmup = max(args.warmup, 3)
    inner = args.inner or (1 if args.workload == "c4" else INNER)

    _log("importing torch")
    import torch
    import torch.distributed as dist
    import skellysim_b200 as skb
    from skellysim_b200 import capi

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    g = make_system(args.workload, world)
    rs = RankSystem(torch, skb, g, rank, world, local_rank, exchange=args.exchange)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)  # > 126 MB L2
    _log("system resident")

    def step_device(s):
        if world > 1 and args.exchange == "nccl":
            d = rs.d_in[s % 2]
            for i in range(inner):
                rs.nccl.apply(d["x"], d["xs"], d["bd"], d["f"], d["t"], d["link"], ETA)
            return
        for i in range(inner):
            rs.matvec_device(s * inner + i)

    def step_e2e(s):
        if world > 1 and args.exchange == "nccl":  # A/B leg: device path only
            return step_device(s)
        for i in range(inner):
            rs.matvec_e2e(s * inner + i)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    sym_samples = []

    def timed(fn, steps, sample_sym=False):
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        barrier()
        wall0 = time.perf_counter()
        for s, (a, b) in enumerate(evs):
            flush.zero_()  # evict L2 between timed steps (not timed)
            a.record()
            fn(s)
            b.record()
            if sample_sym and s < 6:  # the dominant kernel's live duration inside the step (needs the step finished)
                b.synchronize()
                sym_samples.append(rs.fl.last_sym_kernel())
        barrier()
        wall = time.perf_counter() - wall0
        tot_ms = sum(a.elapsed_time(b) for a, b in evs)
        t = torch.tensor([tot_ms], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item()), wall

    # ONE joint warm-up of both paths, then the accuracy gate, then the two timed passes
    for s in range(args.warmup):
        step_device(s)
    for s in range(args.warmup):
        step_e2e(s)
    torch.cuda.synchronize()
    acc = accuracy_gate(rs) if args.exchange == "peer" else {"max_rel_err_vs_oracle": None}
    if world > 1:
        a = torch.tensor([acc["max_rel_err_vs_oracle"] or 0.0], dtype=torch.float64, device=dev)
        dist.all_reduce(a, op=dist.ReduceOp.MAX)
        acc["max_rel_err_vs_oracle_all_ranks"] = float(a.item())
    _log("warm-up + accuracy gate done")

    with ClockSampler(local_rank) as clk:
        n0 = capi.launch_count()
        tot_ms, wall = timed(step_device, args.steps, sample_sym=True)
        launches = capi.launch_count() - n0
    if args.dump_outputs:  # before the e2e pass, which reuses the device buffers
        dump_outputs(rs, args.dump_outputs)
    e2e_ms, _ = timed(step_e2e, args.steps)
    missing = rs.fl.group_error() if world > 1 and args.exchange == "peer" else -1

    pairs = pairs_per_matvec(g)
    n_matvecs = args.steps * inner
    ms_per_step = tot_ms / args.steps
    value = pairs * n_matvecs / (tot_ms * 1e-3)
    e2e_val = pairs * n_matvecs / (e2e_ms * 1e-3)
    launches_all = launches
    if world > 1:
        t = torch.tensor([launches], dtype=torch.int64, device=dev)
        dist.all_reduce(t)
        launches_all = int(t.item())
    h2d, d2h = rs.io_bytes()
    if world > 1:
        t = torch.tensor([h2d, d2h], dtype=torch.int64, device=dev)
        dist.all_reduce(t)
        h2d, d2h = int(t[0].item()), int(t[1].item())

    out = None
    if rank == 0:
        peaks_file = os.path.join(ROOT, "MEASURED_PEAKS.json")
        hbm_peak, hbm_src = 6650.0, "fallback (B200_PROFILING.md)"
        if os.path.exists(peaks_file):
            hbm_peak = float(json.load(open(peaks_file))["hbm_gbs"])
            hbm_src = "measured (MEASURED_PEAKS.json)"
        sym = [(ms, p) for ms, p in sym_samples if ms > 0]
        sym_ms = float(np.mean([m for m, _ in sym])) if sym else None
        sym_pairs = float(sym[0][1]) if sym else 0.0
        achieved = SL_FLOP_PER_PAIR * sym_pairs / (sym_ms * 1e-3) / 1e12 if sym_ms else None
        with skb.Context(1, device_ids=[local_rank]) as c_probe:
            probe = c_probe.measure_fp64_peak() / 1e12
        nf = g["fib"].shape[0]
        roofline = {
            "bound": "fp64", "kernel": "pair_sym_kernel<T=8> (symmetric fiber-fiber block of the Stokeslet call)",
            "achieved": achieved, "peak": NOMINAL_FP64_TFLOPS, "unit": "TFLOP/s",
            "frac": achieved / NOMINAL_FP64_TFLOPS if achieved else None,
            "peak_source": "nominal: 148 SMs x 64 DFMA/clk x 2 x 1.965 GHz (MEASURED_PEAKS.json carries no FP64 figure)",
            "frac_of_ubench_2reg_dfma": achieved / UBENCH_FP64_TFLOPS if achieved else None,
            "frac_of_probe": achieved / probe if achieved else None, "probe_tflops": probe,
            "flop_per_pair": SL_FLOP_PER_PAIR, "kernel_ms": sym_ms, "pairs_per_launch": sym_pairs,
            "pairs_per_s": sym_pairs / (sym_ms * 1e-3) if sym_ms else None,
            "share_of_matvec": (sym_ms / (ms_per_step / inner)) if sym_ms else None,
            "measured": "CUDA events around the kernel on its launch stream inside the timed steps (first 6 steps)",
            "algorithmic": "28 flop x ordered pairs the launch covers (both directions of every block pair of this "
                           "rank's block rows), SURVEY.md 8d",
            "whole_matvec": {"tflops": flop_per_matvec(g) / world / (ms_per_step / inner * 1e-3) / 1e12,
                             "frac_of_nominal": flop_per_matvec(g) / world / (ms_per_step / inner * 1e-3) / 1e12
                             / NOMINAL_FP64_TFLOPS,
                             "note": "28 flop x SL pairs + 40 flop x DL pairs of one matvec / device time per matvec, "
                                     "per GPU"},
            "hbm": {"algorithmic_bytes_per_launch": 48.0 * nf + 48.0 * nf,
                    "achieved": (96.0 * nf) / (sym_ms * 1e-3) / 1e9 if sym_ms else None, "peak": hbm_peak,
                    "unit": "GB/s", "peak_source": hbm_src,
                    "note": "positions + strengths read once, forward partials written: compute bound by design"},
            "traffic": None,
        }
        prof = os.path.join(ROOT, "profiles", "traffic.json")
        if world == 1 and os.path.exists(prof):
            roofline["traffic"] = json.load(open(prof)).get(args.workload + "_r2")
        cfg = config_for(g, world)
        out = {
            "metric": "pair_interactions_per_s", "value": value, "unit": "pairs/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_per_step,
            "ms_per_matvec": ms_per_step / inner, "matvecs_per_step": inner, "higher_is_better": True,
            "scaling": g["scaling"], "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": cfg,
            "timing": {"l2": "flushed between timed steps (256 MiB memset, untimed)",
                       "method": "per-step CUDA events on the launch stream, summed; max over ranks; barrier + "
                                 "synchronize on both sides", "timed_region_s": tot_ms * 1e-3, "wall_s": wall,
                       "parallelism": (f"one rank per GPU x{world}: whole fibers / periphery rows / body rows per rank; "
                                       + ("strengths pushed and partial velocities pulled through peer memory by the "
                                          "library's kernels (no collective call per matvec)" if args.exchange == "peer"
                                          else "NCCL all-gather of strengths, plain kernel on own rows (round-1 path)"))
                       if world > 1 else "single GPU"},
            "e2e": {"value": e2e_val, "unit": "pairs/s", "ms_per_step": e2e_ms / args.steps,
                    "ms_per_matvec": e2e_ms / n_matvecs, "h2d_bytes_per_step": h2d * inner,
                    "d2h_bytes_per_step": d2h * inner,
                    "path": ("skb_flow_apply_matvec_dense (C ABI, host pointers, pinned buffers): H2D solution vector + "
                             "device matvec + D2H result inside every call" if world == 1 else
                             "pinned host slices -> H2D -> skb_flow_apply_matvec_device -> D2H, per rank")},
            "gpu_launches": launches_all, "launches_per_matvec_per_rank": launches_all / n_matvecs / world,
            "clocks": clk.summary(), "roofline": roofline, "accuracy": acc,
        }
        errs = []
        a_all = acc.get("max_rel_err_vs_oracle_all_ranks", acc.get("max_rel_err_vs_oracle"))
        if a_all is not None and not (a_all < 1e-12):
            errs.append(f"accuracy gate failed: {a_all}")
        if not (e2e_ms >= tot_ms * 0.999):
            errs.append(f"e2e ({e2e_ms:.3f} ms) below the device-timed region ({tot_ms:.3f} ms)")
        if missing >= 0:
            errs.append(f"group flag wait timed out (peer {missing})")
        if errs:
            out["error"] = "; ".join(errs)
    _log("headline done")

    # ---- extras -------------------------------------------------------------------------------------------
    if not args.no_extras and world == 1:
        import oracle as orc
        if not args.no_cpu_baseline:
            M_full = rs.M_rows
            cpu = CpuMatvec(g, rs.ops, M_full)
            val, calls, dt = cpu_timed(cpu, rs.inputs_full, 12.0 if args.workload != "c4" else 1.0)
            out["cpu_baseline"] = cpu_baseline_dict(cpu, val, calls, dt, orc)
            _log("cpu baseline done")
        out["solve"] = solve_leg(torch, skb, rs)
        out["fiber_operators"] = fiber_ops_leg(rs, hbm_peak)
        if rs.dn:
            out["overlap"] = overlap_leg(rs)
        _log("solve + fiber legs done")
    rs.close()
    del rs
    torch.cuda.empty_cache()
    if not args.no_extras and world == 1 and rank == 0:
        if args.workload != "c4":
            out["stokeslet_call"] = stokeslet_call_leg(torch, skb, g, dev, local_rank)
            out["ref_gpu_baseline"] = ref_gpu_leg(g)
        if not args.no_dense_leg:
            out["periphery_dense"] = dense_leg(skb, hbm_peak, local_rank)
        _log("extra legs done")
    if not args.no_extras and world > 1:
        if not args.no_strong and args.workload == "c3":
            # the metric's literal second half: the FIXED 1e5-node system strong-scaled over the ranks
            g1 = make_system("c3", 1)
            rs1 = RankSystem(torch, skb, g1, rank, world, local_rank, exchange=args.exchange)
            for k in range(4):
                rs1.matvec_device(k)
            barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for k in range(24):
                rs1.matvec_device(k)
            e1.record()
            barrier()
            t = torch.tensor([e0.elapsed_time(e1) / 24], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            acc1 = accuracy_gate(rs1, n_fibers_checked=16, n_shell_checked=256)
            a1 = torch.tensor([acc1["max_rel_err_vs_oracle"] or 0.0], dtype=torch.float64, device=dev)
            dist.all_reduce(a1, op=dist.ReduceOp.MAX)
            if rank == 0:
                out["matvec_strong_c3"] = {"n_nodes": 102400, "ms_per_matvec": float(t.item()), "scaling": "strong",
                                           "pairs_per_s": pairs_per_matvec(g1) / (float(t.item()) * 1e-3),
                                           "max_rel_err_vs_oracle_all_ranks": float(a1.item()),
                                           "timing": "24 back-to-back matvecs, CUDA events, max over ranks"}
            rs1.close()
            del rs1
            torch.cuda.empty_cache()
        barrier()
        if not args.no_inprocess and rank == 0:
            try:
                out["multi_device_inprocess"] = inprocess_leg(skb, world)
            except Exception as e:  # evidence leg: report, do not lose the headline
                out["multi_device_inprocess"] = {"error": str(e)[:300]}
        barrier()
    if rank == 0:
        print(json.dumps(out))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
