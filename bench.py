#!/usr/bin/env python
"""bench.py -- cost+gradient evaluations per second of the Bose-Hubbard optimal-control hot path.

Workload (BASELINE.json configs[1], "cfg2"): BH chain L=20, Npart=20, d=5 (local dimension 6), J=1,
T=2.0, tstep=0.01 (Nt=201 time points), GROUP basis with M=10 chopped sines on a linsigmoid ramp
U: 2.5 -> 50, Maxm=100, Cutoff=1e-8, gamma=1e-6.  One "step" = one cost+gradient evaluation with the
reference's protocol (main/TestRuntimes.cpp:57-58): getAnalyticGradient(c, new_control=true) followed by
getCost(c, new_control=false): forward sweep + backward sweep (400 Trotter steps), Nt MPO overlaps, the
fidelity overlaps and the basis projections.  Controls are synthetic (seeded); psi_init / psi_target are
the DMRG ground-state fixtures shipped in optimalcontrolmps_b200/data.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--hessian-nt NT] [--dump-outputs DIR]

N>1 (torchrun): every rank evaluates its own control on its own GPU (independent units, weak scaling);
the (cost, gradient) tuples are combined with one NCCL all-gather.  --impl reference times the CPU
restatement of the reference (oracle/, NumPy/OpenBLAS on all host cores) on a bounded sample of the same
workload; the reference's own ITensor build cannot be produced here (DESIGN.md).
"""
import argparse
import json
import os
os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")   # before CUDA starts: one hardware queue per chain stream (see the package __init__)
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np

CFG = dict(L=20, d=5, Npart=20, J=1.0, T=2.0, tstep=0.01, M=10, maxm=100, cutoff=1e-8, gamma=1e-6, U_i=2.5, U_f=50.0)
METRIC = "cost+gradient evals/s (BH N=20 chi=100)"
UNIT = "evals/s"


def nt():
    return int(CFG["T"] / CFG["tstep"] + 1)


_T0 = time.perf_counter()


def log(msg):
    """Progress on stderr (the JSON line on stdout is printed once, at the end)."""
    if int(os.environ.get("RANK", "0")) == 0:
        print(f"[bench {time.perf_counter() - _T0:7.1f}s] {msg}", file=sys.stderr, flush=True)


def config_dict():
    """The `config` object of the JSON line -- identical in both arms."""
    return {"workload": "cfg2: BH L=20 Npart=20 d=5 T=2.0 tstep=0.01 GROUP M=10 chi=100, one cost+gradient evaluation "
                        "(getAnalyticGradient(c,true) + getCost(c,false)) per step; N>1: one independent evaluation per GPU",
            **CFG, "Nt": nt(), "l2": "inputs larger than L2: the two slice stores are rewritten every evaluation (5.7 GB capacity)"}


HESS_M = 20      # cfg3: GROUP basis of the Hessian workload (tests/HessianTests.cpp:212 range for the coefficients)


def make_hessian_problem_host(seed=0):
    """cfg3 (BASELINE.json configs[2]): the cfg2 chain with a GROUP basis of M=20 chopped sines, c ~ U(-2,2)^20."""
    import optimalcontrolmps_b200 as oc
    rng = np.random.default_rng(3000 + seed)
    u0 = oc.SeedGenerator.linsigmoidSeed(CFG["U_i"], CFG["U_f"], nt(), np.random.default_rng(7))
    basis = oc.ControlBasisFactory.buildChoppedSineBasis(u0, CFG["tstep"], CFG["T"], HESS_M)
    c = np.array(oc.SeedGenerator.randomCoeffSeed(-2.0, 2.0, HESS_M, rng))
    for _ in range(40):
        u = np.array(basis.convertControl(list(c)))
        if u.min() >= 2.0 and u.max() <= 100.0:
            break
        c *= 0.8
    return basis, c


def make_problem_host(seed):
    """Basis and coefficient vector of the synthetic control for `seed` (pure host math, shared by both arms)."""
    import optimalcontrolmps_b200 as oc
    rng = np.random.default_rng(1000 + seed)
    u0 = oc.SeedGenerator.linsigmoidSeed(CFG["U_i"], CFG["U_f"], nt(), np.random.default_rng(7))
    basis = oc.ControlBasisFactory.buildChoppedSineBasis(u0, CFG["tstep"], CFG["T"], CFG["M"])
    c = np.array(oc.SeedGenerator.randomCoeffSeed(-4.0, 4.0, CFG["M"], rng))     # range of tests/GradientTests.cpp:199
    for _ in range(40):          # keep every u_i inside the optimiser's box [2, 100] (src/BH_nlp.cpp:55-56)
        u = np.array(basis.convertControl(list(c)))
        if u.min() >= 2.0 and u.max() <= 100.0:
            break
        c *= 0.8
    return basis, c, np.array(basis.convertControl(list(c)))


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self.stop_flag = index, [], False

    def run(self):
        q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
            "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}", "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([x.strip() for x in out.split(",")])
            except Exception:
                pass
            time.sleep(0.5)

    def summary(self):
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        sm = [float(r[0]) for r in self.rows if r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows for i in range(4) if len(r) > 2 + i and r[2 + i].lower().startswith("active")})
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "samples": len(self.rows)}


# ----------------------------------------------------------------------------------------------
# CPU arm: the oracle port, bounded sample
# ----------------------------------------------------------------------------------------------
def oracle_states():
    from oracle import bh_mps as ob
    from optimalcontrolmps_b200.states import ground_state
    gi = ground_state(CFG["L"], CFG["d"], CFG["Npart"], CFG["U_i"])
    gf = ground_state(CFG["L"], CFG["d"], CFG["Npart"], CFG["U_f"])
    conv = lambda h: ob.MPS(h.A, [np.asarray(x, dtype=np.int64) for x in h.q], 0, 2)
    return conv(gi), conv(gf)


def cpu_sample_from_states(psi_samples, xi_samples, u):
    """Times one forward Trotter step from each psi sample (slice index i -> i+1) and one backward step from each
    xi sample (i -> i-1) plus the MPO overlaps with the oracle; returns (seconds per eval extrapolated, details)."""
    from oracle import bh_mps as ob
    D = CFG["d"] + 1
    st = ob.BHStepper(CFG["L"], D, CFG["J"], CFG["tstep"], ob.TruncArgs(cutoff=CFG["cutoff"], maxm=CFG["maxm"]))
    N = nt()
    tf, tb, to = [], [], []
    for (i, psi) in psi_samples:
        p = psi.copy()
        t0 = time.perf_counter()
        st.step(p, u[i], u[i + 1], True)
        tf.append(time.perf_counter() - t0)
    for (i, xi) in xi_samples:
        p = xi.copy()
        t0 = time.perf_counter()
        st.step(p, u[i], u[i - 1], False)
        tb.append(time.perf_counter() - t0)
    for (i, psi), (j, xi) in zip(psi_samples, xi_samples):
        t0 = time.perf_counter()
        ob.overlap_K(xi, psi)
        to.append(time.perf_counter() - t0)
    per_eval = (N - 1) * float(np.mean(tf)) + (N - 1) * float(np.mean(tb)) + (N + 1) * float(np.mean(to))
    return per_eval, dict(fwd_step_s=float(np.mean(tf)), bwd_step_s=float(np.mean(tb)), overlap_s=float(np.mean(to)),
                          cpu_seconds=float(np.sum(tf) + np.sum(tb) + np.sum(to)))


def coarse_samples(u, npts, stride):
    """Representative mid-ramp states for the CPU-only arm: the oracle itself evolves psi forward / xi backward with
    `stride` Trotter steps merged into one (tstep*stride), and hands out the states at `npts` evenly spaced slices."""
    from oracle import bh_mps as ob
    D = CFG["d"] + 1
    psi, xi = oracle_states()
    N = nt()
    coarse = ob.BHStepper(CFG["L"], D, CFG["J"], CFG["tstep"] * stride, ob.TruncArgs(cutoff=CFG["cutoff"], maxm=CFG["maxm"]))
    want = sorted(set(int(round(x)) for x in np.linspace(stride, N - 1 - stride, npts)))
    want = [w - w % stride for w in want]
    ps, xs = [], []
    i = 0
    p = psi.copy()
    while i + stride <= N - 1:
        if i in want:
            ps.append((i, p.copy()))
        coarse.step(p, u[i], u[i + stride], True)
        i += stride
    j = N - 1
    x = xi.copy()
    wantb = [N - 1 - w for w in want]
    while j - stride >= 0:
        if j in wantb:
            xs.append((j, x.copy()))
        coarse.step(x, u[j], u[j - stride], False)
        j -= stride
    return ps, xs


def run_reference(args):
    """CPU arm: the oracle port of the reference path on this box's host cores (OpenBLAS uses all of them).
    Timed step 1 is one COMPLETE cost+gradient evaluation with the reference's protocol (getAnalyticGradient(c,true) then
    getCost(c,false), 400 Trotter steps + overlaps); further steps are bounded samples taken at 8 evenly spaced slices of
    that evaluation's own psi_t / xi_t (exact bond dimensions) and extrapolated, so that the run stays within minutes."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import bh_mps as ob, optimal_control as oo
    ncores = os.cpu_count() or 1
    basis_p, c, u = make_problem_host(max(args.seed, 0))
    psi_i, psi_f = oracle_states()
    D = CFG["d"] + 1
    N = nt()
    st = ob.BHStepper(CFG["L"], D, CFG["J"], CFG["tstep"], ob.TruncArgs(cutoff=CFG["cutoff"], maxm=CFG["maxm"]))
    u0 = list(basis_p._u0)
    basis = oo.ControlBasis(u0, list(basis_p._S), basis_p._f.tolist())
    ocp = oo.OptimalControl(psi_f, psi_i, st, basis=basis, gamma=CFG["gamma"])
    # warm-up: a few Trotter steps (BLAS thread pools, page faults); the CPU needs no more than that
    w = psi_i.copy()
    for k in range(max(1, min(args.warmup, 3))):
        st.step(w, u[k], u[k + 1], True)
    t0 = time.perf_counter()
    grad = ocp.getAnalyticGradient(list(c), True)
    cost = ocp.getCost(list(c), False)
    full = time.perf_counter() - t0
    vals = [full]
    det = {"full_eval_s": full}
    if args.steps > 1:
        idx = [int(round(x)) for x in np.linspace(4, N - 5, 8)]
        ps = [(i, ocp.psi_t[i]) for i in idx]
        xs = [(i, ocp.xi_t[i]) for i in idx]
        for k in range(args.steps - 1):
            per_eval, d2 = cpu_sample_from_states(ps, xs, u)
            vals.append(per_eval)
            det.update(d2)
    per_eval = float(np.mean(vals))
    value = 1.0 / per_eval
    sample = (f"oracle port (NumPy/OpenBLAS, {ncores} threads): step 1 = one complete cost+gradient evaluation ({full:.1f} s); "
              f"steps 2..K = 1 forward + 1 backward Trotter step + 1 MPO overlap from each of 8 evenly spaced slices of that "
              f"evaluation, extrapolated to 2*(Nt-1) steps + Nt+1 overlaps")
    note = ("NumPy/OpenBLAS port of the reference's algorithm (the ITensor build cannot be produced here): interpreter- and "
            "small-LAPACK-bound, not core-bound -- `cores` is the host's core count, the BLAS thread pool is nominal; a "
            "block-sparse C++ ITensor build would be faster than this port.  One CPU process: compare with the GPU arm at N=1 only.")
    # Hessian on the CPU, estimated (a full one is ~20 000 Trotter steps): row steps at the mean forward-step time of this run
    hess_est = None
    if "fwd_step_s" in det:
        hess_est = (N - 2) * (N - 1) / 2.0 * det["fwd_step_s"] + 2 * (N - 1) * det["fwd_step_s"]
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": 1, "n_gpus_requested": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": per_eval * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "complex128 (f64)", "data": "synthetic",
            "config": config_dict(),
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": ncores, "kind": "port", "sample": sample, "note": note,
                             "hessian_wall_s_estimate": hess_est, **det},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0,
            "result": {"cost": float(cost), "grad_norm": float(np.linalg.norm(grad)),
                       "max_bond_dim": int(max(max(p.bond_dims()) for p in ocp.psi_t))}}
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------------------------
# GPU arm
# ----------------------------------------------------------------------------------------------
def fp64_peak_tflops(torch, dev):
    """Measured FP64 GEMM peak of this GPU (cuBLAS DGEMM 4096^3, best of 5) -- the roofline denominator
    (MEASURED_PEAKS.json has no FP64 figure, SURVEY.md 8d)."""
    n = 4096
    a = torch.randn(n, n, dtype=torch.float64, device=dev)
    b = torch.randn(n, n, dtype=torch.float64, device=dev)
    torch.matmul(a, b)
    torch.cuda.synchronize()
    best = 1e9
    for _ in range(5):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        torch.matmul(a, b)
        e1.record()
        torch.cuda.synchronize()
        best = min(best, e0.elapsed_time(e1))
    del a, b
    torch.cuda.empty_cache()
    return 2.0 * n ** 3 / (best * 1e-3) / 1e12


def run_ours(args):
    import torch
    import torch.distributed as dist
    import optimalcontrolmps_b200 as oc
    from optimalcontrolmps_b200.states import ground_state
    from optimalcontrolmps_b200 import distributed as ocd

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the GPU arm has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    ctx = oc.Context.default(local_rank)
    lib = ctx.lib
    L, d = CFG["L"], CFG["d"]
    st = oc.BH_tDMRG(oc.BoseHubbard(L, d), CFG["J"], CFG["tstep"], oc.Args("Cutoff=", CFG["cutoff"], "Maxm=", CFG["maxm"]), ctx=ctx)
    psi_i = ground_state(L, d, CFG["Npart"], CFG["U_i"])
    psi_f = ground_state(L, d, CFG["Npart"], CFG["U_f"])
    # N>1: every rank evaluates one control on its own GPU (independent replicas; a single evaluation does not shard).
    # By default all ranks use the same synthetic control so that the per-GPU work is identical (weak scaling);
    # --distinct-seeds gives every rank its own control (evaluation times then differ by up to ~30 % between seeds).
    basis, c, u = make_problem_host(rank if args.distinct_seeds else max(args.seed, 0))
    ocp = oc.OptimalControl(psi_f, psi_i, st, basis, CFG["gamma"])
    ocp.setThreadCount(2)                          # psi and xi sweeps on two streams (reference: 2 threads)
    N, M = nt(), CFG["M"]

    def one_eval():
        g = ocp.getAnalyticGradient(list(c), True)         # host control in, host gradient out
        cost = ocp.getCost(list(c), False)
        return cost, g

    log("cfg2: warm-up evaluations")
    for _ in range(args.warmup):
        one_eval()
    log("cfg2: timed evaluations")
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    l0 = lib.ocmps_launch_count()
    import ctypes
    t0 = time.perf_counter()
    lib.ocmps_timer_start(ctx.h)                  # CUDA events on the library's own stream (torch's stream sees none of this work)
    res = None
    for _ in range(args.steps):
        res = one_eval()
    dev_ms_c = ctypes.c_double()
    lib.ocmps_timer_stop(ctx.h, ctypes.byref(dev_ms_c))
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    wall = time.perf_counter() - t0
    dev_ms = dev_ms_c.value
    launches = lib.ocmps_launch_count() - l0
    sampler.stop_flag = True
    if rank == 0:
        sampler.join(timeout=2)
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, ocp, list(c), *res)
    # max over ranks of the device-timed region and of the end-to-end wall clock
    tt = torch.tensor([dev_ms * 1e-3, wall], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        # one all-gather of the (cost, gradient) tuples -- the only collective of the batched-controls path
        mine = np.concatenate([[res[0]], res[1]])
        allres = ocd.allgather_array(mine, dev)
    else:
        allres = [np.concatenate([[res[0]], res[1]])]
    t_dev, t_wall = float(tt[0]), float(tt[1])
    value = world * args.steps / t_dev
    e2e = world * args.steps / t_wall

    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": t_dev / args.steps * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "complex128 (f64)", "data": "synthetic",
            "config": config_dict(),
            "timing": "value: CUDA events recorded on the library's own stream around the timed region (every C-ABI call is synchronous, so "
                      "the events bracket all device work of the evaluations); e2e: host wall clock around the same calls made through "
                      "the public API with host control / gradient buffers",
            "e2e": {"value": e2e, "unit": UNIT, "h2d_bytes_per_step": int(8 * M + 8 * N), "d2h_bytes_per_step": int(8 * (1 + M) + 16 * 2 * N)},
            "gpu_launches": int(launches), "clocks": sampler.summary(),
            "result": {"cost": float(allres[0][0]), "grad_norm": float(np.linalg.norm(allres[0][1:])),
                       "max_bond_dim": int(ocp.psi_t.bond_dims().max())}}

    if rank == 0:
        # ---- roofline of the dominant kernel (block SVD), event-timed on its own streams in one extra eval ----
        log("cfg2: roofline evaluation (block-SVD kernels event-timed)")
        lib.ocmps_profile_enable(1)
        one_eval()
        out4 = np.zeros(4)
        lib.ocmps_profile_read(out4.ctypes.data_as(__import__("ctypes").POINTER(__import__("ctypes").c_double)))
        lib.ocmps_profile_enable(0)
        peak = fp64_peak_tflops(torch, dev)
        ms_tot, nl, fl_blk, fl_dense = out4
        traffic = None
        tpath = os.path.join(ROOT, "profiles", "roofline_traffic.json")
        if os.path.exists(tpath):
            try:
                traffic = json.load(open(tpath)).get("dram_bytes_per_launch")
            except Exception:
                traffic = None
        ach = fl_blk / (ms_tot * 1e-3) / 1e12 if ms_tot > 0 else 0.0
        line["roofline"] = {"kernel": "jacobi_blocks_kernel + jacobi_rot_kernel (pivoted QR + block Jacobi SVD of every charge block)",
                            "bound": "latency",
                            "bound_note": "FP64 DFMA kernels (no tensor-core instruction) bound by instruction issue and dependent chains of the "
                                          "sequential Householder steps / rotation rounds on one SM per charge block; the FP64 GEMM peak is the "
                                          "denominator SURVEY.md 8d asks for, not a bound these kernels can approach",
                            "achieved": ach, "peak": peak, "unit": "TFLOP/s", "frac": ach / peak if peak else None,
                            "traffic": traffic, "launches": int(nl), "avg_launch_us": ms_tot * 1e3 / max(nl, 1),
                            "share_of_two_stream_time": ms_tot / (2.0 * t_dev / args.steps * 1e3),
                            "algorithmic_flops": "block-summed F_gram+F_evd = sum_q 8 n_q^2 m_q + 56/3 n_q^3 (SURVEY.md 8d)",
                            "achieved_dense_formula": fl_dense / (ms_tot * 1e-3) / 1e12 if ms_tot > 0 else 0.0,
                            "peak_source": "measured in this run: cuBLAS DGEMM 4096^3 burst (MEASURED_PEAKS.json has no FP64 figure)"}
        if world == 1 and not args.no_cpu_baseline:
            # ---- CPU baseline: the oracle port on this box's host cores, bounded sample taken at real slices ----
            log("cfg2: CPU baseline sample")
            from oracle import bh_mps as ob
            conv = lambda h: ob.MPS(h.A, [np.asarray(x, dtype=np.int64) for x in h.q], 0, 2)
            idx = [int(round(x)) for x in np.linspace(4, N - 5, 8)]
            ps = [(i, conv(ocp.psi_t.get(i).download())) for i in idx]
            xs = [(i, conv(ocp.xi_t.get(i).download())) for i in idx]
            per_eval, det = cpu_sample_from_states(ps, xs, u)
            ncores = os.cpu_count() or 1
            line["cpu_baseline"] = {"value": 1.0 / per_eval, "unit": UNIT, "cores": ncores, "kind": "port",
                                    "sample": f"oracle port (NumPy/OpenBLAS, {ncores} threads): 1 forward + 1 backward Trotter step and 1 MPO "
                                              f"overlap from each of 8 evenly spaced slices of this run's psi_t / xi_t, extrapolated to "
                                              f"2*(Nt-1) steps + Nt+1 overlaps", **det}
        if args.batch > 1 and world == 1:
            # a control owns two slice stores of Nt slots (5.7 GB at this shape): as many at once as fit with 8 GB to spare
            D = CFG["d"] + 1
            caps = [min(CFG["maxm"], D ** min(b, CFG["L"] - b)) for b in range(CFG["L"] + 1)]
            per_control = 2.0 * nt() * 16.0 * sum(caps[j] * D * caps[j + 1] for j in range(CFG["L"]))
            nb = int(max(2, min(args.batch, (float(torch.cuda.mem_get_info(dev)[0]) - 8e9) // per_control)))
            log(f"cfg2: {nb} controls in flight")
            line["batched"] = batched_bench(nb, oc, st, psi_i, psi_f, ocp, c)
        with_cpu = world == 1 and not args.no_cpu_baseline
        if args.cfg1 and world == 1:
            log("cfg1 block")
            line["cfg1"] = cfg1_bench(oc, ctx, peak, with_cpu)
        if args.cfg5 and world == 1:
            log("cfg5 block")
            ctx.trim()
            line["cfg5"] = cfg5_bench(oc, ctx, peak, with_cpu)
    # blocks every rank takes part in
    ctx.trim()
    del ocp                                           # (frees 5.7 GB of slice stores before the larger workloads)
    if args.hessian_nt:
        log("cfg3 Hessian block")
        hb = hessian_bench(args.hessian_nt, oc, ocd, st, psi_i, psi_f, world, rank, dev, torch)
        if rank == 0:
            line["hessian"] = hb
    if args.cfg4_seeds > 0:
        log("cfg4 block")
        ctx.trim()                                    # the Hessian's 58 chains own ~100 GB of rings at the cfg2 shape
        c4, probs4, ctrls4, st4 = cfg4_bench(oc, ocd, ctx, world, rank, dev, torch, args.cfg4_seeds, args.cfg4_inflight)
        if rank == 0:
            if world == 1 and not args.no_cpu_baseline:
                c4["cpu_baseline"] = cfg4_cpu_sample(probs4, st4)
            line["cfg4"] = c4
        del probs4
    log("done")
    if rank == 0:
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def dump_outputs(path, ocp, c, cost, grad):
    """What the last timed evaluation computed, as float64 arrays `path/<name>.npy` (a few kB in all): the cost and the gradient
    the caller receives, divT (overlap derivative at every time point, real / imaginary columns), the fidelity of every slice of
    psi_t and the bond dimensions of every slice of psi_t and xi_t.  The inputs depend on --seed only, so two builds of the
    project can be compared output for output."""
    os.makedirs(path, exist_ok=True)
    out = {"cost": np.array([cost], dtype=np.float64),
           "gradient": np.asarray(grad, dtype=np.float64),
           "divT": np.ascontiguousarray(ocp.divT, dtype=np.complex128).view(np.float64).reshape(-1, 2),
           "fidelities": np.asarray(ocp.getFidelityForAllT(c, False), dtype=np.float64),   # overlaps of the stored psi_t, no new sweep
           "psi_bond_dims": np.asarray(ocp.psi_t.bond_dims(), dtype=np.float64),
           "xi_bond_dims": np.asarray(ocp.xi_t.bond_dims(), dtype=np.float64)}
    for name, a in out.items():
        np.save(os.path.join(path, name + ".npy"), a)
    log(f"cfg2: outputs of the last timed evaluation written to {path}")


def batched_bench(B, oc, st, psi_i, psi_f, ocp0, c0):
    """B independent controls evaluated concurrently on ONE GPU (2B sweeps on 2B streams): the batched-seeds workload of
    the north star.  Reported next to the single-evaluation headline, never instead of it."""
    probs, ctrls = [], []
    for k in range(B):
        basis, c, _ = make_problem_host(100 + k)
        probs.append(oc.OptimalControl(psi_f, psi_i, st, basis, CFG["gamma"]))
        ctrls.append(list(c))
    oc.batch_cost_gradient(probs, ctrls)                    # warm-up (allocates the per-chain workspaces)
    t0 = time.perf_counter()
    res = oc.batch_cost_gradient(probs, ctrls)
    dt = time.perf_counter() - t0
    # consistency with the single-evaluation path on the first control
    g1 = probs[0].getAnalyticGradient(ctrls[0], True)
    c1 = probs[0].getCost(ctrls[0], False)
    return {"evals_in_flight": B, "value": B / dt, "unit": UNIT, "seconds": dt,
            "max_abs_diff_vs_single": float(max(abs(res[0][0] - c1), np.max(np.abs(np.array(res[0][1]) - np.array(g1)))))}


# ----------------------------------------------------------------------------------------------
# the other configs of BASELINE.json as sub-blocks of the line (each with its own CPU sample)
# ----------------------------------------------------------------------------------------------
CFG1 = dict(L=5, d=4, Npart=5, J=1.0, T=2.0, tstep=0.01, maxm=80, cutoff=1e-8, gamma=1e-6, U_i=2.5, U_f=50.0)
CFG4 = dict(L=30, d=5, Npart=30, J=1.0, T=2.0, tstep=0.01, M=10, maxm=150, cutoff=1e-8, gamma=1e-6, U_i=2.5, U_f=50.0)
CFG5 = dict(L=50, d=5, Npart=50, J=1.0, T=5.0, tstep=0.01, maxm=256, cutoff=1e-10, gamma=1e-6)


def cfg1_control():
    import optimalcontrolmps_b200 as oc
    N = int(CFG1["T"] / CFG1["tstep"] + 1)
    u0 = np.array(oc.SeedGenerator.linsigmoidSeed(CFG1["U_i"], CFG1["U_f"], N, np.random.default_rng(7)))
    return np.clip(u0 + np.random.default_rng(2024).uniform(-0.5, 0.5, N), 2.0, 100.0)


def svd_roofline(lib, fn, peak):
    """Runs fn() once with the block-SVD kernels event-timed on their own streams; returns the roofline object."""
    import ctypes
    lib.ocmps_profile_enable(1)
    fn()
    out4 = np.zeros(4)
    lib.ocmps_profile_read(out4.ctypes.data_as(ctypes.POINTER(ctypes.c_double)))
    lib.ocmps_profile_enable(0)
    ms_tot, nl, fl_blk, fl_dense = out4
    ach = fl_blk / (ms_tot * 1e-3) / 1e12 if ms_tot > 0 else 0.0
    return {"kernel": "block SVD launch group: jacobi_blocks_kernel + jacobi_rot_kernel (+ qr_big_kernel + jacobi_big_kernel, the thread-block-"
                      "cluster pair for blocks beyond one SM, when the bond capacities are >= 112)",
            "bound": "latency", "achieved": ach, "peak": peak, "unit": "TFLOP/s",
            "frac": ach / peak if peak else None, "traffic": None, "launches": int(nl), "avg_launch_us": ms_tot * 1e3 / max(nl, 1),
            "algorithmic_flops": "block-summed F_gram+F_evd (SURVEY.md 8d)"}


def cfg1_bench(oc, ctx, peak, with_cpu):
    """BASELINE.json configs[0], the README input (README.md:30-45): L=5 Npart=5 d=4, T=2, Nt=201, Maxm=80, GRAPE.  The GPU runs
    the complete evaluation through the public API; the CPU port runs the complete evaluation too (it takes seconds)."""
    from optimalcontrolmps_b200.states import ground_state
    c = CFG1
    st = oc.BH_tDMRG(oc.BoseHubbard(c["L"], c["d"]), c["J"], c["tstep"], oc.Args("Cutoff=", c["cutoff"], "Maxm=", c["maxm"]), ctx=ctx)
    psi_i = ground_state(c["L"], c["d"], c["Npart"], c["U_i"])
    psi_f = ground_state(c["L"], c["d"], c["Npart"], c["U_f"])
    u = list(cfg1_control())
    N = len(u)
    p = oc.OptimalControl(psi_f, psi_i, st, N, c["gamma"])
    p.setThreadCount(2)

    def one():
        g = p.getAnalyticGradient(u, True)
        return p.getCost(u, False), g

    for _ in range(3):
        one()
    K = 5
    t0 = time.perf_counter()
    for _ in range(K):
        cost, g = one()
    dt = (time.perf_counter() - t0) / K
    out = {"workload": "cfg1 (README input): BH L=5 Npart=5 d=4 T=2.0 tstep=0.01 Maxm=80 GRAPE, one cost+gradient evaluation", "value": 1.0 / dt,
           "unit": UNIT, "ms_per_eval": dt * 1e3, "steps": K, "cost": float(cost), "grad_norm": float(np.linalg.norm(g)),
           "max_bond_dim": int(p.psi_t.bond_dims().max()), "roofline": svd_roofline(ctx.lib, one, peak)}
    if with_cpu:
        from oracle import bh_mps as ob, optimal_control as oo
        conv = lambda h: ob.MPS(h.A, [np.asarray(x, dtype=np.int64) for x in h.q], 0, 2)
        so = ob.BHStepper(c["L"], c["d"] + 1, c["J"], c["tstep"], ob.TruncArgs(cutoff=c["cutoff"], maxm=c["maxm"]))
        po = oo.OptimalControl(conv(psi_f), conv(psi_i), so, N=N, gamma=c["gamma"])
        t0 = time.perf_counter()
        go = po.getAnalyticGradient(u, True)
        co = po.getCost(u, False)
        dtc = time.perf_counter() - t0
        out["cpu_baseline"] = {"value": 1.0 / dtc, "unit": UNIT, "cores": os.cpu_count() or 1, "kind": "port",
                               "sample": "oracle port, one COMPLETE cfg1 evaluation", "seconds": dtc,
                               "cost_rel_diff_vs_gpu": abs(co - cost) / abs(co),
                               "grad_rel_diff_vs_gpu": float(np.max(np.abs(np.array(go) - np.array(g))) / np.max(np.abs(go)))}
    return out


def cfg4_bench(oc, ocd, ctx, world, rank, dev, torch, seeds_per_gpu, inflight):
    """BASELINE.json configs[3]: batched random-seed controls (SeedGenerator fan-out), BH L=30 Npart=30 d=5 chi=150; every GPU
    evaluates `seeds_per_gpu` controls (seeds 1 + rank*spg ...; 64 seeds = 8 per GPU on 8 GPUs), `inflight` of them at a time
    (a control owns two slice stores of 10.6 GB at this shape), results combined with one all-gather.  Weak scaling over GPUs."""
    import torch.distributed as dist
    from optimalcontrolmps_b200.states import ground_state
    c = CFG4
    st = oc.BH_tDMRG(oc.BoseHubbard(c["L"], c["d"]), c["J"], c["tstep"], oc.Args("Cutoff=", c["cutoff"], "Maxm=", c["maxm"]), ctx=ctx)
    psi_i = ground_state(c["L"], c["d"], c["Npart"], c["U_i"])
    psi_f = ground_state(c["L"], c["d"], c["Npart"], c["U_f"])
    N = int(c["T"] / c["tstep"] + 1)
    u0 = oc.SeedGenerator.linsigmoidSeed(c["U_i"], c["U_f"], N, np.random.default_rng(7))
    ref_basis = oc.ControlBasisFactory.buildChoppedSineBasis(u0, c["tstep"], c["T"], c["M"])
    ctrls = []
    for k in range(seeds_per_gpu):
        seed = 1 + rank * seeds_per_gpu + k
        cc = np.array(oc.SeedGenerator.randomCoeffSeed(-4.0, 4.0, c["M"], np.random.default_rng(4000 + seed)))
        for _ in range(40):
            uu = np.array(ref_basis.convertControl(list(cc)))
            if uu.min() >= 2.0 and uu.max() <= 100.0:
                break
            cc *= 0.8
        ctrls.append(list(cc))
    inflight = max(1, min(inflight, seeds_per_gpu))
    # A control owns two slice stores (psi_t, xi_t) of Nt slots; as many controls as fit the device memory with 8 GB to spare run
    # at once, in equal waves (measured on one B200: 2 in flight 0.59, 4: 1.06, 8: 1.59 evaluations/s).
    D = c["d"] + 1
    caps = [min(c["maxm"], D ** min(b, c["L"] - b)) for b in range(c["L"] + 1)]
    per_control = 2.0 * N * 16.0 * sum(caps[j] * D * caps[j + 1] for j in range(c["L"]))
    free_b = float(torch.cuda.mem_get_info(dev)[0])
    waves = [w for w in range(inflight, 0, -1) if seeds_per_gpu % w == 0]
    inflight = next((w for w in waves if w * per_control + 8e9 <= free_b), 1)

    def make(n):       # (a basis caches its last control, so every problem gets its own)
        return [oc.OptimalControl(psi_f, psi_i, st, oc.ControlBasisFactory.buildChoppedSineBasis(u0, c["tstep"], c["T"], c["M"]), c["gamma"])
                for _ in range(n)]

    while True:
        try:
            probs = make(inflight)
            oc.batch_cost_gradient(probs, ctrls[:inflight])     # warm-up (allocates the slice stores and per-chain workspaces, captures graphs)
            break
        except Exception:                                       # out of device memory after all: halve the wave
            if inflight == 1:
                raise
            probs = None
            ctx.trim()
            inflight = next(w for w in waves if w < inflight)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    t0 = time.perf_counter()
    res = []
    for k0 in range(0, seeds_per_gpu, inflight):
        cs = ctrls[k0:k0 + inflight]
        res += oc.batch_cost_gradient(probs[:len(cs)], cs)
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    mine = np.concatenate([np.concatenate([[r[0]], r[1]]) for r in res])
    if world > 1:
        tt = torch.tensor([dt], dtype=torch.float64, device=dev)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        dt = float(tt[0])
        allres = ocd.allgather_array(mine, dev)
    else:
        allres = [mine]
    out = {"workload": f"cfg4: {seeds_per_gpu * world} random-seed controls ({seeds_per_gpu} per GPU, {inflight} in flight), BH L=30 Npart=30 d=5 "
                       f"chi=150 GROUP M=10 T=2.0, cost+gradient each", "n_gpus": world, "scaling": "weak", "seeds": seeds_per_gpu * world,
           "value": seeds_per_gpu * world / dt, "unit": UNIT, "seconds": dt, "max_bond_dim": int(max(p.psi_t.bond_dims().max() for p in probs)),
           "mean_cost": float(np.mean([a.reshape(seeds_per_gpu, -1)[:, 0] for a in allres]))}
    return out, probs, ctrls, st


def cfg4_cpu_sample(probs, st_cfg):
    """CPU port on one forward + one backward step + one MPO overlap at 4 slices of the first cfg4 control, extrapolated."""
    from oracle import bh_mps as ob
    c = CFG4
    so = ob.BHStepper(c["L"], c["d"] + 1, c["J"], c["tstep"], ob.TruncArgs(cutoff=c["cutoff"], maxm=c["maxm"]))
    p = probs[0]
    N = p.getN()
    u = p.basis._ucurrent
    conv = lambda h: ob.MPS(h.A, [np.asarray(x, dtype=np.int64) for x in h.q], 0, 2)
    idx = [int(round(x)) for x in np.linspace(4, N - 5, 4)]
    tf, tb, to = [], [], []
    for i in idx:
        a = conv(p.psi_t.get(i).download()); b = conv(p.xi_t.get(i).download())
        t0 = time.perf_counter(); so.step(a.copy(), u[i], u[i + 1], True); tf.append(time.perf_counter() - t0)
        t0 = time.perf_counter(); so.step(b.copy(), u[i], u[i - 1], False); tb.append(time.perf_counter() - t0)
        t0 = time.perf_counter(); ob.overlap_K(b, a); to.append(time.perf_counter() - t0)
    per_eval = (N - 1) * (np.mean(tf) + np.mean(tb)) + (N + 1) * np.mean(to)
    return {"value": 1.0 / per_eval, "unit": UNIT, "cores": os.cpu_count() or 1, "kind": "port",
            "sample": "oracle port: 1 forward + 1 backward step + 1 MPO overlap at 4 slices of the first control, extrapolated to one evaluation "
                      "(the CPU evaluates the seeds one after the other)", "fwd_step_s": float(np.mean(tf)), "bwd_step_s": float(np.mean(tb)),
            "cpu_seconds": float(np.sum(tf) + np.sum(tb) + np.sum(to))}


def cfg5_bench(oc, ctx, peak, with_cpu):
    """BASELINE.json configs[4]: long chain BH L=50 Npart=50 d=5, chi=256, Cutoff=1e-10, SVD-bound stress on one GPU.  Bounded sample:
    the Mott product state is quenched (steps of 5*tstep at U=2.5) until the largest bond reaches 256, then forward Trotter steps
    and a BFGS-mode gradient (on-the-fly xi, src/OptimalControl.cpp:217-229) over a short horizon are timed; reported per step."""
    c = CFG5
    L, d = c["L"], c["d"]
    D = d + 1
    args = oc.Args("Cutoff=", c["cutoff"], "Maxm=", c["maxm"])
    quench = oc.BH_tDMRG(oc.BoseHubbard(L, d), c["J"], 5 * c["tstep"], args, ctx=ctx)
    st = oc.BH_tDMRG(oc.BoseHubbard(L, d), c["J"], c["tstep"], args, ctx=ctx)
    A = []
    for j in range(L):
        a = np.zeros((1, D, 1), dtype=np.complex128)
        a[0, 1, 0] = 1.0
        A.append(a)
    q = [np.array([b], dtype=np.int32) for b in range(L + 1)]
    psi = quench.to_device(oc.IQMPS(A, q, 0, 2))
    t0 = time.perf_counter()
    nq = 0
    while max(psi.bond_dims()) < c["maxm"] and nq < 400 and time.perf_counter() - t0 < 60.0:
        quench.step(psi, 2.5, 2.5, True)
        nq += 1
    t_quench = time.perf_counter() - t0
    dims = psi.bond_dims()
    K = 5
    st.step(psi, 2.5, 2.6, True)                       # warm (graph capture of the tstep stepper happens on reuse)
    st.step(psi, 2.6, 2.7, True)
    t0 = time.perf_counter()
    for k in range(K):
        st.step(psi, 2.7 + 0.1 * k, 2.8 + 0.1 * k, True)
    ms_step = (time.perf_counter() - t0) / K * 1e3
    # BFGS-mode gradient on a horizon of Nh points starting from the quenched state (target: the same state, so xi is as heavy as psi)
    Nh = 6
    u = list(np.linspace(3.2, 3.7, Nh))
    h = psi.download()
    pb = oc.OptimalControl(h, h, st, Nh, c["gamma"], True)
    pb.getAnalyticGradient(u, True)
    t0 = time.perf_counter()
    g = pb.getAnalyticGradient(u, True)
    cost = pb.getCost(u, False)
    t_bfgs = time.perf_counter() - t0
    Nt = int(c["T"] / c["tstep"] + 1)
    out = {"workload": "cfg5: BH L=50 Npart=50 d=5 chi=256 Cutoff=1e-10; bounded sample at saturated bond dimensions: forward Trotter steps and "
                       f"a BFGS-mode gradient over {Nh} time points", "quench_steps": nq, "quench_seconds": t_quench, "bond_dims_max": int(max(dims)),
           "bonds_at_256": int(sum(1 for x in dims if x >= c["maxm"])), "ms_per_forward_step": ms_step,
           "bfgs_gradient_ms_per_time_point": t_bfgs / Nh * 1e3, "unit": "ms",
           "extrapolated_eval_s_Nt501": (Nt - 1) * ms_step * 1e-3 + Nt * t_bfgs / Nh,
           "roofline": svd_roofline(ctx.lib, lambda: st.step(psi, 3.3, 3.4, True), peak)}
    if with_cpu:
        from oracle import bh_mps as ob
        so = ob.BHStepper(L, D, c["J"], c["tstep"], ob.TruncArgs(cutoff=c["cutoff"], maxm=c["maxm"]))
        hh = psi.download()
        po = ob.MPS(hh.A, [np.asarray(x, dtype=np.int64) for x in hh.q], 0, 2)
        t0 = time.perf_counter()
        so.step(po, 3.4, 3.5, True)
        dtc = time.perf_counter() - t0
        out["cpu_baseline"] = {"value": dtc * 1e3, "unit": "ms per forward step", "cores": os.cpu_count() or 1, "kind": "port",
                               "sample": "oracle port, ONE forward Trotter step from the same saturated state"}
    return out



def hessian_bench(Nt, oc, ocd, st, psi_i, psi_f, world, rank, dev, torch):
    """cfg3 (BASELINE.json configs[2]): full GROUP Hessian (M=20) of the cfg2 chain through the public API -- getHessian on one
    GPU, distributed.sharded_hessian (rows dealt to the ranks, one NCCL all-gather) on N.  Strong scaling: the work is fixed.
    On N>1 rank 0 first times the same Hessian alone on its GPU (the other ranks wait), so that the line carries its own
    1-GPU reference and the strong-scaling efficiency t1 / (N * tN)."""
    import torch.distributed as dist
    basis, c = make_hessian_problem_host(0)
    if Nt != nt():                       # reduced horizon (development): GRAPE on a ramp of Nt points
        basis = None
    och = oc.OptimalControl(psi_f, psi_i, st, basis if basis is not None else Nt, CFG["gamma"])
    och.setThreadCount(4)
    ctrl = list(c) if basis is not None else list(np.linspace(CFG["U_i"], 30.0, Nt))

    def once(sharded):
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        t0 = time.perf_counter()
        if sharded:
            H = ocd.sharded_hessian(och, ctrl, True, dev, convert=True)
        else:
            H = np.array(och.getHessian(ctrl, True))
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        if world > 1:
            tt = torch.tensor([dt], dtype=torch.float64, device=dev)
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            dt = float(tt[0])
        return dt, H

    out = {"workload": f"cfg3: full GROUP Hessian M={HESS_M if basis is not None else 0} (Nt={Nt}, {Nt - 2} rows, "
                       f"{(Nt - 2) * (Nt - 1) // 2} row steps + both sweeps + K.xi), BH L=20 chi=100", "Nt": Nt, "n_gpus": world,
           "scaling": "strong"}
    t1 = None
    if world > 1:
        # 1-GPU reference inside the same run (rank 0 alone; first call allocates and captures, second call is timed)
        if rank == 0:
            och.getHessian(ctrl, True)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            H1 = np.array(och.getHessian(ctrl, True))
            torch.cuda.synchronize()
            t1 = time.perf_counter() - t0
            out["t1_wall_s"] = t1
            out["t1_checksum"] = float(np.abs(H1).sum())
        dist.barrier()
    # first call: allocates the per-row workspaces and captures their step graphs; second call: what every further
    # Hessian of an optimisation run costs
    cold, _ = once(world > 1)
    warm, H = once(world > 1)
    out.update({"wall_s": warm, "first_call_s": cold, "checksum": float(np.abs(H).sum()), "shape": list(H.shape)})
    if world > 1 and t1 is not None:
        out["efficiency"] = t1 / (world * warm)
        out["max_abs_diff_vs_1gpu"] = float(np.max(np.abs(H - H1)))
    elif world == 1:
        out["efficiency"] = 1.0
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=2)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--hessian-nt", type=int, default=201,
                    help="time points of the Hessian block (201 = cfg3, the full GROUP M=20 Hessian; 0 switches the block off)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--seed", type=int, default=0, help="seed of the synthetic control")
    ap.add_argument("--distinct-seeds", action="store_true", help="N>1: rank r evaluates the control of seed r")
    ap.add_argument("--batch", type=int, default=24, help="additionally time this many independent controls in flight on one GPU (measured: 6 -> 2.65, 12 -> 4.99, 24 -> 7.74 evaluations/s; limited by the free device memory)")
    ap.add_argument("--cfg1", type=int, default=1, help="1: add the cfg1 block (README input, GPU and CPU in full; N=1 only)")
    ap.add_argument("--cfg5", type=int, default=1, help="1: add the cfg5 block (L=50 chi=256 bounded sample; N=1 only)")
    ap.add_argument("--cfg4-seeds", type=int, default=8, help="controls per GPU of the cfg4 block (L=30 chi=150 batched seeds); 0 = off")
    ap.add_argument("--cfg4-inflight", type=int, default=8, help="cfg4 controls evaluated concurrently per GPU at most (21 GB of slice stores each; limited by the free device memory)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write what the last timed cfg2 evaluation computed "
                                                          "(rank 0) as DIR/<name>.npy; GPU arm only")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of the GPU arm (--impl ours)")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
