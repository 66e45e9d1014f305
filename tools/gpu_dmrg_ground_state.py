"""Device two-site DMRG ground states (ocmps_ground_state_dmrg) at the project's chain shapes: wall time, energy, 1-F against the
shipped fixture where one exists, largest bond; the imaginary-time generator (ocmps_ground_state) at L=20 and L=30 for comparison;
kernel time per H_eff application at L=20 and L=50 from a torch.profiler pass of its own.  Prints the card and its power limit.
usage: gpu_dmrg_ground_state.py [out_dir]"""
import sys, os, time, json, subprocess
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import optimalcontrolmps_b200 as oc
from optimalcontrolmps_b200.states import ground_state, DATA_DIR

out_dir = sys.argv[1] if len(sys.argv) > 1 else None
card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                      capture_output=True, text=True).stdout.strip()
print(f"card: {card}", flush=True)
ctx = oc.Context.default(0)
rows = []


def fixture(L, d, Np, U):
    path = os.path.join(DATA_DIR, f"bh_L{L}_d{d}_N{Np}_U{U:g}.npz")
    return (ground_state(L, d, Np, U), float(np.load(path)["meta"][7])) if os.path.exists(path) else (None, None)


oc.InitializeStateDMRG(oc.BoseHubbard(8, 4), 8, 1.0, 2.5, 40, 1e-9, ctx=ctx)       # module load, first launches
for (L, d, Np, maxm, cutoff) in ((8, 4, 8, 40, 1e-9), (20, 5, 20, 100, 1e-8), (30, 5, 30, 150, 1e-8), (50, 5, 50, 256, 1e-10)):
    for U in (2.5, 50.0):
        ctx.synchronize()
        t0 = time.perf_counter()
        psi, e, sweeps = oc.InitializeStateDMRG(oc.BoseHubbard(L, d), Np, 1.0, U, maxm, cutoff, ctx=ctx, return_info=True)
        ctx.synchronize()
        dt = time.perf_counter() - t0
        ref, e_fix = fixture(L, d, Np, U)
        infid = None
        if ref is not None:
            dev_ref = oc.DeviceMPS(ctx, L, d + 1, psi.chi_cap).upload(ref)
            infid = 1.0 - abs(oc.overlapC(dev_ref, psi)) ** 2
        r = dict(kind="dmrg", L=L, d=d, N=Np, maxm=maxm, cutoff=cutoff, U=U, seconds=dt, energy=e, fixture_energy=e_fix,
                 one_minus_F=infid, max_bond=max(psi.bond_dims()), sweep_energies=[float(x) for x in sweeps])
        rows.append(r)
        print(json.dumps(r), flush=True)
for (L, d, Np, maxm, cutoff) in ((20, 5, 20, 100, 1e-8), (30, 5, 30, 150, 1e-8)):
    for U in (2.5, 50.0):
        ctx.synchronize()
        t0 = time.perf_counter()
        psi, e, n = oc.InitializeState(oc.BoseHubbard(L, d), Np, 1.0, U, maxm, cutoff, ctx=ctx, return_info=True)
        ctx.synchronize()
        r = dict(kind="tebd", L=L, d=d, N=Np, maxm=maxm, cutoff=cutoff, U=U, seconds=time.perf_counter() - t0, energy=e, steps=n)
        rows.append(r)
        print(json.dumps(r), flush=True)

# kernel time per H_eff application: heff_setup + the two boundary GEMM launches before each heff_combine + heff_combine
import torch
from torch.profiler import profile, ProfilerActivity
for (L, d, maxm, cutoff) in ((20, 5, 100, 1e-8), (50, 5, 256, 1e-10)):
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        oc.InitializeStateDMRG(oc.BoseHubbard(L, d), L, 1.0, 2.5, maxm, cutoff, ctx=ctx)
        ctx.synchronize()
    ev = sorted([e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA], key=lambda e: e.time_range.start)
    names = [e.name for e in ev]
    per = []
    for i, nm in enumerate(names):
        if "heff_combine" in nm and i >= 3 and "heff_setup" in names[i - 3]:
            per.append(sum(ev[k].time_range.elapsed_us() for k in range(i - 3, i + 1)))
    per = np.array(per)
    last = per[-200:] if len(per) else per     # the final sweep: bonds at their full size
    r = dict(kind="heff", L=L, maxm=maxm, applications=int(len(per)), mean_us=float(per.mean()) if len(per) else None,
             final_sweep_mean_us=float(last.mean()) if len(last) else None, max_us=float(per.max()) if len(per) else None)
    rows.append(r)
    print(json.dumps(r), flush=True)
if out_dir:
    os.makedirs(out_dir, exist_ok=True)
    with open(os.path.join(out_dir, "dmrg_ground_state.json"), "w") as f:
        json.dump(dict(card=card, rows=rows), f, indent=1)
