"""Time the energy moments over all 201 psi slices of the cfg2 evaluation (L=20 fixtures, bench.py's seeded GROUP control,
chi=100): the 4-channel pass (<H>), the 16-channel pass (<H>, <H^2>), and ocmps_store_overlaps over the same slices as the
yardstick.  Reports the achieved FP64 rate from the algorithmic flop count of the two gemms per site and channel,
F = sum_slices sum_sites n_ch * 8 (chi_l^2 D chi_r + chi_l D chi_r^2), and the card name and power limit read in the same run."""
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

import bench
import optimalcontrolmps_b200 as oc
from optimalcontrolmps_b200.states import ground_state


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:                                   # noqa: BLE001
        q = f"nvidia-smi unavailable ({e})"
    return q


def timed(fn, reps):
    ts = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        a.record()
        fn()
        b.record()
        torch.cuda.synchronize()
        ts.append(a.elapsed_time(b) * 1e-3)
    return float(np.median(ts)), float(np.min(ts))


def main():
    CFG = bench.CFG
    torch.cuda.init()
    ctx = oc.Context.default(0)
    st = oc.BH_tDMRG(oc.BoseHubbard(CFG["L"], CFG["d"]), CFG["J"], CFG["tstep"], oc.Args("Cutoff=", CFG["cutoff"], "Maxm=", CFG["maxm"]),
                     ctx=ctx)
    psi_i = ground_state(CFG["L"], CFG["d"], CFG["Npart"], CFG["U_i"])
    psi_f = ground_state(CFG["L"], CFG["d"], CFG["Npart"], CFG["U_f"])
    basis, c, _ = bench.make_problem_host(0)
    o = oc.OptimalControl(psi_f, psi_i, st, basis, CFG["gamma"])
    o.getFidelityForAllT(list(c), True)
    u = np.array(basis.convertControl(list(c), False))
    store = o.psi_t
    dims = store.bond_dims()
    D = store.D
    flops1 = float(sum(8.0 * (int(dl) ** 2 * D * int(dr) + int(dl) * D * int(dr) ** 2)
                       for row in dims for dl, dr in zip(row[:-1], row[1:])))
    target = st.to_device(psi_f)
    print(f"card: {card()}")
    print(f"slices {store.nslots}, max chi {int(dims.max())}, saturated slices {int(np.sum(dims.max(axis=1) == store.chi_cap))}")
    reps = 7
    res = {}
    ovl = np.zeros(2 * store.nslots)
    res["overlaps"] = timed(lambda: oc._lib.check(o.lib.ocmps_store_overlaps(store.h, target.h, store.nslots, oc.api._pd(ovl))), reps)
    res["energy 4ch"] = timed(lambda: store.energyMoments(CFG["J"], u, second_moment=False), reps)
    res["energy 16ch"] = timed(lambda: store.energyMoments(CFG["J"], u, second_moment=True), reps)
    res["energies(variance=True)"] = timed(lambda: store.energies(CFG["J"], u, variance=True), reps)
    for name, (med, best) in res.items():
        nch = {"overlaps": 1, "energy 4ch": 4, "energy 16ch": 16, "energies(variance=True)": 20}[name]
        F = nch * flops1
        print(f"{name:26s} median {med * 1e3:8.2f} ms  best {best * 1e3:8.2f} ms  F {F / 1e12:6.3f} TF  "
              f"rate {F / med / 1e12:6.2f} TF/s (median)")
    E, var = store.energies(CFG["J"], u, variance=True)
    print(f"E(t=0) {E[0]:.10f}  E(T) {E[-1]:.10f}  var(T) {var[-1]:.4e}")
    print(f"card after: {card()}")


if __name__ == "__main__":
    main()
