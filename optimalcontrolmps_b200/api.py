"""Host-side mirror of the reference's C++ interface for the hot path, over the libocmps C ABI.

Names, argument order and ``new_control`` caching semantics follow the reference:
``BoseHubbard`` (include/BH_sites.h:58), ``BH_tDMRG`` (include/BH_tDMRG.hpp:16-40),
``OptimalControl`` (include/OptimalControl.hpp:17-76, src/OptimalControl.cpp),
``ControlBasis`` (src/ControlBasis.cpp), ``ControlBasisFactory``
(include/ControlBasisFactory.hpp) and ``SeedGenerator`` (include/SeedGenerator.hpp).
All MPS arithmetic runs on the GPU through ``libocmps.so``; nothing here computes on the CPU
except the O(Nt*M) control-basis projections and regularisation terms, which the reference also
keeps in scalar loops.
"""
from __future__ import annotations

import ctypes as C
import math
from typing import List, Optional, Sequence

import numpy as np

from . import _lib

stdvec = List[float]


def _pd(a):
    return a.ctypes.data_as(C.POINTER(C.c_double))


def _pi(a):
    return a.ctypes.data_as(C.POINTER(C.c_int))


# ----------------------------------------------------------------------------------------------
# context / containers
# ----------------------------------------------------------------------------------------------
class Context:
    """One per GPU (``ocmps_ctx``)."""

    _default = {}

    def __init__(self, device: int = 0):
        self.lib = _lib.load()
        h = C.c_void_p()
        _lib.check(self.lib.ocmps_ctx_create(device, C.byref(h)))
        self.h = h
        self.device = device

    @classmethod
    def default(cls, device: int = 0) -> "Context":
        if device not in cls._default:
            cls._default[device] = cls(device)
        return cls._default[device]

    def synchronize(self):
        _lib.check(self.lib.ocmps_ctx_synchronize(self.h))

    def trim(self):
        """Frees the idle per-chain workspaces (scratch, Hessian rings, step graphs) the library keeps between calls."""
        _lib.check(self.lib.ocmps_ctx_trim(self.h))


class BoseHubbard:
    """``BoseHubbard(N, d)`` site set: N sites with occupations 0..d (local dimension d+1)."""

    def __init__(self, N: int, d: int):
        self._N = int(N)
        self.d = int(d)
        self.D = int(d) + 1

    def N(self):
        return self._N


class Args(dict):
    """ITensor ``Args{"Cutoff=",x,"Maxm=",y}``; keys are accepted with or without the trailing '='."""

    def __init__(self, *pairs, **kw):
        super().__init__()
        if len(pairs) == 1 and isinstance(pairs[0], dict):
            pairs = tuple(x for kv in pairs[0].items() for x in kv)
        for k, v in zip(pairs[0::2], pairs[1::2]):
            self[str(k).rstrip("=")] = v
        for k, v in kw.items():
            self[k] = v

    def defined(self, k):
        return k.rstrip("=") in self

    def getReal(self, k, default=None):
        return float(self.get(k.rstrip("="), default))

    def getInt(self, k, default=None):
        return int(self.get(k.rstrip("="), default))


class IQMPS:
    """Host container of a charge-labelled MPS (the role ITensor's IQMPS plays in the reference's
    signatures).  ``A[j]``: complex128 array (chi_j, D, chi_{j+1}); ``q[b]``: int array with the boson
    number left of bond ``b`` per index.  Holds no arithmetic: everything numeric happens on the GPU."""

    def __init__(self, A: Sequence[np.ndarray], q: Sequence[np.ndarray], llim: int = 0, rlim: int = 2):
        self.A = [np.ascontiguousarray(a, dtype=np.complex128) for a in A]
        self.q = [np.ascontiguousarray(x, dtype=np.int32) for x in q]
        self.llim, self.rlim = int(llim), int(rlim)
        if len(self.q) != len(self.A) + 1:
            raise ValueError("need L+1 charge arrays")
        for j, a in enumerate(self.A):
            if a.ndim != 3 or a.shape[0] != len(self.q[j]) or a.shape[2] != len(self.q[j + 1]):
                raise ValueError(f"site {j}: tensor shape {a.shape} does not match the charge labels")

    def N(self):
        return len(self.A)

    @property
    def D(self):
        return self.A[0].shape[1]

    def bond_dims(self):
        return [len(x) for x in self.q]

    def copy(self):
        return IQMPS([a.copy() for a in self.A], [x.copy() for x in self.q], self.llim, self.rlim)


class DeviceMPS:
    """``ocmps_mps`` handle."""

    def __init__(self, ctx: Context, L: int, D: int, chi_cap: int):
        self.ctx, self.L, self.D, self.chi_cap = ctx, L, D, chi_cap
        h = C.c_void_p()
        _lib.check(ctx.lib.ocmps_mps_create(ctx.h, L, D, chi_cap, C.byref(h)))
        self.h = h

    def __del__(self):
        try:
            if getattr(self, "h", None):
                self.ctx.lib.ocmps_mps_destroy(self.h)
                self.h = None
        except Exception:
            pass

    def upload(self, psi: IQMPS):
        if psi.N() != self.L or psi.D != self.D:
            raise ValueError("shape mismatch")
        dims = np.array(psi.bond_dims(), dtype=np.int32)
        charges = np.ascontiguousarray(np.concatenate(psi.q), dtype=np.int32)
        flat = np.ascontiguousarray(np.concatenate([a.ravel() for a in psi.A]))
        _lib.check(self.ctx.lib.ocmps_mps_upload(self.h, _pi(dims), _pi(charges), _pd(flat.view(np.float64)), psi.llim, psi.rlim))
        return self

    def bond_dims(self):
        dims = np.zeros(self.L + 1, dtype=np.int32)
        _lib.check(self.ctx.lib.ocmps_mps_bond_dims(self.h, _pi(dims)))
        return dims.tolist()

    def download(self) -> IQMPS:
        ne, nq = C.c_longlong(), C.c_longlong()
        _lib.check(self.ctx.lib.ocmps_mps_sizes(self.h, C.byref(ne), C.byref(nq)))
        dims = np.zeros(self.L + 1, dtype=np.int32)
        charges = np.zeros(nq.value, dtype=np.int32)
        flat = np.zeros(ne.value, dtype=np.complex128)
        ll, rl = C.c_int(), C.c_int()
        _lib.check(self.ctx.lib.ocmps_mps_download(self.h, _pi(dims), _pi(charges), _pd(flat.view(np.float64)), C.byref(ll), C.byref(rl)))
        A, q, off, qoff = [], [], 0, 0
        for j in range(self.L):
            n = int(dims[j]) * self.D * int(dims[j + 1])
            A.append(flat[off:off + n].reshape(int(dims[j]), self.D, int(dims[j + 1])).copy())
            off += n
        for b in range(self.L + 1):
            q.append(charges[qoff:qoff + int(dims[b])].copy())
            qoff += int(dims[b])
        return IQMPS(A, q, ll.value, rl.value)

    def position1(self):
        """``psi.position(1)``: gauge moves of the engine from the orthogonality limits of the uploaded state to site 1."""
        _lib.check(self.ctx.lib.ocmps_mps_position1(self.h))
        return self

    def copy_from(self, other: "DeviceMPS"):
        _lib.check(self.ctx.lib.ocmps_mps_copy(self.h, other.h))
        return self

    def norm(self) -> float:
        out = C.c_double()
        _lib.check(self.ctx.lib.ocmps_mps_norm(self.h, C.byref(out)))
        return out.value


class SliceStore:
    """``ocmps_store``: Nt time slices resident in HBM."""

    def __init__(self, ctx: Context, L: int, D: int, chi_cap: int, nslots: int):
        self.ctx, self.L, self.D, self.chi_cap, self.nslots = ctx, L, D, chi_cap, nslots
        h = C.c_void_p()
        _lib.check(ctx.lib.ocmps_store_create(ctx.h, L, D, chi_cap, nslots, C.byref(h)))
        self.h = h

    def __del__(self):
        try:
            if getattr(self, "h", None):
                self.ctx.lib.ocmps_store_destroy(self.h)
                self.h = None
        except Exception:
            pass

    def get(self, slot: int) -> DeviceMPS:
        m = DeviceMPS(self.ctx, self.L, self.D, self.chi_cap)
        _lib.check(self.ctx.lib.ocmps_store_get(self.h, slot, m.h))
        return m

    def put(self, slot: int, m: DeviceMPS):
        _lib.check(self.ctx.lib.ocmps_store_put(self.h, slot, m.h))

    def bond_dims(self):
        out = np.zeros((self.nslots, self.L + 1), dtype=np.int32)
        _lib.check(self.ctx.lib.ocmps_store_bond_dims(self.h, _pi(out)))
        return out

    def entanglementEntropy(self, first=0, count=None):
        """``entanglementEntropy(sites, psi)`` (include/correlations.hpp:119-148) for the resident slices: array
        [slice, bond] of the von Neumann entropies -sum_{p>1e-12} p ln p of the L-1 bonds."""
        count = self.nslots - first if count is None else count
        out = np.zeros((count, self.L - 1))
        _lib.check(self.ctx.lib.ocmps_store_entanglement_entropy(self.h, first, count, _pd(out)))
        return out

    # ---- two-point functions (include/correlations.hpp:10-97), one batched transfer-matrix pass per call ----
    def correlationFunction(self, slot: int, opname1: str, i: int, opname2: str, j: int) -> complex:
        """``correlationFunction(sites, psi, opname1, i, opname2, j)`` for the slice ``slot``: <psi| Op1_i Op2_j |psi>, sites
        1-based.  (For i > j the reference swaps the sites but not the operators, which ITensor then cannot contract; here
        the value is simply the expectation of Op1 at site i and Op2 at site j in either order.)"""
        return complex(_correlation_entries(self, slot, [(opname1, i, opname2, j)])[0])

    def correlationMatrix(self, slot: int, opname1: str, opname2: str) -> np.ndarray:
        """``correlationMatrix`` (:57-80): rho[i, j] = <Op1_i Op2_j> for i <= j, rho[j, i] = conj(rho[i, j]).  The diagonal is
        real (the reference takes ``.real()`` of the same-site value, :24)."""
        L = self.L
        req = [(opname1, i, opname2, j) for i in range(1, L + 1) for j in range(i, L + 1)]
        vals = _correlation_entries(self, slot, req)
        rho = np.zeros((L, L), dtype=np.complex128)
        for (o1, i, o2, j), v in zip(req, vals):
            if i == j:
                rho[i - 1, i - 1] = v.real
            else:
                rho[i - 1, j - 1] = v
                rho[j - 1, i - 1] = np.conj(v)
        return rho

    def correlationTerm(self, slot: int, opname1: str, opname2: str) -> float:
        """``correlationTerm`` (:82-97): largest eigenvalue of the correlation matrix (an L x L Hermitian matrix, diagonalised
        on the host like every other O(L^3) post-processing step of the reference)."""
        return float(np.linalg.eigvalsh(self.correlationMatrix(slot, opname1, opname2))[-1])

    # site operators of include/BH_sites.h:129-171 that are diagonal in the boson number
    SITE_OPS = {"N": lambda n: n, "N(N-1)": lambda n: n * (n - 1.0), "NN": lambda n: n * n, "Id": lambda n: 1.0 + 0.0 * n}

    def expectationValues(self, opnames=("N",), first=0, count=None, return_norm=False):
        """``expectationValues(sites, psi, opname)`` (include/correlations.hpp:109-117) for every resident slice at once:
        array [slice, site, op] of <psi| O_site |psi> (not divided by the norm, like the reference).  Operators by name
        (N, N(N-1), NN, Id) or as explicit diagonals of length D."""
        count = self.nslots - first if count is None else count
        n = np.arange(self.D, dtype=float)
        diags = np.array([self.SITE_OPS[o](n) if isinstance(o, str) else np.asarray(o, dtype=float) for o in opnames], dtype=float)
        if diags.shape != (len(opnames), self.D):
            raise ValueError("operator diagonals must have length D")
        diags = np.ascontiguousarray(diags)
        out = np.zeros((count, self.L, len(opnames)))
        nrm = np.zeros((count, self.L))
        _lib.check(self.ctx.lib.ocmps_store_site_expectations(self.h, first, count, _pd(diags), len(opnames), _pd(out), _pd(nrm)))
        return (out, nrm) if return_norm else out

    # ---- energy of the Bose-Hubbard Hamiltonian H(U) = -J sum (a_i adag_{i+1} + h.c.) + U/2 sum n_i(n_i-1) ----
    def energyMoments(self, J: float, U, first=0, count=None, shift=None, second_moment=True):
        """Raw moments of H(U_z) - c_z on the slices first..first+count-1 in one transfer-matrix pass over the MPO channels:
        arrays ``(norm2, h1, h2)`` of <psi|psi>, <psi|H-c|psi> and <psi|(H-c)^2|psi> (nothing divided by the norm; h2 is NaN
        with ``second_moment=False``, which runs the 4-channel chain at about a quarter of the cost).  ``U`` and ``shift`` are
        scalars or one value per slice.  Any gauge."""
        count = self.nslots - first if count is None else count
        u = np.ascontiguousarray(np.broadcast_to(np.asarray(U, dtype=np.float64), (count,)))
        c = None if shift is None else np.ascontiguousarray(np.broadcast_to(np.asarray(shift, dtype=np.float64), (count,)))
        out = np.full((count, 3), np.nan)
        _lib.check(self.ctx.lib.ocmps_store_energy_moments(self.h, int(first), int(count), float(J), _pd(u),
                                                            None if c is None else _pd(c), 1 if second_moment else 0, _pd(out)))
        return out[:, 0].copy(), out[:, 1].copy(), out[:, 2].copy()

    def energies(self, J: float, U, first=0, count=None, variance=False):
        """<psi|H(U_z)|psi> / <psi|psi> of every slice; with ``variance=True`` ``(E, var)``, var = <H^2> - <H>^2 from a second pass
        of the 16-channel chain shifted by E (so that no E^2 cancels against <H^2>)."""
        n, h1, _ = self.energyMoments(J, U, first, count, second_moment=False)
        E = h1 / n
        if not variance:
            return E
        n2, g1, g2 = self.energyMoments(J, U, first, count, shift=E, second_moment=True)
        return E, g2 / n2 - (g1 / n2) ** 2


def energy(psi: "DeviceMPS", J: float, U: float, variance: bool = False):
    """<psi|H(U)|psi> / <psi|psi> of a device MPS (``(E, var)`` with ``variance=True``), e.g. the convergence check of a DMRG ground
    state: the variance <H^2> - <H>^2 vanishes on an eigenstate."""
    store = SliceStore(psi.ctx, psi.L, psi.D, psi.chi_cap, 1)
    store.put(0, psi)
    out = store.energies(J, [U], 0, 1, variance=variance)
    return (float(out[0][0]), float(out[1][0])) if variance else float(out[0])


def site_operator(opname: str, D: int) -> np.ndarray:
    """<t|Op|s> of the site operators of include/BH_sites.h:129-171 as a real D x D matrix ("Id" is the true identity, which
    is what ITensor's SiteSet hands out for that name)."""
    n = np.arange(D, dtype=float)
    if opname == "N":
        return np.diag(n)
    if opname == "N(N-1)":
        return np.diag(n * (n - 1.0))
    if opname == "NN":
        return np.diag(n * n)
    if opname == "Id":
        return np.eye(D)
    A = np.zeros((D, D))
    for j in range(1, D):
        A[j - 1, j] = math.sqrt(j)                     # <j-1|A|j> = sqrt(j)   (:136-141)
    if opname == "A":
        return A
    if opname == "Adag":
        return A.T.copy()                              # <j|Adag|j-1> = sqrt(j) (:143-148)
    raise ValueError(f"site operator {opname!r} not recognized")


def _correlation_entries(store: "SliceStore", slot: int, requests):
    """requests: list of (opname1, i, opname2, j), sites 1-based like the reference.  Returns complex values
    <psi| Op1_i Op2_j |psi> (include/correlations.hpp:10-55; for i == j the product Op1.Op2 on that site, :17-24)."""
    D = store.D
    table, index = [], {}

    def op_id(mat):
        key = mat.tobytes()
        if key not in index:
            index[key] = len(table)
            table.append(mat)
        return index[key]

    entries = []
    for (o1, i, o2, j) in requests:
        if not (1 <= i <= store.L and 1 <= j <= store.L):
            raise ValueError("site out of range")
        m1, m2 = site_operator(o1, D), site_operator(o2, D)
        if i == j:
            entries.append((i - 1, op_id(m1 @ m2), -1, 0))
        else:
            entries.append((i - 1, op_id(m1), j - 1, op_id(m2)))
    ops = np.ascontiguousarray(np.stack(table), dtype=np.float64)
    ent = np.ascontiguousarray(np.array(entries, dtype=np.int32))
    out = np.zeros(2 * len(entries))
    _lib.check(store.ctx.lib.ocmps_store_correlations(store.h, int(slot), _pd(ops), len(table), _pi(ent), len(entries), _pd(out)))
    return out.view(np.complex128).copy()


def InitializeState(sites: "BoseHubbard", Npart: int, J: float, U: float, maxBondDim: int = 200, threshold: float = 1e-9,
                    tau_final: float = 0.0, ctx: Optional["Context"] = None, chi_cap: Optional[int] = None, return_info: bool = False):
    """``InitializeState(sites, Npart, J, U[, maxBondDim, threshold])`` (include/InitializeState.hpp:18-117): Bose-Hubbard ground
    state as a device-resident MPS.  The reference runs ITensor's DMRG (maxm 10, 20, 50, maxBondDim; cutoff = threshold); here
    the engine's own Trotter-step kernels run in imaginary time with the same start state and bond-dimension schedule
    (``ocmps_ground_state``).  Returns a DeviceMPS (``.download()`` gives the host container)."""
    ctx = ctx or Context.default()
    L, D = sites.N(), sites.D
    cap = int(chi_cap or min(maxBondDim, D ** (L // 2)))
    out = DeviceMPS(ctx, L, D, cap)
    e, n = C.c_double(), C.c_int()
    _lib.check(ctx.lib.ocmps_ground_state(ctx.h, L, D, int(Npart), float(J), float(U), min(int(maxBondDim), cap), float(threshold),
                                          float(tau_final), out.h, C.byref(e), C.byref(n)))
    return (out, e.value, n.value) if return_info else out


def InitializeStateDMRG(sites: "BoseHubbard", Npart: int, J: float, U: float, maxBondDim: int = 200, threshold: float = 1e-9,
                        nsweeps: int = 10, ctx: Optional["Context"] = None, chi_cap: Optional[int] = None, return_info: bool = False):
    """The ground state of ``InitializeState`` computed as the reference computes it (include/InitializeState.hpp:18-117): two-site
    DMRG on the device, ``nsweeps`` sweeps with maxm 10, 20, 50, maxBondDim and cutoff ``threshold``, no noise term
    (``ocmps_ground_state_dmrg``).  Returns a DeviceMPS, or ``(psi, energy, sweep_energies)`` with ``return_info``: ``energy`` is
    <psi|H|psi> of the returned state, ``sweep_energies`` the last Ritz value of every sweep."""
    ctx = ctx or Context.default()
    L, D = sites.N(), sites.D
    cap = int(chi_cap or min(maxBondDim, D ** (L // 2)))
    out = DeviceMPS(ctx, L, D, cap)
    e = C.c_double()
    sweeps = np.zeros(max(int(nsweeps), 1))
    _lib.check(ctx.lib.ocmps_ground_state_dmrg(ctx.h, L, D, int(Npart), float(J), float(U), min(int(maxBondDim), cap), float(threshold),
                                               int(nsweeps), out.h, C.byref(e), _pd(sweeps)))
    return (out, e.value, sweeps) if return_info else out


def overlapC(a: DeviceMPS, b: DeviceMPS) -> complex:
    """<a|b>, first argument conjugated (ITensor ``overlapC``)."""
    out = np.zeros(2)
    _lib.check(a.ctx.lib.ocmps_overlap(a.h, b.h, _pd(out)))
    return complex(out[0], out[1])


def overlapC_K(a: DeviceMPS, b: DeviceMPS) -> complex:
    """<a|K|b> with the stepper's propagator derivative K (``overlapC(a, propDeriv, b)``)."""
    out = np.zeros(2)
    _lib.check(a.ctx.lib.ocmps_overlap_K(a.h, b.h, _pd(out)))
    return complex(out[0], out[1])


# ----------------------------------------------------------------------------------------------
# BH_tDMRG
# ----------------------------------------------------------------------------------------------
class BH_tDMRG:
    """Time stepper (include/BH_tDMRG.hpp:16-40).  ``chi_cap`` is the allocated bond capacity on the
    GPU; it defaults to ``Maxm`` when given, else to min(D^(L/2), 256)."""

    def __init__(self, sites: BoseHubbard, J: float, tstep: float, args: Args, chi_cap: Optional[int] = None,
                 ctx: Optional[Context] = None, rel_cutoff: bool = False):
        self.sites = sites
        self.J = float(J)
        self.args = args if isinstance(args, Args) else Args(args)
        self.ctx = ctx or Context.default()
        L, D = sites.N(), sites.D
        cutoff = self.args.getReal("Cutoff") if self.args.defined("Cutoff") else -1.0
        maxm = self.args.getInt("Maxm") if self.args.defined("Maxm") else 0
        if chi_cap is None:
            chi_cap = maxm if maxm > 0 else min(D ** (L // 2), 256)
        chi_cap = min(chi_cap, D ** (L // 2))
        self.L, self.D, self.chi_cap = L, D, int(chi_cap)
        h = C.c_void_p()
        _lib.check(self.ctx.lib.ocmps_stepper_create(self.ctx.h, L, D, self.J, float(tstep), cutoff, maxm, self.chi_cap,
                                                      1 if rel_cutoff else 0, C.byref(h)))
        self.h = h

    def __del__(self):
        try:
            if getattr(self, "h", None):
                self.ctx.lib.ocmps_stepper_destroy(self.h)
                self.h = None
        except Exception:
            pass

    # -- reference API
    def setTstep(self, tstep: float):
        _lib.check(self.ctx.lib.ocmps_stepper_set_tstep(self.h, float(tstep)))

    def getTstep(self) -> float:
        return self.ctx.lib.ocmps_stepper_get_tstep(self.h)

    def getArgs(self) -> Args:
        return self.args

    def getJ(self) -> float:
        return self.J

    def propagatorDeriv(self, control_n: float = 0.0):
        """The constant MPO K = sum_j 1/2 n_j(n_j-1) (src/BH_tDMRG.cpp:10-14,238-241); it lives inside the
        library, so this returns only a tag accepted by ``overlapC_K`` / ``exactApplyMPO``."""
        return "K"

    def step(self, psi, from_: float, to: float, propagateForward: bool = True):
        """In-place Trotter step.  ``psi`` may be a DeviceMPS (stays on the GPU) or a host IQMPS
        (uploaded, stepped, written back -- the drop-in behaviour of ``BH_tDMRG::step``)."""
        if isinstance(psi, DeviceMPS):
            _lib.check(self.ctx.lib.ocmps_step(self.h, psi.h, float(from_), float(to), 1 if propagateForward else 0))
            return psi
        dev = self.to_device(psi)
        _lib.check(self.ctx.lib.ocmps_step(self.h, dev.h, float(from_), float(to), 1 if propagateForward else 0))
        res = dev.download()
        psi.A, psi.q, psi.llim, psi.rlim = res.A, res.q, res.llim, res.rlim
        return psi

    # -- helpers
    def to_device(self, psi: IQMPS) -> DeviceMPS:
        """Uploads a host state; if its orthogonality limits say the centre is not at site 1 it is gauged there with the
        engine's own moves (the reference's step starts with psi.position(), src/BH_tDMRG.cpp:139-148)."""
        dev = DeviceMPS(self.ctx, self.L, self.D, self.chi_cap).upload(psi)
        if (psi.llim, psi.rlim) != (0, 2):
            dev.position1()
        return dev

    def new_mps(self) -> DeviceMPS:
        return DeviceMPS(self.ctx, self.L, self.D, self.chi_cap)

    def new_store(self, nslots: int) -> SliceStore:
        return SliceStore(self.ctx, self.L, self.D, self.chi_cap, nslots)

    def exactApplyMPO(self, psi: DeviceMPS) -> DeviceMPS:
        out = self.new_mps()
        _lib.check(self.ctx.lib.ocmps_apply_K(self.h, psi.h, out.h))
        return out

    def schedule(self):
        buf = np.zeros(4 * 4096, dtype=np.int32)
        n = self.ctx.lib.ocmps_stepper_schedule(self.h, _pi(buf), 4096)
        return buf[:4 * n].reshape(n, 4).tolist()

    def gate(self, forward=True) -> np.ndarray:
        n = self.D * self.D
        out = np.zeros((n, n), dtype=np.complex128)
        _lib.check(self.ctx.lib.ocmps_stepper_gate(self.h, 1 if forward else 0, _pd(out.view(np.float64))))
        return out


# ----------------------------------------------------------------------------------------------
# SeedGenerator / ControlBasis / ControlBasisFactory
# ----------------------------------------------------------------------------------------------
class SeedGenerator:
    """include/SeedGenerator.hpp.  The random seeds take a ``numpy.random.Generator`` instead of libc
    ``rand()`` (whose stream is not reproducible across platforms)."""

    @staticmethod
    def linspace(a: float, b: float, n: int) -> stdvec:
        out, step = [], (b - a) / (n - 1)
        while a <= b + 1e-7:
            out.append(a)
            a += step
        return out

    @staticmethod
    def generateRange(a: float, b: float, c: float) -> stdvec:
        out = []
        while a <= c + 1e-7:
            out.append(a)
            a += b
        return out

    @staticmethod
    def sigmoid(x: Sequence[float], k: float, offset: float) -> stdvec:
        return [1.0 / (1.0 + math.exp(-k * (v - offset))) for v in x]

    @staticmethod
    def linsigmoidSeed(u_start: float, u_end: float, length: int, rng=None) -> stdvec:
        rng = rng or np.random.default_rng()
        x = SeedGenerator.linspace(0, 100, length)
        a = float(rng.uniform(0.01, 0.15))
        b = u_end - u_start - a * x[-1]
        c = float(rng.uniform(0.06, 0.18))
        d = float(rng.uniform(60, 80))
        s1 = SeedGenerator.sigmoid(x, 0.7, 5)
        s2 = SeedGenerator.sigmoid(x, -0.9, 100 - 7)
        half = len(s1) // 2
        s1[half:] = s2[half:]
        s1[0] = 0.0
        s1[-1] = 0.0
        ramp = []
        for w, fx in zip(s1, x):
            inner = a * fx + b / (1 + math.exp(-c * (fx - d))) + u_start
            outer = (u_end - u_start) / (1 + math.exp(-0.2 * (fx - 40))) + u_start
            ramp.append(w * inner + (1 - w) * outer)
        return ramp

    @staticmethod
    def adiabaticSeed(u_start: float, u_end: float, length: int) -> stdvec:
        p, k, xs, a = 3.5, 1.0 / 3.0, 40.0, 0.01
        out = []
        for x in SeedGenerator.linspace(0, 100, length):
            if x < xs:
                out.append((p - u_start - a * xs) / (1 + math.exp(-k * (x - xs / 2.0))) + u_start + a * x)
            else:
                out.append(math.exp(math.log(u_end - p + 1) / (100 - xs) * (x - xs)) + p - 1)
        return out

    @staticmethod
    def randomCoeffSeed(lo: float, hi: float, N: int, rng=None) -> stdvec:
        rng = rng or np.random.default_rng()
        return [float(v) for v in rng.uniform(lo, hi, N)]


class ControlBasis:
    """u(t_i) = u0(t_i) + S(t_i) * sum_n c_n f_n(t_i)   (include/ControlBasis.hpp, src/ControlBasis.cpp)."""

    def __init__(self, u0: Optional[Sequence[float]] = None, S: Optional[Sequence[float]] = None, f=None):
        if u0 is None:
            self._N = self._M = 0
            return
        self._u0 = np.array(u0, dtype=float)
        self._S = np.array(S, dtype=float)
        self._f = np.array(f, dtype=float)
        self._N, self._M = self._f.shape
        self._jac = self._f * self._S[:, None]           # du_i/dc_n (:14-24)
        self._ucurrent = self._u0.copy()                 # :27

    def getM(self):
        return self._M

    def getN(self):
        return self._N

    def convertControl(self, control: Sequence[float], new_control: bool = True) -> stdvec:
        if new_control:                                  # :53-63, cached otherwise
            c = np.asarray(control, dtype=float)
            assert c.size == self._M
            u = self._u0.copy()
            for i in range(self._N):
                acc = 0.0
                for n in range(self._M):
                    acc += self._f[i, n] * c[n]
                u[i] += self._S[i] * acc
            self._ucurrent = u
        return self._ucurrent.tolist()

    def convertGradient(self, gradu: Sequence[float]) -> stdvec:
        g = np.asarray(gradu, dtype=float)
        assert g.size == self._N
        out = []
        for n in range(self._M):                         # :77-86
            acc = 0.0
            for i in range(self._N):
                acc += self._S[i] * g[i] * self._f[i, n]
            out.append(acc)
        return out

    def convertHessian(self, Hessu) -> List[List[float]]:
        H = np.asarray(Hessu, dtype=float)
        assert H.shape == (self._N, self._N)
        V = self._jac.T                                  # rows are S*f_n (:30-38)
        out = np.zeros((self._M, self._M))
        for i in range(self._M):
            for j in range(i, self._M):                  # upper triangle, mirrored (:99-116)
                out[i, j] = float(V[i] @ (H @ V[j]))
                out[j, i] = out[i, j]
        return out.tolist()

    def getControlJacobian(self) -> List[List[float]]:
        return self._jac.tolist()


class ControlBasisFactory:
    PI = 3.14159265      # include/ControlBasisFactory.hpp:10

    @staticmethod
    def buildChoppedSineBasis(u0: Sequence[float], tstep: float, T: float, M: int) -> ControlBasis:
        N = len(u0)
        x = SeedGenerator.linspace(0, 100, N)
        S = SeedGenerator.sigmoid(x, 8.0, 1.1)
        S2 = SeedGenerator.sigmoid(x, -8.0, 100 - 1.1)
        S[N // 2:] = S2[N // 2:]
        S[0] = 0.0
        S[N - 1] = 0.0
        f = [[math.sin((n + 1) * ControlBasisFactory.PI * tstep * i / T) for n in range(M)] for i in range(N)]
        return ControlBasis(u0, S, f)


# ----------------------------------------------------------------------------------------------
# OptimalControl
# ----------------------------------------------------------------------------------------------
class OptimalControl:
    """``OptimalControl<BH_tDMRG>``: GRAPE constructor ``(psi_target, psi_init, stepper, N, gamma, BFGS)``,
    GROUP constructor ``(psi_target, psi_init, stepper, basis, gamma, BFGS)`` -- target first, init second
    (include/OptimalControl.hpp:54-56).  psi_t / xi_t / xiHlist are slice stores resident in HBM."""

    def __init__(self, psi_target, psi_init, timeStepper: BH_tDMRG, N_or_basis, gamma: float, BFGS: bool = False):
        self.timeStepper = timeStepper
        self.ctx = timeStepper.ctx
        self.lib = self.ctx.lib
        self.tstep = timeStepper.getTstep()
        self.gamma = float(gamma)
        self.BFGS = bool(BFGS)
        self.calculatedXi = False
        self.threadCount = 1
        if isinstance(N_or_basis, ControlBasis):
            self.basis = N_or_basis
            self.GRAPE = False
            self.N = self.basis.getN()
            self.M = self.basis.getM()
        else:
            self.basis = ControlBasis()
            self.GRAPE = True
            self.N = int(N_or_basis)
            self.M = 0
        st = timeStepper
        self.psi_target = self._own(psi_target)
        self.psi_init = self._own(psi_init)
        self.psi_t = st.new_store(self.N)
        self.divT = np.zeros(self.N, dtype=np.complex128)
        self.xi_t = None if self.BFGS else st.new_store(self.N)
        self.xiHlist = None
        self.rows = None            # Hessian rows owned by this process (None: all); set by the multi-GPU driver
        self.hessian_chains = None  # rows in flight at once (default: derived from threadCount)

    def _own(self, psi) -> DeviceMPS:
        st = self.timeStepper
        if isinstance(psi, DeviceMPS):
            return st.new_mps().copy_from(psi)
        return st.to_device(psi)

    # -- setters (src/OptimalControl.cpp:55-85)
    def setThreadCount(self, n: int):
        if n < 1:
            raise ValueError("Mininum threadCount is 1.")
        self.threadCount = int(n)

    def setGRAPE(self, useGRAPE: bool):
        self.GRAPE = bool(useGRAPE)
        self.calculatedXi = False

    def setBFGS(self, useBFGS: bool):
        self.BFGS = bool(useBFGS)
        self.calculatedXi = False
        if self.BFGS:
            self.xi_t = None
            self.xiHlist = None
        else:
            self.xi_t = self.timeStepper.new_store(self.N)

    def useBFGS(self):
        return self.BFGS

    def setGamma(self, g: float):
        self.gamma = float(g)

    def getM(self):
        return self.M

    def getN(self):
        return self.N

    def getPsit(self) -> List[IQMPS]:
        return [self.psi_t.get(i).download() for i in range(self.N)]

    def getControl(self, control):
        return list(control) if self.GRAPE else self.basis.convertControl(control)

    def getTimeAxis(self) -> stdvec:
        out, t = [], 0.0
        while abs(t - self.N * self.tstep) > 1e-2 * self.tstep:      # :188-201
            out.append(t)
            t += self.tstep
        return out

    # -- regularisation (:89-143)
    def _calcRegularization(self, u) -> float:
        acc = 0.0
        for i in range(self.N - 1):
            d = u[i + 1] - u[i]
            acc += d * d / self.tstep
        return self.gamma / 2.0 * acc

    def _calcRegularizationGrad(self, u) -> stdvec:
        N, g, t = self.N, self.gamma, self.tstep
        out = [-g * (-5.0 * u[1] + 4.0 * u[2] - u[3] + 2.0 * u[0]) / t]
        out += [-g * (u[i + 1] + u[i - 1] - 2.0 * u[i]) / t for i in range(1, N - 1)]
        out.append(-g * (-5.0 * u[N - 2] + 4.0 * u[N - 3] - u[N - 4] + 2.0 * u[N - 1]) / t)
        return out

    def _calcRegularizationHessian(self, u) -> np.ndarray:
        N = self.N
        H = np.zeros((N, N))
        got = self.gamma / self.tstep
        for i in range(1, N - 1):
            H[i, i - 1] = -got
            H[i, i + 1] = -got
            H[i, i] = 2.0 * got
        H[1, 0] = 0.0
        H[N - 2, N - 1] = 0.0
        return H

    # -- sweeps (:376-438)
    def _u(self, control) -> np.ndarray:
        u = np.ascontiguousarray(control, dtype=np.float64)
        assert u.size == self.N, "control must have N entries"
        return u

    def _calcPsi(self, control):
        u = self._u(control)
        _lib.check(self.lib.ocmps_forward_sweep(self.timeStepper.h, self.psi_init.h, _pd(u), self.N, self.psi_t.h))
        self.calculatedXi = False

    def _calcXi(self, control):
        u = self._u(control)
        _lib.check(self.lib.ocmps_backward_sweep(self.timeStepper.h, self.psi_target.h, _pd(u), self.N, self.xi_t.h))
        self.calculatedXi = True

    def _calcDivT(self):
        assert self.calculatedXi
        out = np.zeros(2 * self.N)
        _lib.check(self.lib.ocmps_store_divT(self.xi_t.h, self.psi_t.h, self.N, _pd(out)))
        self.divT = out.view(np.complex128).copy()

    def _calcPsiXiDivT(self, control):
        u = self._u(control)
        if self.threadCount > 1:      # the reference's two threads (:424-430) -> two CUDA streams
            _lib.check(self.lib.ocmps_sweep_pair(self.timeStepper.h, self.psi_init.h, self.psi_target.h, _pd(u), self.N,
                                                 self.psi_t.h, self.xi_t.h))
            self.calculatedXi = True
        else:
            self._calcPsi(u)
            self._calcXi(u)
        self._calcDivT()

    def _overlapFactor(self) -> complex:
        """overlapC(psi_t.back(), psi_target) (:242)."""
        out = np.zeros(2 * self.N)
        _lib.check(self.lib.ocmps_store_overlaps(self.psi_t.h, self.psi_target.h, self.N, _pd(out)))
        self._fid_ovl = out.view(np.complex128).copy()       # <target|psi_i> for all i
        return complex(np.conj(self._fid_ovl[-1]))

    # -- cost (:441-453)
    def _calcCost(self, control, new_control=True) -> float:
        if new_control:
            self.calculatedXi = False
            self._calcPsi(control)
        self._overlapFactor()
        ov = self._fid_ovl[-1]
        return 0.5 * (1.0 - (ov.real * ov.real + ov.imag * ov.imag)) + self._calcRegularization(control)

    # -- gradient (:205-249, :457-467)
    def _calcFidelityGrad(self, control, new_control=True) -> stdvec:
        if new_control:
            self.calculatedXi = False
            if self.BFGS:
                self._calcPsi(control)
            else:
                self._calcPsiXiDivT(control)
        if self.BFGS:
            u = self._u(control)
            out = np.zeros(2 * self.N)
            _lib.check(self.lib.ocmps_backward_sweep_divT(self.timeStepper.h, self.psi_target.h, _pd(u), self.N, self.psi_t.h, _pd(out)))
            self.divT = out.view(np.complex128).copy()
        elif not self.calculatedXi:
            self._calcXi(control)
            self._calcDivT()
        of = self._overlapFactor()
        return [self.tstep * (self.divT[i] * of * 1j).real for i in range(self.N)]

    def _calcAnalyticGradient(self, control, new_control=True) -> stdvec:
        fg = self._calcFidelityGrad(control, new_control)
        rg = self._calcRegularizationGrad(control)
        return [a + b for a, b in zip(fg, rg)]

    # -- Hessian (:252-372)
    def _calcHessian(self, control, new_control=True) -> np.ndarray:
        """calcHessian_parallel (:282-338).  The prerequisites the reference computes one after the other -- psi_t, xi_t
        and divT if the cache flags ask for them (:284-294), xiHlist (:300-303) -- and the rows (:305-335) go to the GPU as
        one event-ordered schedule (``ocmps_hessian_eval``); the cache flags end up as the reference leaves them."""
        if self.BFGS:
            raise RuntimeError("getHessian is undefined in BFGS mode (xi_t / xiHlist are not allocated)")
        do_psi = bool(new_control)
        do_xi = bool(new_control) or not self.calculatedXi
        u = self._u(control)
        N = self.N
        H = self._calcRegularizationHessian(control)
        if self.xiHlist is None:
            self.xiHlist = self.timeStepper.new_store(N)
        rows = np.array(list(range(1, N - 1)) if self.rows is None else list(self.rows), dtype=np.int32)
        ovl = np.zeros(2 * N * N)
        norms = np.zeros(N)
        divT = np.zeros(2 * N)
        fid = np.zeros(2 * N)
        nch = self.hessian_chains or max(1, min(64, 16 * self.threadCount))   # measured (Nt=201, chi=100): 12 -> much slower, 48 -> 8.84 s, 64 -> 8.43 s; the engine also bounds it by the free memory
        _lib.check(self.lib.ocmps_hessian_eval(self.timeStepper.h, self.psi_init.h, self.psi_target.h, _pd(u), N, self.psi_t.h,
                                               self.xi_t.h, self.xiHlist.h, _pi(rows), rows.size, nch, 1 if do_psi else 0,
                                               1 if do_xi else 0, _pd(divT), _pd(fid), _pd(ovl), _pd(norms)))
        self.calculatedXi = True
        self.divT = divT.view(np.complex128).copy()
        self._fid_ovl = fid.view(np.complex128).copy()
        of = complex(np.conj(self._fid_ovl[-1]))                                                            # :297
        ovl = ovl.view(np.complex128).reshape(N, N)
        ts2 = self.tstep * self.tstep
        Hf = np.zeros((N, N))
        dT = self.divT
        for r in rows:
            r = int(r)
            Hf[r, r] += ts2 * ((of * ovl[r, r]).real - (dT[r] * np.conj(dT[r])).real)                      # :260-264
            v = ts2 * ((of * ovl[r, r + 1:N - 1] * norms[r]).real - (dT[r] * np.conj(dT[r + 1:N - 1])).real)   # :272-277
            Hf[r, r + 1:N - 1] += v
            Hf[r + 1:N - 1, r] += v
        self._hessian_fidelity_part = Hf
        self._hessian_reg_part = H
        return H + Hf

    def _calcFidelityForAllT(self, control, new_control=True) -> stdvec:
        if new_control:
            self.calculatedXi = False
            self._calcPsi(control)
        self._overlapFactor()
        return [float(o.real * o.real + o.imag * o.imag) for o in self._fid_ovl]

    # -- public API (:495-589)
    def propagatePsi(self, control):
        self._calcPsi(control if self.GRAPE else self.basis.convertControl(control))

    def getCost(self, control, new_control: bool = True) -> float:
        if self.GRAPE:
            return self._calcCost(control, new_control)
        return self._calcCost(self.basis.convertControl(control, new_control), new_control)

    def getAnalyticGradient(self, control, new_control: bool = True) -> stdvec:
        if self.GRAPE:
            return self._calcAnalyticGradient(control, new_control)
        return self.basis.convertGradient(
            self._calcAnalyticGradient(self.basis.convertControl(control, new_control), new_control))

    def getHessian(self, control, new_control: bool = True):
        if self.GRAPE:
            return self._calcHessian(control, new_control).tolist()
        return self.basis.convertHessian(self._calcHessian(self.basis.convertControl(control, new_control), new_control))

    def getFidelityForAllT(self, control, new_control: bool = True) -> stdvec:
        if self.GRAPE:
            return self._calcFidelityForAllT(control, new_control)
        return self._calcFidelityForAllT(self.basis.convertControl(control, new_control), new_control)

    # <psi_i|H(u_i)|psi_i> / <psi_i|psi_i> along the ramp: the excess energy over the instantaneous ground state, and its variance.
    # Same caching as getFidelityForAllT: new_control=True re-propagates psi; with False the cached slices are kept and the
    # control passed only sets u_i.
    def _calcEnergyForAllT(self, control, new_control=True, variance=False):
        u = self._u(control)
        if new_control:
            self.calculatedXi = False
            self._calcPsi(u)
        return self.psi_t.energies(self.timeStepper.getJ(), u, 0, self.N, variance=variance)

    def getEnergyForAllT(self, control, new_control: bool = True) -> stdvec:
        u = control if self.GRAPE else self.basis.convertControl(control, new_control)
        return [float(e) for e in self._calcEnergyForAllT(u, new_control)]

    def getEnergyVarianceForAllT(self, control, new_control: bool = True) -> stdvec:
        u = control if self.GRAPE else self.basis.convertControl(control, new_control)
        return [float(v) for v in self._calcEnergyForAllT(u, new_control, variance=True)[1]]

    def getControlJacobian(self):
        if self.GRAPE:
            return np.eye(self.N).tolist()
        return self.basis.getControlJacobian()


def batch_cost_gradient(problems: Sequence["OptimalControl"], controls: Sequence[Sequence[float]]):
    """Cost and analytic gradient of several independent controls at once on one GPU (batched seeds of the north
    star).  ``problems[k]`` evaluates ``controls[k]``; all problems share one stepper and are in non-BFGS mode.  The
    2*len(problems) sweeps run concurrently on their own streams (``ocmps_sweep_batch``); each problem ends in exactly
    the state ``getAnalyticGradient(c, True); getCost(c, False)`` leaves it in.  Returns [(cost, gradient), ...]."""
    assert len(problems) == len(controls) and len(problems) >= 1
    st = problems[0].timeStepper
    N = problems[0].N
    us, starts, fwd, stores = [], [], [], []
    for p, c in zip(problems, controls):
        assert p.timeStepper is st and p.N == N and not p.BFGS
        u = np.ascontiguousarray(c if p.GRAPE else p.basis.convertControl(c, True), dtype=np.float64)
        assert u.size == N
        us += [u, u]
        starts += [p.psi_init.h, p.psi_target.h]
        fwd += [1, 0]
        stores += [p.psi_t.h, p.xi_t.h]
    n = len(starts)
    U = np.ascontiguousarray(np.stack(us))
    a_starts = (C.c_void_p * n)(*starts)
    a_stores = (C.c_void_p * n)(*stores)
    a_fwd = np.array(fwd, dtype=np.int32)
    _lib.check(st.ctx.lib.ocmps_sweep_batch(st.h, n, a_starts, _pi(a_fwd), _pd(U), N, a_stores))
    out = []
    for k, (p, c) in enumerate(zip(problems, controls)):
        u = us[2 * k]
        p.calculatedXi = True
        p._calcDivT()
        of = p._overlapFactor()
        fg = [p.tstep * (p.divT[i] * of * 1j).real for i in range(N)]
        g = [x + y for x, y in zip(fg, p._calcRegularizationGrad(u))]
        ov = p._fid_ovl[-1]
        cost = 0.5 * (1.0 - (ov.real * ov.real + ov.imag * ov.imag)) + p._calcRegularization(u)
        out.append((cost, g if p.GRAPE else p.basis.convertGradient(g)))
    return out
