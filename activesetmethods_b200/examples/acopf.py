"""AC optimal power flow (polar, "ACP") as a host-side NLP — the *user model* that sits above the hot path.

In the reference this layer is third-party Julia: PowerModels' ``build_opf`` on an ``ACPPowerModel`` driven
through JuMP's ``NLPEvaluator`` (reference ``examples/acopf/opf.jl:18-36``, ``test/opf.jl:6-22``).  It hands
the SLP driver exactly what ``src/MOI_wrapper.jl:1014-1156`` builds: bounds, the COO Jacobian pattern
``j_str`` (row-class order of ``MOI_wrapper.jl:683-689``: lin<=, lin>=, lin==, quad<=, quad>=, quad==, NLP),
a start point and the four callbacks ``eval_f / eval_grad_f / eval_g / eval_jac_g``.

Neither Julia nor PowerModels exist in this image, so this module restates that model in numpy.  It is an
input generator for tests and benchmarks, not part of the accelerated path: everything here runs on the
host exactly as the JuMP evaluator does in the reference.

Contents
  * ``parse_matpower``          – minimal MATPOWER ``.m`` reader (enough for ``examples/acopf/case3.m``)
  * ``CASE3_M`` / ``case9``     – the two small public networks (case3 is read from text, see tests)
  * ``synthetic_network``       – seeded generator matching the (bus, gen, branch) counts of the pegase cases
  * ``perturb_loads``           – load scenarios  pd,qd * (1 + 0.1 N(0,1)) clipped to +-30 %
  * ``branch_contingencies``    – N-1 scenarios: one network per non-islanding single-branch outage
  * ``generator_contingencies`` – one network per single-generator outage
  * ``AcopfModel``              – the NLP: sizes, bounds, ``j_str`` (1-based like the reference), callbacks

Variable order (PowerModels creation order): va[nb], vm[nb], pg[ng], qg[ng], p[2nl arcs], q[2nl arcs],
p_dc[2nd], q_dc[2nd].  Arc order: all "from" arcs then all "to" arcs (PowerModels ``arcs``).
Row order: angmax rows (lin<=), angmin rows (lin>=), theta_ref + dcline loss rows (lin==),
thermal limits from/to per branch (quad<=), P and Q balance per bus (quad==), Ohm rows
p_fr,q_fr,p_to,q_to per branch (NLP).
"""
from __future__ import annotations

import math
import re
from dataclasses import dataclass, field

import numpy as np

__all__ = [
    "Network", "parse_matpower", "case9", "synthetic_network", "perturb_loads", "AcopfModel",
    "PEGASE_SHAPES", "branch_contingencies", "generator_contingencies",
]

# (buses, gens, branches) of the named configs in BASELINE.json (SURVEY.md App. D)
PEGASE_SHAPES = {
    "case118": (118, 54, 186),
    "case1354pegase": (1354, 260, 1991),
    "case2869pegase": (2869, 510, 4582),
    "case13659pegase": (13659, 4092, 20467),
}


@dataclass
class Network:
    """Per-unit network data (already divided by baseMVA, angles in radians).

    ``br_status[nl]`` and ``gen_status[ng]`` are 0/1 like MATPOWER's BR_STATUS / GEN_STATUS and default to all in
    service.  ``parse_matpower`` drops the elements a file marks out of service, so the base network has only
    in-service elements; a status set to 0 afterwards (a contingency) keeps the element in the arrays, and
    ``AcopfModel`` keeps its variables, rows and Jacobian entries and takes it out of service by values and bounds
    only, so that every contingency of a network shares the base case's Jacobian pattern."""
    baseMVA: float
    # buses
    bus_id: np.ndarray
    pd: np.ndarray
    qd: np.ndarray
    gs: np.ndarray
    bs: np.ndarray
    vmin: np.ndarray
    vmax: np.ndarray
    ref_bus: int                      # index into bus arrays
    # generators
    gen_bus: np.ndarray
    pmin: np.ndarray
    pmax: np.ndarray
    qmin: np.ndarray
    qmax: np.ndarray
    cost2: np.ndarray                 # $/h per pu^2
    cost1: np.ndarray
    cost0: np.ndarray
    # branches
    f_bus: np.ndarray
    t_bus: np.ndarray
    br_r: np.ndarray
    br_x: np.ndarray
    br_b: np.ndarray
    tap: np.ndarray
    shift: np.ndarray
    rate_a: np.ndarray
    angmin: np.ndarray
    angmax: np.ndarray
    # dc lines
    dc_f: np.ndarray = field(default_factory=lambda: np.zeros(0, dtype=np.int64))
    dc_t: np.ndarray = field(default_factory=lambda: np.zeros(0, dtype=np.int64))
    dc_pminf: np.ndarray = field(default_factory=lambda: np.zeros(0))
    dc_pmaxf: np.ndarray = field(default_factory=lambda: np.zeros(0))
    dc_pmint: np.ndarray = field(default_factory=lambda: np.zeros(0))
    dc_pmaxt: np.ndarray = field(default_factory=lambda: np.zeros(0))
    dc_qminf: np.ndarray = field(default_factory=lambda: np.zeros(0))
    dc_qmaxf: np.ndarray = field(default_factory=lambda: np.zeros(0))
    dc_qmint: np.ndarray = field(default_factory=lambda: np.zeros(0))
    dc_qmaxt: np.ndarray = field(default_factory=lambda: np.zeros(0))
    dc_loss0: np.ndarray = field(default_factory=lambda: np.zeros(0))
    dc_loss1: np.ndarray = field(default_factory=lambda: np.zeros(0))
    # in-service flags (None: all in service)
    br_status: np.ndarray = None
    gen_status: np.ndarray = None

    def __post_init__(self):
        if self.br_status is None:
            self.br_status = np.ones(len(self.f_bus), dtype=np.int64)
        if self.gen_status is None:
            self.gen_status = np.ones(len(self.gen_bus), dtype=np.int64)

    @property
    def nb(self):
        return len(self.bus_id)

    @property
    def ng(self):
        return len(self.gen_bus)

    @property
    def nl(self):
        return len(self.f_bus)

    @property
    def nd(self):
        return len(self.dc_f)


# ----------------------------------------------------------------------------------------------------------
# MATPOWER reader
# ----------------------------------------------------------------------------------------------------------
def _matrix(text: str, name: str):
    m = re.search(r"mpc\." + name + r"\s*=\s*\[(.*?)\]", text, re.S)
    if m is None:
        return None
    rows = []
    for line in m.group(1).replace(";", "\n").splitlines():
        line = line.split("%")[0].strip()
        if line:
            rows.append([float(t) for t in line.split()])
    return rows


def parse_matpower(text: str) -> Network:
    """Read a MATPOWER v2 case (bus/gen/gencost/branch/dcline) and apply the data clean-ups PowerModels
    performs on load that matter for ``build_opf``: per-unit scaling, degrees→radians, tap 0 → 1,
    reference-bus selection when none is flagged (bus of the largest in-service generator), dcline flow
    bounds derived from pmin/pmax/loss terms, polynomial costs rescaled to per-unit."""
    base = float(re.search(r"mpc\.baseMVA\s*=\s*([0-9.eE+-]+)", text).group(1))
    bus = np.array(_matrix(text, "bus"), dtype=float)
    gen = np.array(_matrix(text, "gen"), dtype=float)
    branch = np.array(_matrix(text, "branch"), dtype=float)
    gencost_rows = _matrix(text, "gencost")
    dcl = _matrix(text, "dcline")

    bus = bus[bus[:, 1] != 4]
    ids = bus[:, 0].astype(np.int64)
    pos = {int(b): k for k, b in enumerate(ids)}
    gen_on = gen[:, 7] > 0
    br_on = branch[:, 10] > 0

    gen_u = gen[gen_on]
    gen_bus = np.array([pos[int(b)] for b in gen_u[:, 0]], dtype=np.int64)
    ng = len(gen_u)
    c2 = np.zeros(ng)
    c1 = np.zeros(ng)
    c0 = np.zeros(ng)
    if gencost_rows is not None:
        k = 0
        for row, on in zip(gencost_rows, gen_on):
            if not on:
                continue
            if int(row[0]) != 2:
                raise ValueError("only polynomial gencost is supported")
            ncoef = int(row[3])
            coef = row[4:4 + ncoef]
            coef = [0.0] * (3 - len(coef)) + list(coef[-3:])
            c2[k], c1[k], c0[k] = coef[0] * base * base, coef[1] * base, coef[2]
            k += 1

    ref = np.nonzero(bus[:, 1] == 3)[0]
    if len(ref) >= 1:
        ref_bus = int(ref[0])
    else:  # PowerModels picks the bus of the biggest generator
        ref_bus = int(gen_bus[int(np.argmax(gen_u[:, 8]))])

    br = branch[br_on]
    tap = br[:, 8].copy()
    tap[tap == 0.0] = 1.0
    angmin = np.deg2rad(br[:, 11]) if br.shape[1] > 11 else np.full(len(br), -math.pi / 3)
    angmax = np.deg2rad(br[:, 12]) if br.shape[1] > 12 else np.full(len(br), math.pi / 3)
    # PowerModels: angle differences outside +-90 deg (e.g. MATPOWER's +-360) are tightened to +-60 deg
    wide = (angmin <= -math.pi / 2) | (angmax >= math.pi / 2) | ((angmin == 0.0) & (angmax == 0.0))
    angmin = np.where(wide, -math.pi / 3, angmin)
    angmax = np.where(wide, math.pi / 3, angmax)
    rate_a = br[:, 5] / base
    if np.any(rate_a <= 0):
        raise ValueError("unrated branches are not supported by this reader")

    net = Network(
        baseMVA=base,
        bus_id=ids, pd=bus[:, 2] / base, qd=bus[:, 3] / base, gs=bus[:, 4] / base, bs=bus[:, 5] / base,
        vmin=bus[:, 12].copy(), vmax=bus[:, 11].copy(), ref_bus=ref_bus,
        gen_bus=gen_bus, pmin=gen_u[:, 9] / base, pmax=gen_u[:, 8] / base,
        qmin=gen_u[:, 4] / base, qmax=gen_u[:, 3] / base, cost2=c2, cost1=c1, cost0=c0,
        f_bus=np.array([pos[int(b)] for b in br[:, 0]], dtype=np.int64),
        t_bus=np.array([pos[int(b)] for b in br[:, 1]], dtype=np.int64),
        br_r=br[:, 2].copy(), br_x=br[:, 3].copy(), br_b=br[:, 4].copy(), tap=tap,
        shift=np.deg2rad(br[:, 9]), rate_a=rate_a, angmin=angmin, angmax=angmax,
    )
    if dcl:
        d = np.array([r for r in dcl if r[2] > 0], dtype=float)
        pmin, pmax = d[:, 9] / base, d[:, 10] / base
        loss0, loss1 = d[:, 15] / base, d[:, 16]
        pminf = np.empty(len(d)); pmaxf = np.empty(len(d)); pmint = np.empty(len(d)); pmaxt = np.empty(len(d))
        for k in range(len(d)):
            lo, hi, l0, l1 = pmin[k], pmax[k], loss0[k], loss1[k]
            if lo >= 0 and hi >= 0:
                pminf[k], pmaxf[k] = lo, hi
                pmint[k], pmaxt[k] = l0 - hi * (1 - l1), l0 - lo * (1 - l1)
            elif lo >= 0 > hi:
                pminf[k], pmint[k] = lo, hi
                pmaxf[k], pmaxt[k] = (-hi + l0) / (1 - l1), l0 - lo * (1 - l1)
            elif lo < 0 <= hi:
                pmaxt[k], pmaxf[k] = -lo, hi
                pminf[k], pmint[k] = (lo + l0) / (1 - l1), l0 - hi * (1 - l1)
            else:
                pmaxt[k], pmint[k] = -lo, hi
                pmaxf[k], pminf[k] = (-hi + l0) / (1 - l1), (lo + l0) / (1 - l1)
        net.dc_f = np.array([pos[int(b)] for b in d[:, 0]], dtype=np.int64)
        net.dc_t = np.array([pos[int(b)] for b in d[:, 1]], dtype=np.int64)
        net.dc_pminf, net.dc_pmaxf, net.dc_pmint, net.dc_pmaxt = pminf, pmaxf, pmint, pmaxt
        net.dc_qminf, net.dc_qmaxf = d[:, 11] / base, d[:, 12] / base
        net.dc_qmint, net.dc_qmaxt = d[:, 13] / base, d[:, 14] / base
        net.dc_loss0, net.dc_loss1 = loss0, loss1
    return net


_CASE9 = """
mpc.baseMVA = 100;
mpc.bus = [
 1 3 0 0 0 0 1 1 0 345 1 1.1 0.9;
 2 2 0 0 0 0 1 1 0 345 1 1.1 0.9;
 3 2 0 0 0 0 1 1 0 345 1 1.1 0.9;
 4 1 0 0 0 0 1 1 0 345 1 1.1 0.9;
 5 1 90 30 0 0 1 1 0 345 1 1.1 0.9;
 6 1 0 0 0 0 1 1 0 345 1 1.1 0.9;
 7 1 100 35 0 0 1 1 0 345 1 1.1 0.9;
 8 1 0 0 0 0 1 1 0 345 1 1.1 0.9;
 9 1 125 50 0 0 1 1 0 345 1 1.1 0.9;
];
mpc.gen = [
 1 72.3 27.03 300 -300 1.04 100 1 250 10;
 2 163 6.54 300 -300 1.025 100 1 300 10;
 3 85 -10.95 300 -300 1.025 100 1 270 10;
];
mpc.branch = [
 1 4 0 0.0576 0 250 250 250 0 0 1 -360 360;
 4 5 0.017 0.092 0.158 250 250 250 0 0 1 -360 360;
 5 6 0.039 0.17 0.358 150 150 150 0 0 1 -360 360;
 3 6 0 0.0586 0 300 300 300 0 0 1 -360 360;
 6 7 0.0119 0.1008 0.209 150 150 150 0 0 1 -360 360;
 7 8 0.0085 0.072 0.149 250 250 250 0 0 1 -360 360;
 8 2 0 0.0625 0 250 250 250 0 0 1 -360 360;
 8 9 0.032 0.161 0.306 250 250 250 0 0 1 -360 360;
 9 4 0.01 0.085 0.176 250 250 250 0 0 1 -360 360;
];
mpc.gencost = [
 2 1500 0 3 0.11 5 150;
 2 2000 0 3 0.085 1.2 600;
 2 3000 0 3 0.1225 1 335;
];
"""


def case9() -> Network:
    """The public 9-bus WSCC system (MATPOWER ``case9``); AC-OPF optimum 5296.69 $/h."""
    return parse_matpower(_CASE9)


# ----------------------------------------------------------------------------------------------------------
# Synthetic networks with the pegase shapes (the real files are not shipped with the reference)
# ----------------------------------------------------------------------------------------------------------
def synthetic_network(nb: int, ng: int, nl: int, seed: int | None = None) -> Network:
    """Seeded random network: spanning tree + extra local edges (plus a few long ties above 5000 buses, see below),
    log-normal impedances, loads on ~60 % of buses, generation capacity 1.8x load, quadratic costs, thermal ratings from a DC power flow
    (SURVEY.md §8(d) recipe).  ``seed`` defaults to the bus count."""
    rng = np.random.default_rng(nb if seed is None else seed)
    assert nl >= nb - 1
    # topology: random tree with locality (attach to a recent bus), then extra edges between near buses
    f = np.empty(nl, dtype=np.int64)
    t = np.empty(nl, dtype=np.int64)
    for k in range(1, nb):
        lo = max(0, k - 12)
        f[k - 1] = rng.integers(lo, k)
        t[k - 1] = k
    extra = nl - (nb - 1)
    a = rng.integers(0, nb, size=extra)
    off = rng.integers(2, 40, size=extra)
    if nb >= 5000:
        # continental grids have an extra-high-voltage backbone: without long ties the local windows above give a
        # chain-like graph whose hop diameter grows like nb / 35 (390 hops for 13 659 buses, against ~50 for the real
        # European cases); 2 % of the extra branches become ties of log-uniform length up to a quarter of the network
        long_tie = rng.random(extra) < 0.02
        off = np.where(long_tie, np.exp(rng.uniform(math.log(40.0), math.log(nb / 4.0), extra)).astype(np.int64), off)
    b = (a + off) % nb
    f[nb - 1:] = np.minimum(a, b)
    t[nb - 1:] = np.maximum(a, b)
    same = f == t
    t[same] = (f[same] + 1) % nb

    r = np.exp(rng.normal(math.log(0.01), 0.5, nl))
    x = np.exp(rng.normal(math.log(0.06), 0.5, nl))
    bch = rng.uniform(0.0, 0.05, nl)

    has_load = rng.random(nb) < 0.6
    pd = np.where(has_load, rng.uniform(0.05, 0.5, nb), 0.0)
    qd = 0.3 * pd

    gen_bus = np.sort(rng.choice(nb, size=ng, replace=(ng > nb)))
    share = rng.uniform(0.5, 1.5, ng)
    pmax = 1.8 * pd.sum() * share / share.sum()
    pmin = np.zeros(ng)
    qmax = 0.75 * pmax + 0.1
    qmin = -qmax
    c2 = rng.uniform(0.01, 0.12, ng) * 100.0      # the recipe's $/MW^2 h figures at baseMVA 100 ...
    c1 = rng.uniform(1.0, 5.0, ng) * 100.0        # ... expressed per unit
    c0 = np.zeros(ng)

    # DC power flow with generation proportional to capacity, to size the thermal ratings
    inj = -pd.copy()
    np.add.at(inj, gen_bus, pmax * (pd.sum() / pmax.sum()))
    import scipy.sparse as sp
    import scipy.sparse.linalg as spla
    w = 1.0 / x
    A = sp.coo_matrix((np.r_[w, w, -w, -w], (np.r_[f, t, f, t], np.r_[f, t, t, f])), shape=(nb, nb)).tocsc()
    keep = np.arange(1, nb)
    theta = np.zeros(nb)
    theta[keep] = spla.spsolve(A[keep][:, keep], inj[keep])
    flow = np.abs((theta[f] - theta[t]) * w)
    rate = np.maximum(1.5 * flow, 0.25) * 1.15 + 0.05

    return Network(
        baseMVA=100.0, bus_id=np.arange(1, nb + 1), pd=pd, qd=qd, gs=np.zeros(nb), bs=np.zeros(nb),
        vmin=np.full(nb, 0.9), vmax=np.full(nb, 1.1), ref_bus=int(gen_bus[int(np.argmax(pmax))]),
        gen_bus=gen_bus, pmin=pmin, pmax=pmax, qmin=qmin, qmax=qmax, cost2=c2, cost1=c1, cost0=c0,
        f_bus=f, t_bus=t, br_r=r, br_x=x, br_b=bch, tap=np.ones(nl), shift=np.zeros(nl), rate_a=rate,
        angmin=np.full(nl, -math.pi / 6), angmax=np.full(nl, math.pi / 6),
    )


def perturb_loads(net: Network, scenario: int, sigma: float = 0.1, clip: float = 0.3) -> Network:
    """Load scenario ``scenario`` (seed = scenario id): pd, qd scaled by 1 + sigma*N(0,1), clipped to +-clip."""
    import copy
    rng = np.random.default_rng(scenario)
    fac = 1.0 + np.clip(sigma * rng.standard_normal(net.nb), -clip, clip)
    out = copy.copy(net)
    out.pd = net.pd * fac
    out.qd = net.qd * fac
    return out


def _islands(net: Network, status: np.ndarray) -> bool:
    """True if the branches with ``status`` != 0 leave the network in more pieces than the base network's in-service
    branches do."""
    from scipy.sparse import coo_matrix
    from scipy.sparse.csgraph import connected_components

    def pieces(on):
        G = coo_matrix((np.ones(int(on.sum())), (net.f_bus[on], net.t_bus[on])), shape=(net.nb, net.nb))
        return connected_components(G, directed=False)[0]
    return pieces(status != 0) > pieces(net.br_status != 0)


def branch_contingencies(net: Network, count: int | None = None) -> list:
    """N-1 branch scenarios: one network per in-service branch whose outage does not island the network (the branch
    set out of service with ``br_status``), in branch order; the first ``count`` of them if given.  Copies ``net``
    like ``perturb_loads``; every scenario shares the base case's Jacobian pattern."""
    import copy
    out = []
    for l in np.nonzero(net.br_status != 0)[0]:
        if count is not None and len(out) == count:
            break
        status = net.br_status.copy()
        status[l] = 0
        if _islands(net, status):
            continue
        c = copy.copy(net)
        c.br_status = status
        out.append(c)
    return out


def generator_contingencies(net: Network) -> list:
    """One network per in-service generator with that generator out of service (``gen_status``), in generator order.
    Copies ``net`` like ``perturb_loads``."""
    import copy
    out = []
    for k in np.nonzero(net.gen_status != 0)[0]:
        c = copy.copy(net)
        c.gen_status = net.gen_status.copy()
        c.gen_status[k] = 0
        out.append(c)
    return out


def _angle_paths(net: Network, lines: np.ndarray) -> np.ndarray:
    """For each branch in ``lines``: the shortest path from its from-bus to its to-bus over the in-service branches,
    each weighted by the widest angle difference its rows allow, max(angmax, -angmin).  Summed along any in-service
    path, the angle-difference rows bound |va_f - va_t| by that length, so it is a bound the in-service network
    already implies.  Raises ValueError if the terminals are not connected: the outage islands the network."""
    from scipy.sparse import coo_matrix
    from scipy.sparse.csgraph import dijkstra
    on = net.br_status != 0
    a = np.minimum(net.f_bus, net.t_bus)[on]
    b = np.maximum(net.f_bus, net.t_bus)[on]
    w = np.maximum(net.angmax, -net.angmin)[on]
    # parallel branches: the smallest weight of each bus pair (a sparse matrix would add duplicates up)
    order = np.lexsort((w, b, a))
    a, b, w = a[order], b[order], w[order]
    first = np.ones(len(a), dtype=bool)
    first[1:] = (a[1:] != a[:-1]) | (b[1:] != b[:-1])
    G = coo_matrix((w[first], (a[first], b[first])), shape=(net.nb, net.nb)).tocsr()
    src = np.unique(net.f_bus[lines])
    dist = dijkstra(G, directed=False, indices=src)
    d = dist[np.searchsorted(src, net.f_bus[lines]), net.t_bus[lines]]
    cut = ~np.isfinite(d)
    if cut.any():
        l = int(lines[np.argmax(cut)])
        raise ValueError(f"the outage of branch {l} (buses {net.bus_id[net.f_bus[l]]}-{net.bus_id[net.t_bus[l]]}) "
                         "islands the network: islanding contingencies are not supported")
    return d


# ----------------------------------------------------------------------------------------------------------
# The NLP
# ----------------------------------------------------------------------------------------------------------
class AcopfModel:
    """ACP-polar OPF as (n, m, bounds, j_str, callbacks) — the tuple ``Model(...)`` receives at
    reference ``src/MOI_wrapper.jl:1093-1099``.  ``j_str`` is an (nnz, 2) int64 array of **1-based**
    (row, col) pairs, like the reference's ``Vector{Tuple{Int64,Int64}}`` (``src/model.jl:10``).

    Out-of-service elements (``Network.br_status`` / ``gen_status`` = 0) change values and bounds only: ``n``, ``m``
    and ``j_str`` are those of the all-in-service network.
      * branch: its 12 admittance coefficients are 0, so its Ohm rows read p = 0, q = 0 on both arcs and the arcs drop
        out of the balance rows by value.  Its thermal rows and flow bounds stay (inactive at zero flow).  Its angle-
        difference rows are relaxed to +- the shortest in-service path between its terminals (``_angle_paths``): a
        bound the rest of the network implies, so the feasible set is that of the network without the branch, and the
        rows stay bounded (a free row is not accepted by the sub-LP builder).  An outage that islands the network
        raises ValueError.
      * generator: pmin = pmax = qmin = qmax = 0.  Its ``cost0`` stays in the objective as a constant (costs are
        shared by a batch), so compare objectives with the network without it after subtracting that constant."""

    def __init__(self, net: Network, start: str = "midpoint"):
        self.net = net
        nb, ng, nl, nd = net.nb, net.ng, net.nl, net.nd
        self.nb, self.ng, self.nl, self.nd = nb, ng, nl, nd
        # variable offsets
        o = 0
        self.o_va = o; o += nb
        self.o_vm = o; o += nb
        self.o_pg = o; o += ng
        self.o_qg = o; o += ng
        self.o_p = o; o += 2 * nl        # from arcs [0,nl), to arcs [nl,2nl)
        self.o_q = o; o += 2 * nl
        self.o_pdc = o; o += 2 * nd
        self.o_qdc = o; o += 2 * nd
        self.n = o
        # row offsets
        r = 0
        self.r_angmax = r; r += nl
        self.r_angmin = r; r += nl
        self.r_ref = r; r += 1
        self.r_dc = r; r += nd
        self.r_thermal = r; r += 2 * nl   # per branch: from, to
        self.r_bal = r; r += 2 * nb       # per bus: P, Q
        self.r_ohm = r; r += 4 * nl       # per branch: p_fr, q_fr, p_to, q_to
        self.m = r

        # admittance terms (PowerModels calc_branch_y / calc_branch_t)
        z2 = net.br_r ** 2 + net.br_x ** 2
        g = net.br_r / z2
        b = -net.br_x / z2
        tr = net.tap * np.cos(net.shift)
        ti = net.tap * np.sin(net.shift)
        tm2 = net.tap ** 2
        half_b = net.br_b / 2.0
        on = net.br_status != 0
        cf = dict(
            a_pf=(g + 0.0) / tm2, b_pf=(-g * tr + b * ti) / tm2, c_pf=(-b * tr - g * ti) / tm2,
            a_qf=-(b + half_b) / tm2, b_qf=-(-b * tr - g * ti) / tm2, c_qf=(-g * tr + b * ti) / tm2,
            a_pt=(g + 0.0), b_pt=(-g * tr - b * ti) / tm2, c_pt=(-b * tr + g * ti) / tm2,
            a_qt=-(b + half_b), b_qt=-(-b * tr + g * ti) / tm2, c_qt=(-g * tr - b * ti) / tm2,
        )
        self._cf = {k: np.where(on, v, 0.0) for k, v in cf.items()}

        # bounds
        inf = np.inf
        xl = np.full(self.n, -inf)
        xu = np.full(self.n, inf)
        xl[self.o_vm:self.o_vm + nb] = net.vmin; xu[self.o_vm:self.o_vm + nb] = net.vmax
        gon = net.gen_status != 0
        xl[self.o_pg:self.o_pg + ng] = np.where(gon, net.pmin, 0.0); xu[self.o_pg:self.o_pg + ng] = np.where(gon, net.pmax, 0.0)
        xl[self.o_qg:self.o_qg + ng] = np.where(gon, net.qmin, 0.0); xu[self.o_qg:self.o_qg + ng] = np.where(gon, net.qmax, 0.0)
        ra2 = np.r_[net.rate_a, net.rate_a]
        xl[self.o_p:self.o_p + 2 * nl] = -ra2; xu[self.o_p:self.o_p + 2 * nl] = ra2
        xl[self.o_q:self.o_q + 2 * nl] = -ra2; xu[self.o_q:self.o_q + 2 * nl] = ra2
        if nd:
            xl[self.o_pdc:self.o_pdc + 2 * nd] = np.r_[net.dc_pminf, net.dc_pmint]
            xu[self.o_pdc:self.o_pdc + 2 * nd] = np.r_[net.dc_pmaxf, net.dc_pmaxt]
            xl[self.o_qdc:self.o_qdc + 2 * nd] = np.r_[net.dc_qminf, net.dc_qmint]
            xu[self.o_qdc:self.o_qdc + 2 * nd] = np.r_[net.dc_qmaxf, net.dc_qmaxt]
        self.x_L, self.x_U = xl, xu

        gl = np.full(self.m, -inf)
        gu = np.full(self.m, inf)
        gu[self.r_angmax:self.r_angmax + nl] = net.angmax
        gl[self.r_angmin:self.r_angmin + nl] = net.angmin
        out = np.nonzero(~on)[0]
        if len(out):
            d = _angle_paths(net, out)
            gu[self.r_angmax + out] = d
            gl[self.r_angmin + out] = -d
        gl[self.r_ref] = gu[self.r_ref] = 0.0
        if nd:
            gl[self.r_dc:self.r_dc + nd] = gu[self.r_dc:self.r_dc + nd] = net.dc_loss0
        gu[self.r_thermal:self.r_thermal + 2 * nl] = np.repeat(net.rate_a ** 2, 2)
        gl[self.r_bal:self.r_bal + 2 * nb:2] = gu[self.r_bal:self.r_bal + 2 * nb:2] = -net.pd
        gl[self.r_bal + 1:self.r_bal + 2 * nb:2] = gu[self.r_bal + 1:self.r_bal + 2 * nb:2] = -net.qd
        gl[self.r_ohm:] = 0.0
        gu[self.r_ohm:] = 0.0
        self.g_L, self.g_U = gl, gu

        self._build_pattern()

        # start point (reference examples/acopf/init_opf.jl:25-29: midpoint of the bounds where both
        # exist; PowerModels' own defaults otherwise: va = 0, vm = 1, everything else 0)
        x0 = np.zeros(self.n)
        x0[self.o_vm:self.o_vm + nb] = 1.0
        if start == "midpoint":
            both = np.isfinite(xl) & np.isfinite(xu)
            x0[both] = 0.5 * (xl[both] + xu[both])
        self.x0 = x0

    # -- sparsity ------------------------------------------------------------------------------------------
    def _build_pattern(self):
        net = self.net
        nb, ng, nl, nd = self.nb, self.ng, self.nl, self.nd
        f, t = net.f_bus, net.t_bus
        rows = []
        cols = []
        br = np.arange(nl)

        def add(r, c):
            rows.append(np.asarray(r, dtype=np.int64).ravel())
            cols.append(np.asarray(c, dtype=np.int64).ravel())

        # lin<= / lin>= : va_f - va_t
        add(np.stack([self.r_angmax + br] * 2, 1), np.stack([self.o_va + f, self.o_va + t], 1))
        add(np.stack([self.r_angmin + br] * 2, 1), np.stack([self.o_va + f, self.o_va + t], 1))
        # lin== : theta_ref, dcline losses (1-loss1) p_f + p_t = loss0
        add([self.r_ref], [self.o_va + net.ref_bus])
        if nd:
            d = np.arange(nd)
            add(np.stack([self.r_dc + d] * 2, 1), np.stack([self.o_pdc + d, self.o_pdc + nd + d], 1))
        # quad<= thermal limits: p^2 + q^2 <= rate^2, rows (from_l, to_l) per branch
        rt = self.r_thermal + 2 * br
        add(np.stack([rt, rt, rt + 1, rt + 1], 1),
            np.stack([self.o_p + br, self.o_q + br, self.o_p + nl + br, self.o_q + nl + br], 1))
        self._nnz_fixed_end = sum(len(r) for r in rows)

        # quad== balances.  Affine part: arcs at the bus (from arcs then to arcs, by branch index),
        # dc arcs, generators; quadratic part: vm_i^2 (only when a shunt is present).
        arcs_of = [[] for _ in range(nb)]
        for l in range(nl):
            arcs_of[f[l]].append(l)
        for l in range(nl):
            arcs_of[t[l]].append(nl + l)
        dcs_of = [[] for _ in range(nb)]
        for d in range(nd):
            dcs_of[net.dc_f[d]].append(d)
        for d in range(nd):
            dcs_of[net.dc_t[d]].append(nd + d)
        gens_of = [[] for _ in range(nb)]
        for k in range(ng):
            gens_of[net.gen_bus[k]].append(k)
        bal_rows = []
        bal_cols = []
        bal_coef = []          # constant coefficient, or nan for the vm^2 slot
        bal_shunt = []         # (position, bus, is_q)
        pos = 0
        for i in range(nb):
            for is_q in (0, 1):
                row = self.r_bal + 2 * i + is_q
                oa = self.o_q if is_q else self.o_p
                od = self.o_qdc if is_q else self.o_pdc
                og = self.o_qg if is_q else self.o_pg
                for a in arcs_of[i]:
                    bal_rows.append(row); bal_cols.append(oa + a); bal_coef.append(1.0); pos += 1
                for a in dcs_of[i]:
                    bal_rows.append(row); bal_cols.append(od + a); bal_coef.append(1.0); pos += 1
                for k in gens_of[i]:
                    bal_rows.append(row); bal_cols.append(og + k); bal_coef.append(-1.0); pos += 1
                sh = net.bs[i] if is_q else net.gs[i]
                if sh != 0.0:
                    bal_rows.append(row); bal_cols.append(self.o_vm + i); bal_coef.append(np.nan)
                    bal_shunt.append((pos, i, is_q)); pos += 1
        add(bal_rows, bal_cols)
        self._bal_coef = np.array(bal_coef, dtype=float)
        self._bal_shunt = bal_shunt
        self._bal_rows = np.array(bal_rows, dtype=np.int64)
        self._bal_cols = np.array(bal_cols, dtype=np.int64)
        self._nnz_bal = len(bal_rows)

        # NLP Ohm rows: [p_arc, vm_f, vm_t, va_f, va_t]
        ro = self.r_ohm + 4 * br
        vmf, vmt, vaf, vat = self.o_vm + f, self.o_vm + t, self.o_va + f, self.o_va + t
        oc = np.stack([
            np.stack([self.o_p + br, vmf, vmt, vaf, vat], 1),
            np.stack([self.o_q + br, vmf, vmt, vaf, vat], 1),
            np.stack([self.o_p + nl + br, vmf, vmt, vaf, vat], 1),
            np.stack([self.o_q + nl + br, vmf, vmt, vaf, vat], 1)], 1)           # (nl, 4, 5)
        orow = np.repeat(np.stack([ro, ro + 1, ro + 2, ro + 3], 1)[:, :, None], 5, axis=2)
        add(orow, oc)

        rows = np.concatenate(rows)
        cols = np.concatenate(cols)
        self.j_str = np.stack([rows + 1, cols + 1], 1)       # 1-based, like the reference
        self.nnz = len(rows)

    # -- callbacks -----------------------------------------------------------------------------------------
    def eval_f(self, x):
        pg = x[self.o_pg:self.o_pg + self.ng]
        net = self.net
        return float(np.sum(net.cost2 * pg * pg + net.cost1 * pg + net.cost0))

    def eval_grad_f(self, x, grad):
        pg = x[self.o_pg:self.o_pg + self.ng]
        grad[:] = 0.0
        grad[self.o_pg:self.o_pg + self.ng] = 2.0 * self.net.cost2 * pg + self.net.cost1
        return grad

    def _flows(self, x):
        net, c = self.net, self._cf
        va = x[self.o_va:self.o_va + self.nb]
        vm = x[self.o_vm:self.o_vm + self.nb]
        f, t = net.f_bus, net.t_bus
        vf, vt = vm[f], vm[t]
        d = va[f] - va[t]
        return vf, vt, np.cos(d), np.sin(d), c

    def eval_g(self, x, g):
        net = self.net
        nb, nl, nd = self.nb, self.nl, self.nd
        va = x[self.o_va:self.o_va + nb]
        vm = x[self.o_vm:self.o_vm + nb]
        f, t = net.f_bus, net.t_bus
        dva = va[f] - va[t]
        g[self.r_angmax:self.r_angmax + nl] = dva
        g[self.r_angmin:self.r_angmin + nl] = dva
        g[self.r_ref] = va[net.ref_bus]
        if nd:
            pdc = x[self.o_pdc:self.o_pdc + 2 * nd]
            g[self.r_dc:self.r_dc + nd] = (1.0 - net.dc_loss1) * pdc[:nd] + pdc[nd:]
        p = x[self.o_p:self.o_p + 2 * nl]
        q = x[self.o_q:self.o_q + 2 * nl]
        s2 = p * p + q * q
        g[self.r_thermal:self.r_thermal + 2 * nl:2] = s2[:nl]
        g[self.r_thermal + 1:self.r_thermal + 2 * nl:2] = s2[nl:]
        # balances
        vals = np.where(np.isnan(self._bal_coef), 0.0, self._bal_coef) * x[self._bal_cols]
        bal = np.bincount(self._bal_rows - self.r_bal, weights=vals, minlength=2 * nb)
        bal[0::2] += net.gs * vm * vm
        bal[1::2] -= net.bs * vm * vm
        g[self.r_bal:self.r_bal + 2 * nb] = bal
        # Ohm rows: arc flow minus its expression in (vm, va)
        vf, vt, cs, sn, c = self._flows(x)
        vv = vf * vt
        pf = c["a_pf"] * vf * vf + c["b_pf"] * vv * cs + c["c_pf"] * vv * sn
        qf = c["a_qf"] * vf * vf + c["b_qf"] * vv * cs + c["c_qf"] * vv * sn
        pt = c["a_pt"] * vt * vt + c["b_pt"] * vv * cs - c["c_pt"] * vv * sn
        qt = c["a_qt"] * vt * vt + c["b_qt"] * vv * cs - c["c_qt"] * vv * sn
        ro = self.r_ohm
        g[ro:ro + 4 * nl:4] = p[:nl] - pf
        g[ro + 1:ro + 4 * nl:4] = q[:nl] - qf
        g[ro + 2:ro + 4 * nl:4] = p[nl:] - pt
        g[ro + 3:ro + 4 * nl:4] = q[nl:] - qt
        return g

    def eval_jac_g(self, x, mode, rows, cols, values):
        """Reference callback signature ``eval_jac_g(x, mode, rows, cols, values)``
        (``src/MOI_wrapper.jl:1059-1069``): ``mode == "Structure"`` fills 1-based rows/cols,
        anything else fills ``values`` (length nnz, ``j_str`` order)."""
        if mode == "Structure":
            rows[:] = self.j_str[:, 0]
            cols[:] = self.j_str[:, 1]
            return
        net = self.net
        nb, nl, nd = self.nb, self.nl, self.nd
        k = 0
        v = values
        blk = np.empty((nl, 2)); blk[:, 0] = 1.0; blk[:, 1] = -1.0
        v[k:k + 2 * nl] = blk.ravel(); k += 2 * nl
        v[k:k + 2 * nl] = blk.ravel(); k += 2 * nl
        v[k] = 1.0; k += 1
        if nd:
            d = np.empty((nd, 2)); d[:, 0] = 1.0 - net.dc_loss1; d[:, 1] = 1.0
            v[k:k + 2 * nd] = d.ravel(); k += 2 * nd
        p = x[self.o_p:self.o_p + 2 * nl]
        q = x[self.o_q:self.o_q + 2 * nl]
        th = np.stack([2.0 * p[:nl], 2.0 * q[:nl], 2.0 * p[nl:], 2.0 * q[nl:]], 1)
        v[k:k + 4 * nl] = th.ravel(); k += 4 * nl
        bal = self._bal_coef.copy()
        vm = x[self.o_vm:self.o_vm + nb]
        for pos, i, is_q in self._bal_shunt:
            bal[pos] = (-2.0 * net.bs[i] if is_q else 2.0 * net.gs[i]) * vm[i]
        v[k:k + self._nnz_bal] = bal; k += self._nnz_bal
        vf, vt, cs, sn, c = self._flows(x)
        vv = vf * vt
        J = np.empty((nl, 4, 5))
        J[:, :, 0] = 1.0
        # d/dvm_f, d/dvm_t, d/dva_f, d/dva_t of -(expr)
        for r, (a, bb, cc, own_from, sgn) in enumerate((
                (c["a_pf"], c["b_pf"], c["c_pf"], True, 1.0), (c["a_qf"], c["b_qf"], c["c_qf"], True, 1.0),
                (c["a_pt"], c["b_pt"], c["c_pt"], False, -1.0), (c["a_qt"], c["b_qt"], c["c_qt"], False, -1.0))):
            # expr = a*v_own^2 + bb*vv*cos(d) + sgn*cc*vv*sin(d),  d = va_f - va_t
            cross = bb * cs + sgn * cc * sn
            if own_from:
                J[:, r, 1] = -(2.0 * a * vf + cross * vt)
                J[:, r, 2] = -(cross * vf)
            else:
                J[:, r, 1] = -(cross * vt)
                J[:, r, 2] = -(2.0 * a * vt + cross * vf)
            dd = vv * (-bb * sn + sgn * cc * cs)
            J[:, r, 3] = -dd
            J[:, r, 4] = dd
        v[k:k + 20 * nl] = J.ravel(); k += 20 * nl
        assert k == self.nnz
        return values


class AcrModel:
    """The same OPF in rectangular voltage coordinates ("ACR", PowerModels' ``ACRPowerModel``, one of the formulations
    the reference's example builds: ``examples/acopf/opf.jl:18-21``).  Every row and the objective are affine or
    quadratic in (vr, vi), so the model is a ``qcqp.QcqpModel`` and runs on the device-side QCQP evaluator with no
    formulation-specific kernel.  Built by ``AcrModel(net)``, which returns the ``QcqpModel``.

    Variables: vr[nb], vi[nb] (bounds +-vmax) in the slots of AcopfModel's va, vm; then pg, qg, p, q, p_dc, q_dc with
    AcopfModel's order, bounds and costs.
    Row order (attributes ``r_*`` of the returned model):
      angmax[nl]   (vi_f vr_t - vr_f vi_t) - tan(angmax) (vr_f vr_t + vi_f vi_t) <= 0
      angmin[nl]   (vi_f vr_t - vr_f vi_t) - tan(angmin) (vr_f vr_t + vi_f vi_t) >= 0
                   (exact: the reader keeps every limit inside (-90, 90) degrees)
      ref          vi_ref = 0
      dc[nd]       (1 - loss1) p_dc_f + p_dc_t = loss0
      vm[nb]       vmin^2 <= vr^2 + vi^2 <= vmax^2
      thermal[2nl] p^2 + q^2 <= rate^2 per branch, from then to
      balance[2nb] P, Q per bus: AcopfModel's affine terms, shunt gs (vr^2 + vi^2), -bs (vr^2 + vi^2)
      ohm[4nl]     p_fr, q_fr, p_to, q_to per branch: the arc flow minus AcopfModel's expression with the same 12
                   coefficients, vm_f vm_t cos(va_f - va_t) -> vr_f vr_t + vi_f vi_t and
                   vm_f vm_t sin(va_f - va_t) -> vi_f vr_t - vr_f vi_t.
    Start: vr at the midpoint of [vmin, vmax] and vi = 0 (AcopfModel's start as a physical point; the midpoint of the
    +-vmax box would be the all-zero voltage, where every Ohm row's Jacobian vanishes); the rest as AcopfModel.
    Out-of-service generators enter through the bounds; an out-of-service branch raises ValueError (its zero
    coefficients would change the term lists, which the device evaluator shares over a batch)."""

    def __new__(cls, net: Network):
        from .qcqp import QcqpModel
        if np.any(net.br_status == 0):
            raise ValueError("AcrModel: out-of-service branches are not supported (the term lists are shared by a batch)")
        P = AcopfModel(net)
        nb, ng, nl, nd = P.nb, P.ng, P.nl, P.nd
        cf = P._cf
        o_vr, o_vi = 0, nb
        f, t = np.asarray(net.f_bus, dtype=np.int64), np.asarray(net.t_bus, dtype=np.int64)
        br = np.arange(nl)
        x_L, x_U = P.x_L.copy(), P.x_U.copy()
        x_L[:2 * nb] = -np.tile(net.vmax, 2)
        x_U[:2 * nb] = np.tile(net.vmax, 2)
        x0 = P.x0.copy()
        x0[:nb] = 0.5 * (net.vmin + net.vmax)
        x0[nb:2 * nb] = 0.0
        inf = np.inf
        r = 0
        r_angmax = r; r += nl
        r_angmin = r; r += nl
        r_ref = r; r += 1
        r_dc = r; r += nd
        r_vm = r; r += nb
        r_thermal = r; r += 2 * nl
        r_bal = r; r += 2 * nb
        r_ohm = r; r += 4 * nl
        m = r
        gl, gu = np.full(m, -inf), np.full(m, inf)
        gu[r_angmax:r_angmax + nl] = 0.0
        gl[r_angmin:r_angmin + nl] = 0.0
        gl[r_ref] = gu[r_ref] = 0.0
        if nd:
            gl[r_dc:r_dc + nd] = gu[r_dc:r_dc + nd] = net.dc_loss0
        gl[r_vm:r_vm + nb] = net.vmin ** 2
        gu[r_vm:r_vm + nb] = net.vmax ** 2
        gu[r_thermal:r_thermal + 2 * nl] = np.repeat(net.rate_a ** 2, 2)
        gl[r_bal:r_bal + 2 * nb:2] = gu[r_bal:r_bal + 2 * nb:2] = -net.pd
        gl[r_bal + 1:r_bal + 2 * nb:2] = gu[r_bal + 1:r_bal + 2 * nb:2] = -net.qd
        gl[r_ohm:] = gu[r_ohm:] = 0.0

        A = ([], [], [])          # affine terms: row, col, coef
        Q = ([], [], [], [])      # quadratic terms: row, i, j, coef

        def aff(row, col, coef):
            for lst, v in zip(A, (row, col, coef)):
                lst.append(np.asarray(v).reshape(-1))

        def quad(row, i, j, coef):
            for lst, v in zip(Q, (row, i, j, coef)):
                lst.append(np.asarray(v).reshape(-1))

        vrf, vrt, vif, vit = o_vr + f, o_vr + t, o_vi + f, o_vi + t

        def cols(*a):             # per-branch columns interleaved term by term
            return np.stack(a, 1)
        for r0, lim in ((r_angmax, net.angmax), (r_angmin, net.angmin)):
            ta = np.tan(lim)
            rows = np.repeat(r0 + br, 4)
            quad(rows, cols(vif, vrf, vrf, vif), cols(vrt, vit, vrt, vit),
                 cols(np.ones(nl), -np.ones(nl), -ta, -ta))
        aff([r_ref], [o_vi + net.ref_bus], [1.0])
        if nd:
            d = np.arange(nd)
            aff(np.repeat(r_dc + d, 2), cols(P.o_pdc + d, P.o_pdc + nd + d), cols(1.0 - net.dc_loss1, np.ones(nd)))
        bus = np.arange(nb)
        quad(np.repeat(r_vm + bus, 2), cols(o_vr + bus, o_vi + bus), cols(o_vr + bus, o_vi + bus), np.ones(2 * nb))
        rt = np.stack([r_thermal + 2 * br, r_thermal + 2 * br + 1], 1)
        quad(np.repeat(rt.reshape(-1), 2),
             cols(P.o_p + br, P.o_q + br, P.o_p + nl + br, P.o_q + nl + br).reshape(nl, 2, 2),
             cols(P.o_p + br, P.o_q + br, P.o_p + nl + br, P.o_q + nl + br).reshape(nl, 2, 2), np.ones(4 * nl))
        # balances: AcopfModel's affine terms in its order, the shunt on vr^2 + vi^2
        lin = ~np.isnan(P._bal_coef)
        aff(P._bal_rows[lin] - P.r_bal + r_bal, P._bal_cols[lin], P._bal_coef[lin])
        for i in range(nb):
            for is_q, sh in ((0, net.gs[i]), (1, -net.bs[i])):
                if sh != 0.0:
                    quad([r_bal + 2 * i + is_q] * 2, [o_vr + i, o_vi + i], [o_vr + i, o_vi + i], [sh, sh])
        # Ohm rows: arc - (a v_own^2 + b (vr_f vr_t + vi_f vi_t) + sg c (vi_f vr_t - vr_f vi_t))
        for k, (key, arc, own_f, sg) in enumerate((("pf", P.o_p + br, True, 1.0), ("qf", P.o_q + br, True, 1.0),
                                                   ("pt", P.o_p + nl + br, False, -1.0),
                                                   ("qt", P.o_q + nl + br, False, -1.0))):
            a, b, c = cf["a_" + key], cf["b_" + key], cf["c_" + key]
            row = r_ohm + 4 * br + k
            own_r, own_i = (vrf, vif) if own_f else (vrt, vit)
            aff(row, arc, np.ones(nl))
            quad(np.repeat(row, 6), cols(own_r, own_i, vrf, vif, vif, vrf), cols(own_r, own_i, vrt, vit, vrt, vit),
                 cols(-a, -a, -b, -b, -sg * c, sg * c))
        cat = lambda lst, dt: np.concatenate(lst).astype(dt) if lst else np.zeros(0, dt)   # noqa: E731
        a_row, a_col, a_coef = cat(A[0], np.int64), cat(A[1], np.int64), cat(A[2], float)
        q_row, q_i, q_j, q_coef = cat(Q[0], np.int64), cat(Q[1], np.int64), cat(Q[2], np.int64), cat(Q[3], float)
        # terms of one row must stay together in the order listed above: sort rows stably
        oa, oq = np.argsort(a_row, kind="stable"), np.argsort(q_row, kind="stable")
        pg = P.o_pg + np.arange(ng)
        mdl = QcqpModel(P.n, x_L, x_U, gl, gu, x0, obj_const=float(np.sum(net.cost0)),
                        obj_aff=(pg, net.cost1), obj_quad=(pg, pg, net.cost2),
                        aff=(a_row[oa], a_col[oa], a_coef[oa]), quad=(q_row[oq], q_i[oq], q_j[oq], q_coef[oq]))
        mdl.net = net
        mdl.nb, mdl.ng, mdl.nl, mdl.nd = nb, ng, nl, nd
        mdl.o_vr, mdl.o_vi = o_vr, o_vi
        for name in ("o_pg", "o_qg", "o_p", "o_q", "o_pdc", "o_qdc"):
            setattr(mdl, name, getattr(P, name))
        mdl.r_angmax, mdl.r_angmin, mdl.r_ref, mdl.r_dc, mdl.r_vm = r_angmax, r_angmin, r_ref, r_dc, r_vm
        mdl.r_thermal, mdl.r_bal, mdl.r_ohm = r_thermal, r_bal, r_ohm
        return mdl
