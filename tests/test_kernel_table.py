"""The kernel instantiation tables read as data (no device).

Every batch path of the library is a template instantiation picked from a table by tableau width, CTA shape and
memory layout: `k_simplex<NWC, KC, resident, NWR>` (csrc/ktab_base.cu, ktab_split_{a,b,c}.cu, both layouts of every
entry), `k_simplex_cluster<NW, KC, NWR, grid>` (ktab_cluster.cu, each entry as KC and as KG) and `k_bnb<NWC, KC, NWR>`
(ktab_bnb.cu).  This module parses those tables, restates the host rules that choose an entry (pick_kernel,
choose_route for a forced path, plan_cluster, plan_gridres, bnb_config_for) and the shared-memory carve-ups they
consult, and derives from the table data alone the width window and the tallest tableau of every entry.  It also
builds the inputs of tests/test_gpu_kernel_table.py -- which forces every entry on a B200 and checks by kernel name
that exactly that instantiation ran -- and runs the oracle side of every one of those cases here, so their shapes,
statuses and runtimes are known without a device.
"""
import math
import os
import re
from collections import namedtuple

import numpy as np
import pytest

from conftest import ROOT

CSRC = os.path.join(ROOT, "yalps_b200", "csrc")
SIMPLEX_FILES = ("ktab_base.cu", "ktab_split_a.cu", "ktab_split_b.cu", "ktab_split_c.cu")
B200_SMEM_OPTIN = 232448  # cudaDevAttrMaxSharedMemoryPerBlockOptin of a B200 (227 KB)
B200_SMS = 148
PATH_SMEM, PATH_GMEM = 1, 2  # enum yalps_path (include/yalps_b200.h)
TOO_LARGE = -3               # YALPS_ERR_TOO_LARGE
KMAX_CLUSTER = 16            # cluster_kernel.cuh kMaxCluster
KBNB_MAX_CUTS = 96           # bnb_kernel.cuh kBnbMaxCuts
STATIC_SMEM = 16             # static shared memory of k_simplex and k_simplex_cluster (ptxas -v: "16 bytes smem")

Entry = namedtuple("Entry", "nwc kc nwr")


# ------------------------------------------------------------------------------------------------ the tables
def parse_macro_uses(fname, macro):
    """The argument tuples of every use of `macro(...)` in csrc/<fname> (its #define line excluded), and the number of
    uses -- a use with an argument that is not a plain integer is counted but not parsed."""
    with open(os.path.join(CSRC, fname)) as f:
        src = f.read()
    src = re.sub(r"//[^\n]*", "", src)
    src = re.sub(r"#\s*define[^\n]*", "", src)
    uses = len(re.findall(rf"\b{macro}\s*\(", src))
    tuples = [tuple(int(x) for x in m.group(1).split(","))
              for m in re.finditer(rf"\b{macro}\s*\(\s*(\d+(?:\s*,\s*\d+)*)\s*\)", src)]
    return tuples, uses


def simplex_table():
    """k_simplex entries in the order all_kernels() (yalps_b200.cu) concatenates the four files."""
    out = []
    for fname in SIMPLEX_FILES:
        tuples, _ = parse_macro_uses(fname, "KENTRY")
        out += [Entry(t[0], t[1], t[2] if len(t) == 3 else 1) for t in tuples]
    return out


def cluster_table():
    return [Entry(*t) for t in parse_macro_uses("ktab_cluster.cu", "KENTRY")[0]]


def bnb_table():
    return [Entry(*t) for t in parse_macro_uses("ktab_bnb.cu", "BENTRY")[0]]


def simplex_name(e, resident):
    return f"k_simplex<{e.nwc},{e.kc},{int(resident)},{e.nwr}>"


def cluster_name(e, grid):
    return f"k_simplex_cluster<{e.nwc},{e.kc},{e.nwr},{int(grid)}>"


def bnb_name(e):
    return f"k_bnb<{e.nwc},{e.kc},{e.nwr}>"


def all_instantiations():
    """Every kernel the three tables instantiate, by canonical name."""
    names = [simplex_name(e, r) for e in simplex_table() for r in (True, False)]
    names += [cluster_name(e, g) for e in cluster_table() for g in (False, True)]
    names += [bnb_name(e) for e in bnb_table()]
    return names


_KNAME = re.compile(r"\b(k_simplex_cluster|k_simplex|k_bnb)<([^>]*)>")


def canonical_kernel_name(name):
    """A demangled kernel name as the profiler reports it ('void yalps::k_simplex<1, 2, true, 4>(yalps::BatchArgs)',
    or with '(int)1'/'(bool)1' casts) -> 'k_simplex<1,2,1,4>'; None for a kernel outside the three tables."""
    m = _KNAME.search(name)
    if not m:
        return None
    args = []
    for a in m.group(2).split(","):
        a = re.sub(r"^\(\w+\)", "", a.strip())
        args.append({"true": "1", "false": "0"}.get(a, a))
    return f"{m.group(1)}<{','.join(args)}>"


# ------------------------------------------------------------------------------------------------ carve-ups
def ld_for(W):
    """SmemLayout::ld_for (kernels.cuh): even row stride >= W+1 whose half is odd."""
    ld = (W - 1 + 2 + 1) & ~1
    if ((ld >> 1) & 1) == 0:
        ld += 2
    return ld


class SmemLayout:
    """Restatement of `SmemLayout` (yalps_b200/csrc/kernels.cuh:72-111), the shared-memory carve-up of k_simplex that
    the host checks against the device's opt-in limit: the resident tableau (Hcap rows of ld_for(Wcap) doubles), the
    pivot-column staging (colbuf/colnew) or, for the row-split kernels, the compacted row list (cc, list, cnt), the
    misc cells, the cross-warp reduction slots (nw > 1), variableAtPosition (resident or split) and the RHS column of
    the HBM/L2-resident split kernels."""

    def __init__(self, Hcap, Wcap, resident, nw, split=False):
        o = 0
        self.ldA = ld_for(Wcap)
        if resident:
            o += Hcap * self.ldA * 8
        if split:
            o += (Hcap + 8) * 16
            o += ((Hcap + 3) & ~3) * 4
            o += 16
        else:
            o += ((Hcap + 7) & ~7) * 8
            if not resident:
                o += ((Hcap + 1) & ~1) * 8
        o += 16
        if nw > 1:
            o += 192 * 4
        if resident or split:
            o += (Wcap + Hcap) * 4
        o = (o + 15) & ~15
        if not resident and split:
            o += ((Hcap + 1) & ~1) * 8
        self.total = (o + 15) & ~15


class ClusterSmem:
    """Restatement of `ClusterSmem` (cluster_kernel.cuh): rows 1..H-1 dealt over C CTAs, Hloc rows per CTA."""

    def __init__(self, Hcap, Wcap, C):
        ld = ld_for(Wcap)
        self.Hloc = hloc = (Hcap - 1 + C - 1) // C
        o = hloc * ld * 8 + 2 * ld * 8 + (hloc + 8) * 16 + ((hloc + 3) & ~3) * 4 + 16 + 32 + 192 * 4
        o += 2 * KMAX_CLUSTER * 16 + (Wcap + Hcap) * 4
        self.total = (o + 15) & ~15


def update_rows(e, vw):
    """RU, the height of the straight-line rank-1 update block: pivot_cta (simplex_device.cuh) for one row group,
    simplex_cta_split (simplex_split.cuh) for the row-split kernels."""
    if e.nwr == 1:
        return 8 if e.kc == 1 else (4 if e.kc == 2 else (2 if e.kc <= 4 else 1))
    if vw == 1:
        return 1 if e.kc >= 8 else 8 // e.kc
    return 1 if e.kc >= 4 else 4 // e.kc


# ------------------------------------------------------------------------------------------------ the host rules
def cap_of(e, vw):
    """Coefficient columns the pivot-row registers of an entry cover: 32 * NWC * KC * VW >= W-1 is required."""
    return 32 * e.nwc * e.kc * vw


def simplex_window(e, vw, table=None):
    """(prev, cap): the entry serves prev < W-1 <= cap.  prev is the largest cap of an entry with the same NWC and NWR
    and a smaller KC (0 if there is none) -- pick_kernel takes the smallest covering KC."""
    table = table or simplex_table()
    prev = max([cap_of(o, vw) for o in table if o.nwc == e.nwc and o.nwr == e.nwr and o.kc < e.kc], default=0)
    return prev, cap_of(e, vw)


def pick_kernel(nwc_want, nwr, W, resident, table):
    """pick_kernel (yalps_b200.cu): among the entries with `nwr` row groups that cover the row, the smallest NWC >=
    nwc_want (else the largest NWC), then the smallest KC."""
    vw = 2 if resident else 1
    wm1 = max(W - 1, 1)
    best = None
    for k in table:
        if k.nwr != nwr or cap_of(k, vw) < wm1:
            continue
        if best is None:
            best = k
            continue
        k_ok, b_ok = k.nwc >= nwc_want, best.nwc >= nwc_want
        if k_ok != b_ok:
            if k_ok:
                best = k
            continue
        if k_ok:
            if k.nwc < best.nwc or (k.nwc == best.nwc and k.kc < best.kc):
                best = k
        elif k.nwc > best.nwc or (k.nwc == best.nwc and k.kc < best.kc):
            best = k
    return best


def forced_route(path, threads, rows, H, W, optin=B200_SMEM_OPTIN, table=None):
    """choose_route (yalps_b200.cu) for a batch forced onto the k_simplex table: set_tuning(PATH_SMEM or PATH_GMEM,
    threads, rows).  Returns (kernel name, shared memory bytes) or TOO_LARGE.  The staging checks use the 32-warp
    carve-up against the opt-in limit; the chosen kernel's own carve-up must also leave room for its static shared
    memory.  (The occupancy query is taken to succeed whenever that holds.)"""
    table = table or simplex_table()
    resident = SmemLayout(H, W, True, 32).total <= optin
    if path == PATH_SMEM and not resident:
        return TOO_LARGE
    if path == PATH_GMEM:
        resident = False
    if not resident and SmemLayout(H, W, False, 32).total > optin:
        return TOO_LARGE
    nw = max(1, threads // 32)
    nwr = rows if rows > 0 else 1
    k = None
    if nwr > 1:
        k = pick_kernel(max(1, nw // nwr), nwr, W, resident, table)
        if k and SmemLayout(H, W, resident, k.nwc * k.nwr, True).total > optin - STATIC_SMEM:
            k = None
    if k is None:
        k = pick_kernel(nw, 1, W, resident, table)
        if k and SmemLayout(H, W, resident, k.nwc, False).total > optin - STATIC_SMEM:
            return TOO_LARGE
    if k is None:
        return TOO_LARGE
    return simplex_name(k, resident), SmemLayout(H, W, resident, k.nwc * k.nwr, k.nwr > 1).total


def forcing(e, resident):
    """set_tuning arguments that force entry e: (path, threads per LP, row groups)."""
    return (PATH_SMEM if resident else PATH_GMEM), 32 * e.nwc * e.nwr, e.nwr


def tallest_height(e, resident, W, optin=B200_SMEM_OPTIN):
    """The tallest H for which the forced path of e still runs e at width W (0 if none does)."""
    path, threads, rows = forcing(e, resident)
    want = simplex_name(e, resident)

    def runs(H):
        r = forced_route(path, threads, rows, H, W, optin)
        return r != TOO_LARGE and r[0] == want

    if not runs(1):
        return 0
    lo, hi = 1, 1 << 16
    while lo < hi:  # runs() is monotone: taller tableaus only ever need more shared memory
        mid = (lo + hi + 1) // 2
        if runs(mid):
            lo = mid
        else:
            hi = mid - 1
    return lo


def first_covering_window(table, i, vw=2):
    """plan_cluster / bnb_config_for: the first entry whose cap covers W-1.  Entry i serves max(cap of the entries
    before it) < W-1 <= cap_i (an empty window when an earlier entry is at least as wide)."""
    prev = max([cap_of(o, vw) for o in table[:i]], default=0)
    return prev, cap_of(table[i], vw)


def narrowest_covering_window(table, i, vw=2):
    """plan_gridres: the narrowest covering cap, ties to the CTA with more threads (then the first).  (prev, cap), or
    None when another entry wins every width of i."""
    cap = cap_of(table[i], vw)
    for j, o in enumerate(table):
        if j != i and cap_of(o, vw) == cap:
            ti, tj = table[i].nwc * table[i].nwr, o.nwc * o.nwr
            if tj > ti or (tj == ti and j < i):
                return None
    return max([cap_of(o, vw) for o in table if cap_of(o, vw) < cap], default=0), cap


def plan_cluster(H, W, optin=B200_SMEM_OPTIN):
    """plan_cluster (yalps_b200.cu): (cluster entry, C) or None.  The smallest C of 2, 4, 8, 16 whose carve-up fits,
    skipping C < 16 while a CTA would own more than 40 rows.  (Co-scheduling is taken to succeed.)"""
    tab = cluster_table()
    k = next((e for e in tab if cap_of(e, 2) >= max(W - 1, 1)), None)
    if k is None:
        return None
    C = 2
    while C <= KMAX_CLUSTER:
        L = ClusterSmem(H, W, C)
        if L.total <= optin - STATIC_SMEM and not (L.Hloc > 40 and C < KMAX_CLUSTER):
            return k, C
        C *= 2
    return None


def plan_gridres(H, W, optin=B200_SMEM_OPTIN, sms=B200_SMS):
    """plan_gridres (yalps_b200.cu): (cluster entry run as KG, CTAs) or None."""
    tab = cluster_table()
    k = None
    for e in tab:
        cap, threads = cap_of(e, 2), e.nwc * e.nwr * 32
        if cap < max(W - 1, 1) or threads > 512:
            continue
        if k is None or cap < cap_of(k, 2) or (cap == cap_of(k, 2) and threads > k.nwc * k.nwr * 32):
            k = e
    if k is None:
        return None
    C = max(1, min(min(sms, 160), H - 1))
    if ClusterSmem(H, W, C).total > optin - STATIC_SMEM:
        return None
    return k, C


def bnb_config_for(W):
    """bnb_config_for (ktab_bnb.cu): the first config with 32 * NWC * KC * 2 >= W-1."""
    return next((c for c in bnb_table() if cap_of(c, 2) >= W - 1), None)


def bnb_cut_capacity(H, W, nints, optin=B200_SMEM_OPTIN):
    """Cut rows a node may carry in the device-resident search (bnb.inl:464-467), or None when the search does not
    go to the device kernel at all."""
    cfg = bnb_config_for(W)
    if cfg is None:
        return None
    nw = cfg.nwc * cfg.nwr
    room = optin - 4096
    extra = min(2 * nints, KBNB_MAX_CUTS)
    while extra >= 8 and SmemLayout(H + extra, W, True, nw, True).total > room:
        extra -= 8
    if extra < min(2 * nints, 8):
        return None
    return extra


# ------------------------------------------------------------------------------------------------ the cases
CHVATAL = np.array([[0, 10, -57, -9, -24], [0, 0.5, -5.5, -2.5, 9], [0, 0.5, -1.5, -0.5, 1], [1, 1, 0, 0, 0]], float)
KINDS = ("dense", "boundary", "sparse", "special", "infeasible", "unbounded")


def edge_batch(H, W, seed, n=12):
    """n synthetic H x W tableaus edited so that the trajectories reach the edges of a kernel's shape class, LP i of
    kind KINDS[i % 6]:
      dense       the generator's LP (phase 1 on a third of the rows);
      boundary    column W-1 has the largest objective cell, so the last coefficient column enters first;
      sparse      85 % of the constraint cells zeroed: partial updates, row skips;
      special     signed zeros, 1e-16 and 1.0000000000000001e-16 (either side of the flush threshold) in the last two
                  coefficient columns -- the last vector-column of the resident layout;
      infeasible  the most negative RHS on a row without a negative coefficient;
      unbounded   column W-1 enters and has no positive cell."""
    from oracle import lib as O
    m, nv = H - 1, W - 1
    mats = O.generate_synthetic(seed, n, m, nv, m // 3).reshape(n, H, W)
    rng = np.random.default_rng(seed)
    for i in range(n):
        t = mats[i]
        kind = KINDS[i % len(KINDS)]
        if kind == "boundary" and nv >= 1:
            t[0, W - 1] = t[0, 1:].max() + 0.5
            if m >= 1:
                t[1 + (i % m), W - 1] = abs(t[1 + (i % m), W - 1]) + 1.0
        elif kind == "sparse" and m >= 1:
            t[1:, 1:] *= rng.random((m, nv)) < 0.15
        elif kind == "special" and m >= 1:
            vals = [-0.0, 1e-16, 1.0000000000000001e-16, 0.0, -1e-16, -1.0000000000000001e-16]
            for r in range(1, H):
                for c in (W - 2, W - 1):
                    if c >= 1 and (r + c) % 2 == 0:
                        t[r, c] = vals[(r * 3 + c) % len(vals)]
            t[0, W - 1] = -0.0 if i % 4 else 1.0000000000000001e-16
        elif kind == "infeasible" and m >= 1:
            r = 1 + (i % m)
            t[r, 1:] = np.abs(t[r, 1:])
            t[r, 0] = -1e3
        elif kind == "unbounded" and nv >= 1:
            t[0, W - 1] = t[0, 1:].max() + 1.0
            t[1:, 0] = np.abs(t[1:, 0])  # phase 2 at once
            t[1:, W - 1] = -np.abs(t[1:, W - 1])
            if m >= 2:
                t[m, W - 1] = -0.0
    return np.ascontiguousarray(mats.reshape(n, H * W))


def chvatal_batch(H, W, seed):
    """The Chvatal cycling LP embedded in an H x W tableau: its three constraint rows in the last three rows, its four
    columns in the last four, everything else zero -- the cycle runs through the boundary column.  Followed by one
    copy in the first rows and columns and two edge_batch LPs.  (A tableau of fewer than 4 rows or 5 columns cannot
    hold it: four edge_batch LPs then.)"""
    out = edge_batch(H, W, seed, 4).reshape(4, H, W)
    if H >= 4 and W >= 5:
        out[:2] = 0.0
        rows, cols = [0, H - 3, H - 2, H - 1], [0, W - 4, W - 3, W - 2, W - 1]
        out[0][np.ix_(rows, cols)] = CHVATAL
        out[1][:4, :5] = CHVATAL
    return np.ascontiguousarray(out.reshape(4, H * W))


def budget_shape(c):
    """The maxPivots batch: the tallest of the cases at the wide edge."""
    W = max(w for _, w in c["shapes"])
    return max(h for h, w in c["shapes"] if w == W), W


def cycle_shape(e, resident):
    """The checkCycles batch: the narrowest width of the window that holds the Chvatal LP, 4 rows if they fit."""
    prev, cap = simplex_window(e, 2 if resident else 1)
    W = min(max(prev + 2, 5), cap + 1)
    return min(max(4, update_rows(e, 2 if resident else 1)), tallest_height(e, resident, W)), W


def queue_shape(c):
    """The queue-mode batch (more LPs than CTAs): the smallest case."""
    return min(c["shapes"], key=lambda s: s[0] * s[1])


def tall_tableau(H, W, seed):
    """One sparse H x W tableau for the tallest shapes (up to ~10^8 cells): a phase-1 pivot, then column W-1 enters and
    the last row leaves; a scatter of positive cells and special values in the last columns.  Sparse, so that the
    oracle's pivots skip almost every row."""
    rng = np.random.default_rng(seed)
    t = np.zeros((H, W))
    t[1:, 0] = 2.0 + rng.random(H - 1)
    rr = np.arange(1, H)
    t[rr, 1 + rng.integers(0, W - 1, H - 1)] = rng.random(H - 1) + 0.25
    t[0, W - 1] = 1.0
    if W > 2:
        t[0, 1] = -0.5
    if H > 3:
        t[1:H:max(1, H // 7), W - 1] = 1.0
    if H > 3 and W > 2:
        t[H - 2, 0] = -1.0
        t[H - 2, 1] = -1.0
    t[H - 1, 0] = 1.0
    t[H - 1, W - 1] = 4.0
    if W > 2:
        t[H - 1, W - 2] = -0.0
        t[max(1, H - 3), W - 2] = 1.0000000000000001e-16
        t[max(1, H - 4), W - 2] = 1e-16
    return t.reshape(1, H * W)


def simplex_cases(e, resident, optin=B200_SMEM_OPTIN):
    """The shapes test_gpu_kernel_table runs entry e on: both edges of its width window (W-1 = cap: every lane's last
    vector-column full; W-1 = prev+1: the first width that needs this KC, odd, so the resident layout's padding cell
    is live), each with the heights H = 2 (H-1 < RU), RU and 3*RU ((H-1) mod RU = RU-1) that fit at that width --
    at the widest resident widths only H = 1 does --, and the tallest H at the narrow edge."""
    vw = 2 if resident else 1
    prev, cap = simplex_window(e, vw)
    ru = update_rows(e, vw)
    shapes = []
    for W in (cap + 1, prev + 2):
        tallest = tallest_height(e, resident, W, optin)
        hs = sorted({h for h in (2, max(2, ru), 3 * ru) if h <= tallest}) or [tallest]
        shapes += [(H, W) for H in hs]
    tall = tallest_height(e, resident, prev + 2, optin)
    return {"shapes": shapes, "ru": ru, "window": (prev, cap), "tall": (tall, prev + 2)}


SIMPLEX_ENTRIES = [(e, r) for e in simplex_table() for r in (True, False)]


def entry_id(p):
    e, r = p
    return simplex_name(e, r)


def oracle_batch(mats, H, W, **kw):
    """Oracle outputs, the final tableaus and the reduced vectors the kernels write with want_duals."""
    from oracle import lib as O
    from yalps_b200.sensitivity import reduced_from_tableau
    work = mats.copy()
    res = O.simplex_batch(work, W, H, **kw)
    res["matrices"] = work
    res["reduced"] = np.stack([reduced_from_tableau(work[i], W, H, res["pos"][i]) for i in range(work.shape[0])])
    return res


# ------------------------------------------------------------------------------------------------ MILPs for k_bnb
def knapsack_milp(nvars, ncons, seed, max_iterations=None):
    """A seeded MILP in model form: maximise a positive profit over `nvars` integer variables under `ncons` <=
    constraints with positive weights (every variable appears in every constraint), plus one bound per variable's
    pair.  Its root tableau is (ncons + 1) x (nvars + 1)."""
    rng = np.random.default_rng(seed)
    w = rng.integers(5, 60, (ncons, nvars))
    p = rng.integers(10, 100, nvars)
    cap = (w.sum(axis=1) // 7).astype(int)
    variables = []
    for j in range(nvars):
        coefs = [("profit", float(p[j]))] + [(f"c{i}", float(w[i, j])) for i in range(ncons)]
        variables.append((f"x{j}", coefs))
    model = {"direction": "maximize", "objective": "profit",
             "constraints": [(f"c{i}", {"max": float(cap[i])}) for i in range(ncons)],
             "variables": variables, "integers": [f"x{j}" for j in range(nvars)]}
    options = {} if max_iterations is None else {"maxIterations": max_iterations}
    return model, options


# (name, variables, constraints, seed, maxIterations): one MILP per k_bnb config window of width, and one whose cut depth
# passes the device's cut-row capacity at its width
BNB_CASES = [("bnb<4,1,4>", 180, 12, 3, 60), ("bnb<4,2,4>", 300, 10, 5, 40), ("deep", 512, 40, 1, 400)]


# ================================================================================================ tests
def test_every_macro_use_is_parsed():
    """A new table entry cannot be missed: every KENTRY/BENTRY use parses to a tuple."""
    counts = {}
    for fname, macro, arity in [(f, "KENTRY", 2 if f == "ktab_base.cu" else 3) for f in SIMPLEX_FILES] + [
            ("ktab_cluster.cu", "KENTRY", 3), ("ktab_bnb.cu", "BENTRY", 3)]:
        tuples, uses = parse_macro_uses(fname, macro)
        assert len(tuples) == uses and uses > 0, fname
        assert all(len(t) == arity for t in tuples), fname
        assert len(set(tuples)) == len(tuples), f"{fname}: duplicate entry"
        counts[fname] = uses
    assert sum(counts[f] for f in SIMPLEX_FILES) == len(simplex_table()) == 52
    assert len(cluster_table()) == 6 and len(bnb_table()) == 3
    names = all_instantiations()
    assert len(names) == len(set(names)) == 104 + 12 + 3


def test_profiler_names_parse():
    assert canonical_kernel_name("void yalps::k_simplex<1, 2, true, 4>(yalps::BatchArgs)") == "k_simplex<1,2,1,4>"
    assert canonical_kernel_name("void yalps::k_simplex<(int)8, (int)8, (bool)0, (int)1>(yalps::BatchArgs)") == \
        "k_simplex<8,8,0,1>"
    assert canonical_kernel_name("void yalps::k_simplex_cluster<8, 4, 1, false>(yalps::BatchArgs)") == \
        "k_simplex_cluster<8,4,1,0>"
    assert canonical_kernel_name("void yalps::k_bnb<4, 2, 4>(yalps::BnbArgs)") == "k_bnb<4,2,4>"
    assert canonical_kernel_name("void yalps::k_simplex_tmem<2, true, false>(yalps::BatchArgs)") is None
    assert canonical_kernel_name("yalps::k_simplex_grid(yalps::GridArgs)") is None


def test_smem_layout_restatement_is_pinned_to_design():
    """DESIGN section 3: the 33x65 tableau, one warp, resident: ldA = 66, 18.2 KB per CTA (18,160 B)."""
    L = SmemLayout(33, 65, True, 1)
    assert L.ldA == 66 and L.total == 18160
    for W in range(2, 600):
        ld = ld_for(W)
        assert ld % 2 == 0 and (ld // 2) % 2 == 1 and ld >= W + 1


@pytest.mark.parametrize("p", SIMPLEX_ENTRIES, ids=entry_id)
def test_every_simplex_entry_has_a_window_and_a_height(p):
    """Both edges of the width window select the entry under its forcing, up to the tallest H; one row more selects
    another instantiation or nothing."""
    e, resident = p
    c = simplex_cases(e, resident)
    prev, cap = c["window"]
    assert prev < cap
    path, threads, rows = forcing(e, resident)
    want = simplex_name(e, resident)
    assert {W for _, W in c["shapes"]} == {cap + 1, prev + 2}
    for H, W in c["shapes"]:
        assert H >= 1 and prev < W - 1 <= cap
        r = forced_route(path, threads, rows, H, W)
        assert r != TOO_LARGE and r[0] == want, (W, H, r)
    tall, W = c["tall"]
    assert tall >= max(H for H, w in c["shapes"] if w == W)
    assert forced_route(path, threads, rows, tall, W)[0] == want
    after = forced_route(path, threads, rows, tall + 1, W)
    assert after == TOO_LARGE or after[0] != want


def test_split_entries_at_capacity_fall_back_to_one_row_group():
    """choose_route: a row-split entry whose carve-up does not fit runs the one-row-group kernel in its place."""
    fell_back = 0
    for e, resident in SIMPLEX_ENTRIES:
        if e.nwr == 1:
            continue
        tall, W = simplex_cases(e, resident)["tall"]
        after = forced_route(*forcing(e, resident), tall + 1, W)
        if after != TOO_LARGE:
            assert after[0].endswith(",1>"), (e, resident, after)
            fell_back += 1
    assert fell_back > 0


def test_cluster_and_grid_windows():
    tab = cluster_table()
    for i, e in enumerate(tab):
        prev, cap = first_covering_window(tab, i)
        assert prev < cap, e
        assert narrowest_covering_window(tab, i) == (prev, cap), e
        for W in (prev + 2, cap + 1):
            assert plan_cluster(3, W)[0] == e and plan_gridres(3, W)[0] == e
    for i, e in enumerate(bnb_table()):
        prev, cap = first_covering_window(bnb_table(), i)
        assert prev < cap and bnb_config_for(cap + 1) == e and bnb_config_for(prev + 2) == e


def cluster_cases():
    """(entry, W, H, expected C) for the KC runs: both width edges of every entry, and heights that give every
    cluster size at least once."""
    tab = cluster_table()
    out = []
    for i, e in enumerate(tab):
        prev, cap = first_covering_window(tab, i)
        for j, W in enumerate((prev + 2, cap + 1)):
            for H in ((20, 100) if j == 0 else (40, 200)) + ((400,) if i == 0 and j == 0 else ()):
                plan = plan_cluster(H, W)
                if plan is None:
                    continue
                out.append((e, W, H, plan[1]))
    return out


def test_cluster_cases_cover_every_cluster_size():
    cases = cluster_cases()
    assert {C for *_, C in cases} == {2, 4, 8, 16}
    assert {e for e, *_ in cases} == set(cluster_table())


def test_oracle_side_of_the_simplex_cases():
    """The inputs reach the edges: each statuses is seen, the boundary column enters, special cells are present."""
    from oracle import lib as O
    seen, entered = set(), 0
    for e, resident in SIMPLEX_ENTRIES:
        c = simplex_cases(e, resident)
        for H, W in c["shapes"]:
            exp = oracle_batch(edge_batch(H, W, 17 * W + H), H, W)
            seen |= set(exp["status"].tolist())
            entered += int((exp["pos"][:, W - 1] >= W).any())
        H, W = budget_shape(c)
        seen |= set(oracle_batch(edge_batch(H, W, 5), H, W, max_pivots=2)["status"].tolist())
        H, W = cycle_shape(e, resident)
        exp = oracle_batch(chvatal_batch(H, W, 3), H, W, check_cycles=True)
        if H >= 4:  # checkCycles stops the cycle wherever it sits
            assert exp["status"][0] == 4 and exp["status"][1] == 4, (e, resident, H, W)
    assert {0, 1, 2, 4} <= seen
    assert entered > 100


def test_oracle_side_of_the_tall_cases():
    """The tallest shapes pivot through phase 1 and phase 2 with the last row leaving; their cell counts bound the
    memory the GPU test needs."""
    from oracle import lib as O
    cells = []
    for e, resident in SIMPLEX_ENTRIES:
        tall, W = simplex_cases(e, resident)["tall"]
        cells.append(tall * W)
        if tall * W > 4_000_000:
            continue  # same generator, cheaper shapes suffice here
        m = tall_tableau(tall, W, 1)
        exp = oracle_batch(m, tall, W)
        assert exp["status"][0] == 0 and exp["pivots"][0, 1] >= 1, (e, resident, exp["status"], exp["pivots"])
    assert max(cells) < 80_000_000


def test_bnb_cases_fall_in_the_config_windows():
    """The generated MILPs: root widths in the <4,1,4> and <4,2,4> windows, a search with nodes, and one search whose
    cut depth passes the device's cut-row capacity at its width."""
    from oracle import model as M
    for name, nv, nc, seed, iters in BNB_CASES:
        model, options = knapsack_milp(nv, nc, seed, iters)
        tm = M.tableau_model(model)
        W, H = tm.tableau.width, tm.tableau.height
        cfg = bnb_config_for(W)
        info = {}
        M.solve(model, {**M.DEFAULT_OPTIONS, **options}, info)
        assert info["nodes"] > 0, name
        capacity = bnb_cut_capacity(H, W, len(tm.integers))
        assert capacity is not None, name
        if name == "deep":
            assert info["max_cuts"] > capacity, (info["max_cuts"], capacity)
        else:
            assert bnb_name(cfg) == name.replace("bnb", "k_bnb") and info["max_cuts"] <= capacity, (name, info["max_cuts"])
