"""Plain-Python mirror of how the persistent fused GMRES kernel (csrc/gmres_fused.cu) splits a solve over ranks and CTAs.

Host side, gmres_fused_solve (csrc/gmres.cu): bemb200_partition gives every rank its row slab; inside the slab the G CTAs
of the rank get

* "units"   -- CTA boundaries at (row, segment) granularity, shares proportional to the measured speeds (equal before the
               calibration), when the slab has at least 4 G rows, every CTA keeps two whole rows and no CTA needs more than
               256 row slots (head fragment included);
* "row_off" -- whole-row shares proportional to the measured speeds, when the unit table was refused, speeds are known and
               the slab has at least 8 G rows;
* "equal"   -- S = ceil(nloc / G) rows each;

then rblk = fused_pick_rblk(S) rows per matvec pass and fused_smem_bytes(S, rblk, restart) bytes of dynamic shared memory,
over 200 KB of which (or with a restart above FUSED_MAX_RESTART) the solve is "not fused" and takes the per-iteration
kernels.  Device side, the kernel decodes the table into (rb, sc, head fragment, s0, s1) per CTA and matvec_rows visits,
pass by pass and segment by segment, a range of row slots.  `matvec_work` replays that loop so a test can check that every
(row, segment) of the slab is computed exactly once and that every fragment wait has its producer.
"""
from __future__ import annotations

import math
from dataclasses import dataclass, field
from typing import List, Optional, Sequence

FUSED_THREADS = 512
NW = FUSED_THREADS // 32
FUSED_KMAX = 160
FUSED_MAX_RESTART = 63
FUSED_SEGMENT_WIDTH = FUSED_THREADS * 4
SMEM_LIMIT = 200 * 1024
CPLX = 16
MAX_PEERS = 8


def bemb200_partition(n: int, nranks: int, rank: int):
    """api.cu bemb200_partition: block rows [b, e) of rank `rank`."""
    chunk = (n + nranks - 1) // nranks
    b = min(chunk * rank, n)
    e = min(b + chunk, n)
    return b, e


def fused_pick_rblk(S: int) -> int:
    r = min(S, 256)
    return r if r else 1


def fused_smem_bytes(S: int, rblk: int, restart: int) -> int:
    m, m1 = restart, restart + 1

    def al(b):
        return (b + 15) & ~15

    yb = max(rblk * NW * 2 * 8, FUSED_THREADS * CPLX)
    t = al(yb) + 2 * al(S * CPLX) + 2 * al(FUSED_KMAX * CPLX) + al((FUSED_THREADS + 32) * CPLX) + al(FUSED_KMAX * CPLX)
    t += 2 * al((m1 * m // 2 + 1) * CPLX) + 2 * al(m1 * CPLX) + 2 * al((m1 + 1) * CPLX) + al(m1 * CPLX)
    return t


def _llround(x: float) -> int:
    """std::llround for x >= 0: halfway cases away from zero (Python's round() rounds them to even)."""
    f = math.floor(x)
    return f + 1 if x - f >= 0.5 else f


@dataclass
class RankPlan:
    rank: int
    row0: int
    nloc: int
    mode: str                   # "equal" | "units" | "row_off" | "not fused"
    S: int = 0
    rblk: int = 0
    smem: int = 0
    nseg: int = 0               # segments per row (= units per row of the unit table)
    table: Optional[List[int]] = None   # unit_off (units) or row_off (row_off), G + 1 entries


def plan_rank(n: int, nranks: int, rank: int, G: int, restart: int, speeds: Optional[Sequence[float]] = None) -> RankPlan:
    """gmres_fused_solve's split for one rank (the part after the eligibility checks of `fused_applies`), with `speeds`
    the rank's calibrated per-CTA speeds (None: not calibrated yet)."""
    r0, r1 = bemb200_partition(n, nranks, rank)
    nloc = r1 - r0
    nseg = (n + FUSED_SEGMENT_WIDTH - 1) // FUSED_SEGMENT_WIDTH
    pl = RankPlan(rank=rank, row0=r0, nloc=nloc, mode="equal", nseg=nseg)
    if restart > FUSED_MAX_RESTART or n > 0x7FFFFFFF or nranks > MAX_PEERS:
        pl.mode = "not fused"
        return pl
    have_speed = speeds is not None and len(speeds) == G
    S = (nloc + G - 1) // G or 1
    if nloc >= 4 * G:
        total_units = nloc * nseg
        sp = [float(v) for v in speeds] if have_speed else [1.0] * G
        tot = 0.0
        for v in sp:
            tot += v
        off = [0] * (G + 1)
        cum = 0.0
        smax = 0
        ok_units = total_units < 0xFFFFFFFF
        for c in range(G):
            if not ok_units:
                break
            cum += sp[c] / tot
            e = total_units if c + 1 == G else _llround(cum * float(total_units))
            e = min(e, total_units)
            if e < off[c] + 2 * nseg:
                ok_units = False
            off[c + 1] = e
            own0, own1 = -(-off[c] // nseg), -(-off[c + 1] // nseg)
            smax = max(smax, own1 - own0 + 1)
        if ok_units and smax <= 256:
            pl.mode, pl.table, S = "units", off, smax
    if pl.mode == "equal" and have_speed and nloc >= 8 * G:
        tot = 0.0
        for v in speeds:
            tot += float(v)
        off = [0] * (G + 1)
        cum = 0.0
        smax = 0
        for c in range(G):
            cum += float(speeds[c]) / tot
            e = nloc if c + 1 == G else _llround(cum * float(nloc))
            e = min(max(e, off[c]), nloc)
            off[c + 1] = e
            smax = max(smax, e - off[c])
        pl.mode, pl.table, S = "row_off", off, smax or 1
    pl.S = S
    pl.rblk = fused_pick_rblk(S)
    pl.smem = fused_smem_bytes(S, pl.rblk, restart)
    if pl.smem > SMEM_LIMIT:
        pl.mode = "not fused"
    return pl


def plan(n: int, nranks: int, G: int, restart: int, speeds=None) -> List[RankPlan]:
    """Every rank's plan; `speeds` is None, one list for every rank, or a list of per-rank lists."""
    out = []
    for r in range(nranks):
        sp = speeds
        if speeds is not None and len(speeds) and isinstance(speeds[0], (list, tuple)):
            sp = speeds[r]
        out.append(plan_rank(n, nranks, r, G, restart, sp))
    return out


def fused_applies(restart: int, nranks: int, group: bool, polite: bool, env: Optional[int] = None) -> bool:
    """The eligibility checks at the top of gmres_fused_solve that do not depend on the split (env: value of
    BEMB200_GMRES_FUSED, None when unset).  A single-process group always takes the fused kernel; a lone rank only when
    forced, also in the polite build."""
    if env == 0 or restart > FUSED_MAX_RESTART or nranks > MAX_PEERS:
        return False
    if env is None and not group and (nranks < 2 or polite):
        return False
    return True


@dataclass
class Cta:
    rb: int
    sc: int
    has_head: bool = False
    s0: int = 0
    s1: int = 0xFFFFFFFF


def decode(pl: RankPlan, G: int) -> List[Cta]:
    """gmres_body's decoding of the split into this CTA's rows (gmres_fused.cu, `rows of this CTA inside the rank's slab`)."""
    out = []
    for c in range(G):
        if pl.mode == "units":
            nsegu = pl.nseg
            U0, U1 = pl.table[c], pl.table[c + 1]
            rb = -(-U0 // nsegu)
            own1 = -(-U1 // nsegu)
            sc = own1 - rb if own1 > rb else 0
            s0 = U0 % nsegu
            has_head = s0 != 0 and U1 > U0
            s1 = (U1 % nsegu) or nsegu
            if sc == 0:
                s1 = nsegu
            out.append(Cta(rb, sc, has_head, s0, s1))
        elif pl.mode == "row_off":
            out.append(Cta(pl.table[c], pl.table[c + 1] - pl.table[c]))
        else:
            rb = min(c * pl.S, pl.nloc)
            out.append(Cta(rb, min(rb + pl.S, pl.nloc) - rb))
    return out


@dataclass
class MatvecWork:
    # per segment sg: list of (first slab row, end slab row, cta) row ranges computed in that segment
    cover: List[list] = field(default_factory=list)
    frag_put: dict = field(default_factory=dict)    # cta -> (slab row of its head fragment, first position s0)
    frag_wait: dict = field(default_factory=dict)   # cta -> (slab row waiting for the rest, first missing position s1)
    max_slots: int = 0                              # max over CTAs of sc + head


def matvec_work(pl: RankPlan, ctas: List[Cta], n: int) -> MatvecWork:
    """matvec_rows' loop over passes, segments and slot ranges for every CTA of a rank (the `cbase >= n` skip is per
    warp inside a segment and is not modelled: a segment is the unit here)."""
    nseg = (n + FUSED_SEGMENT_WIDTH - 1) // FUSED_SEGMENT_WIDTH
    w = MatvecWork(cover=[[] for _ in range(nseg)])
    if nseg == 0:
        return w
    sg0 = ((pl.row0 + FUSED_SEGMENT_WIDTH // 2) // FUSED_SEGMENT_WIDTH) % nseg
    for c, ct in enumerate(ctas):
        head = 1 if ct.has_head else 0
        w.max_slots = max(w.max_slots, ct.sc + head)
        blk = 0
        while blk < ct.sc + head:
            nslots = min(ct.sc + head - blk, pl.rblk)
            for si in range(nseg):
                sg = si + sg0 if si + sg0 < nseg else si + sg0 - nseg
                lo, hi = 0, nslots
                if blk == 0 and head and si < ct.s0:
                    lo = 1
                if blk + nslots == ct.sc + head and ct.sc > 0 and si >= ct.s1:
                    hi -= 1
                if lo >= hi:
                    continue
                first = ct.rb - head + blk
                w.cover[sg].append((first + lo, first + hi, c))
            blk += pl.rblk
        if head:
            w.frag_put[c] = (ct.rb - 1, ct.s0)
        if ct.sc > 0 and ct.s1 < nseg:
            w.frag_wait[c] = (ct.rb + ct.sc - 1, ct.s1)
    return w


def check_rank(pl: RankPlan, n: int, G: int, decoder=None) -> List[str]:
    """Problems of one rank's split (empty list: sound).  Every (row, segment) of the slab is computed exactly once, the
    owned rows tile the slab, every fragment wait has its producer in CTA c + 1 (same row, same position), every fragment
    produced is consumed, sc + head <= S and the shared memory fits.  `decoder` replaces `decode` (to show that the
    checks catch a wrong decoding)."""
    errs = []
    if pl.mode == "not fused":
        return errs
    if pl.smem > SMEM_LIMIT:
        errs.append(f"smem {pl.smem} > {SMEM_LIMIT}")
    ctas = (decoder or decode)(pl, G)
    # owned rows: contiguous, in CTA order, covering [0, nloc)
    at = 0
    for c, ct in enumerate(ctas):
        if ct.sc and ct.rb != at:
            errs.append(f"cta {c}: owns rows from {ct.rb}, expected {at}")
        at = ct.rb + ct.sc if ct.sc else at
        if ct.sc + (1 if ct.has_head else 0) > pl.S:
            errs.append(f"cta {c}: sc + head = {ct.sc + ct.has_head} > S = {pl.S}")
    if at != pl.nloc:
        errs.append(f"owned rows end at {at}, slab has {pl.nloc}")
    w = matvec_work(pl, ctas, n)
    for sg, ranges in enumerate(w.cover):
        ranges = sorted(ranges)
        pos = 0
        for a, b, c in ranges:
            if a != pos:
                errs.append(f"segment {sg}: rows [{pos}, {a}) {'missing' if a > pos else 'computed twice'} (cta {c})")
                break
            pos = b
        if pos != pl.nloc and not errs:
            errs.append(f"segment {sg}: rows covered up to {pos} of {pl.nloc}")
        if errs:
            break
    for c, (row, s1) in w.frag_wait.items():
        if w.frag_put.get(c + 1) != (row, s1):
            errs.append(f"cta {c}: waits for row {row} from position {s1}, cta {c + 1} produces {w.frag_put.get(c + 1)}")
    for c in w.frag_put:
        if c - 1 not in w.frag_wait:
            errs.append(f"cta {c}: produces a fragment nobody waits for")
    return errs


# ---- the cases tests/test_gpu_fused_gmres.py runs, with the branch each is there for ---------------------------------
# (name, ranks on device 0, unknowns, expected mode of every rank on the first, uncalibrated solve)
GROUP_CASES = [
    ("k1_equal", 1, 591, "equal"),       # one rank, 148 CTAs: nloc < 4 G = 592, equal shares of 4 rows
    ("k1_units", 1, 593, "units"),       # nloc >= 4 G: (row, segment) units, one segment per row
    ("k1_frag", 1, 5120, "units"),       # three segments per row: CTA boundaries cut rows (head fragments)
    ("k2_frag", 2, 5120, "units"),       # 74 CTAs a rank; calibrated shares from the second solve on
    ("k3_frag", 3, 5120, "units"),       # 49 CTAs a rank, uneven slabs (1707 + 1707 + 1706), per-rank calibrated sizes
    ("k8_tiny", 8, 5, "equal"),          # 18 CTAs a rank, fewer rows than ranks: ranks 5 .. 7 own no rows
    ("k8_big", 8, 38720, "equal"),       # S = 269 > 256: no unit table, two matvec passes; row_off once calibrated
]
GROUP_RESTART = 50
# single-rank solves forced onto the fused kernel (148 CTAs): n -> mode
FORCED_SIZES = {1: "equal", 2: "equal", 100: "equal", 300: "equal", 2100: "units"}


def group_ctas(k: int, sms: int = 148) -> int:
    """CTAs per rank when k ranks share one device (bemb200_multi_create)."""
    return sms // k if k > 1 else sms


def calibrated_modes(n: int, k: int, restart: int = GROUP_RESTART, seed: int = 7, trials: int = 20) -> set:
    """Modes the ranks of a k-rank group land in once calibrated, over speed vectors within +-10 % (the spread measured
    between SMs of one B200)."""
    import random

    G = group_ctas(k)
    rng = random.Random(seed)
    out = set()
    for _ in range(trials):
        for pl in plan(n, k, G, restart, [rng.uniform(0.9, 1.1) for _ in range(G)]):
            out.add(pl.mode)
    return out
