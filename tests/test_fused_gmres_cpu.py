"""The work split of the persistent fused GMRES kernel, checked on the CPU through its mirror (fused_split_reference.py).

For every rank count, CTA count, size and speed vector of the grid below, every (row, segment) of every rank's slab must be
computed by exactly one CTA, every head-fragment wait must have its producer (next CTA, same row, same position), no CTA
may need more row slots than the S its shared memory was sized for, and the shared memory of a fused launch stays within
200 KB.  A second group of tests pins the branch that every case of test_gpu_fused_gmres.py lands in, so that a change of
that case list which stops reaching a branch fails here, without a GPU.
"""
from __future__ import annotations

import random
import sys
from pathlib import Path

import pytest

sys.path.insert(0, str(Path(__file__).resolve().parent))
import fused_split_reference as F  # noqa: E402

CTAS = [148, 74, 49, 37, 29, 24, 21, 18]  # 148 // k for k ranks on one device


def _sizes(G: int):
    seg = F.FUSED_SEGMENT_WIDTH
    out = {1, 2, G - 1, G, G + 1, 4 * G - 1, 4 * G, 4 * G + 1, 8 * G - 1, 8 * G, 16 * G, seg - 1, seg, seg + 1,
           2 * seg + 1, 5120, 20480, 65535}
    # the S = 256 edge of a single rank's equal shares and of the unit table
    out |= {256 * G - 1, 256 * G, 256 * G + 1, 255 * G, 257 * G}
    return sorted(v for v in out if v >= 1)


def _speed_sets(G: int, seed: int):
    rng = random.Random(seed)
    yield "uncalibrated", None
    yield "equal", [1.0] * G
    yield "random", [rng.uniform(0.5, 1.5) for _ in range(G)]
    # a few slow CTAs among fast ones (the shape a fuller GPC gives), and the reverse
    yield "skewed", [0.5 if c % 7 == 0 else 1.5 for c in range(G)]
    yield "skewed_rev", [1.5 if c % 9 == 0 else 0.5 for c in range(G)]


@pytest.mark.parametrize("G", CTAS)
def test_split_covers_every_row_segment_once(G):
    checked = 0
    modes = set()
    for P in range(1, 9):
        for n in _sizes(G):
            for ns in sorted({n, n * P}):  # per-rank slabs around the edges, and whole problems split P ways
                if ns > 70000:
                    continue
                for name, sp in _speed_sets(G, seed=G * 1000 + P * 10 + ns % 997):
                    restart = 63  # the largest shared-memory footprint the fused kernel takes
                    plans = F.plan(ns, P, G, restart, sp)
                    assert sum(p.nloc for p in plans) == ns
                    for pl in plans:
                        errs = F.check_rank(pl, ns, G)
                        assert not errs, f"G={G} P={P} n={ns} speeds={name} rank={pl.rank}: {errs[:3]}"
                        modes.add(pl.mode)
                        checked += 1
    assert checked > 1000
    assert {"equal", "units", "row_off"} <= modes, modes


def test_mirror_detects_a_broken_split():
    """The checker is not vacuous: a last-row cut one position late, and equal shares one row short, are reported."""
    G, n = 148, 5120
    pl = F.plan_rank(n, 1, 0, G, 50)
    assert pl.mode == "units" and not F.check_rank(pl, n, G)

    def late_cut(p, g):
        out = F.decode(p, g)
        for ct in out:
            if ct.s1 < p.nseg:
                ct.s1 += 1
        return out

    assert any("twice" in e or "waits" in e for e in F.check_rank(pl, n, G, decoder=late_cut))
    eq = F.plan_rank(100, 1, 0, G, 50)
    eq.S -= 1  # equal shares one row short: the last rows are nobody's
    assert F.check_rank(eq, 100, G)


def test_smem_and_restart_limits():
    assert F.fused_smem_bytes(256, 256, 63) <= F.SMEM_LIMIT
    assert F.plan_rank(5120, 1, 0, 148, 63).mode == "units"
    assert F.plan_rank(5120, 1, 0, 148, 64).mode == "not fused"
    # equal shares past the shared-memory budget fall back to the per-iteration kernels
    big = F.plan_rank(400_000, 1, 0, 148, 63)
    assert big.mode == "not fused" and big.smem > F.SMEM_LIMIT
    assert F.fused_applies(63, 1, group=False, polite=False, env=1)
    assert F.fused_applies(63, 1, group=False, polite=True, env=1)
    assert not F.fused_applies(64, 1, group=False, polite=False, env=1)
    assert not F.fused_applies(50, 1, group=False, polite=False, env=None)
    assert F.fused_applies(50, 1, group=True, polite=False, env=None)
    assert F.fused_applies(50, 2, group=False, polite=False, env=None)
    assert not F.fused_applies(50, 2, group=False, polite=True, env=None)
    assert not F.fused_applies(50, 2, group=True, polite=False, env=0)


def test_llround_rounds_halves_away_from_zero():
    assert F._llround(2.5) == 3 and F._llround(3.5) == 4 and F._llround(0.49999999999999994) == 0


# ---- the modes of the GPU cases ----------------------------------------------------------------------------------------
@pytest.mark.parametrize("name,k,n,mode", F.GROUP_CASES, ids=[c[0] for c in F.GROUP_CASES])
def test_gpu_group_case_lands_in_its_branch(name, k, n, mode):
    G = F.group_ctas(k)
    assert F.fused_applies(F.GROUP_RESTART, k, group=True, polite=False)
    plans = F.plan(n, k, G, F.GROUP_RESTART)
    for pl in plans:
        assert pl.mode == mode, (name, pl)
        assert not F.check_rank(pl, n, G)
    work = [F.matvec_work(pl, F.decode(pl, G), n) for pl in plans]
    frags = sum(len(w.frag_wait) for w in work)
    multipass = any(pl.S > pl.rblk for pl in plans)
    empty = sum(pl.nloc == 0 for pl in plans)
    if name.endswith("_frag"):
        assert plans[0].nseg > 1 and frags > 0, name
    else:
        assert frags == 0, name
    if name == "k1_equal":
        assert plans[0].nloc < 4 * G <= plans[0].nloc + 1
    if name == "k1_units":
        assert plans[0].nloc >= 4 * G and plans[0].nseg == 1
    if name == "k8_tiny":
        assert empty == 3 and n < k
    else:
        assert empty == 0
    if name == "k8_big":
        assert multipass and all(pl.S == 269 and pl.rblk == 256 for pl in plans)
        # calibrated: no unit table fits 256 slots, the weighted row table takes over (any speeds within +-10 %)
        rng = random.Random(7)
        for _ in range(20):
            sp = [rng.uniform(0.9, 1.1) for _ in range(G)]
            cal = F.plan(n, k, G, F.GROUP_RESTART, sp)
            assert all(pl.mode == "row_off" and pl.S > 256 and not F.check_rank(pl, n, G) for pl in cal)
            assert all(F.fused_smem_bytes(256, 256, F.GROUP_RESTART) < pl.smem <= F.SMEM_LIMIT for pl in cal)
    else:
        assert not multipass
    if name in ("k1_frag", "k2_frag", "k3_frag"):
        # calibrated on the first solve (nloc >= 16 G): speeds within +-10 % keep the unit table
        assert all(pl.nloc >= 16 * G for pl in plans)
        rng = random.Random(11)
        for _ in range(20):
            sp = [rng.uniform(0.9, 1.1) for _ in range(G)]
            assert all(pl.mode == "units" for pl in F.plan(n, k, G, F.GROUP_RESTART, sp))


def test_gpu_cases_reach_every_branch():
    """The GPU cases, uncalibrated and calibrated, reach equal shares, units, the row table and the two-pass matvec."""
    modes = {c[3] for c in F.GROUP_CASES} | set(F.FORCED_SIZES.values())
    for name, k, n, _ in F.GROUP_CASES:
        if all(pl.nloc >= 16 * F.group_ctas(k) for pl in F.plan(n, k, F.group_ctas(k), F.GROUP_RESTART)):
            modes |= F.calibrated_modes(n, k)
    assert {"equal", "units", "row_off"} <= modes, modes
    assert any(pl.S > pl.rblk for _, k, n, _ in F.GROUP_CASES for pl in F.plan(n, k, F.group_ctas(k), F.GROUP_RESTART))
    assert any(k >= 3 for _, k, _, _ in F.GROUP_CASES)
    for n, mode in F.FORCED_SIZES.items():
        pl = F.plan_rank(n, 1, 0, 148, 63)
        assert pl.mode == mode, (n, pl)
        assert not F.check_rank(pl, n, 148)
    assert any(n < 148 for n in F.FORCED_SIZES)  # CTAs without rows
    assert F.plan_rank(max(F.FORCED_SIZES), 1, 0, 148, 63).nseg > 1
