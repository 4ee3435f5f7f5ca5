"""Parity of the solve paths that only large or unusual batches reach.

`WaitImpl` / `EnqueueSolve` / `LaunchFused` (yadcc_b200/csrc/ydsched.cu) choose among the one-launch fused kernel
(solo or in front of the coupled solvers), the kernel-by-kernel pipeline, the one-launch or three-pass final, a kept
or a per-solve slot table and narrow or wide slot keys by host-side size thresholds.  Every case here plays one event
sequence into the CUDA backend and into the CPU restatement (oracle/port.cc) and compares, bit for bit, the grants
(status, servant index, task id), `servant_state()`, `num_tasks()` and `next_task_id()`, through the plain and the
packed interface.  Each case also asserts

* a witness: `Path` restates the thresholds and the case's shape lands on the intended side of them; the
  library's own report (`YDSCHED_DEBUG` / `YDSCHED_FUSED_PROF` stderr lines, `last_solve_stats()`) says the same;
* sensitivity: grants land where the path's arithmetic acts (every 1024-request block of a three-pass final,
  request tiles the fused kernel reaches only in its second grid-stride round, ...), so an off-by-one there moves
  task ids or servants.

The narrow-key case also has a CPU test: an exact-rational model of the decision (integer cross-multiplication
instead of the reference's double r/cap) against the port, on a workload where the runner-up is often within 2^-25
of the winner.
"""
from __future__ import annotations

import re
from dataclasses import dataclass
from fractions import Fraction

import numpy as np
import pytest

from yadcc_b200 import _abi
from yadcc_b200 import streams as S
from yadcc_b200.dispatcher import Servant, pack_requests

GPU = pytest.mark.gpu
GRANTED, TIMEOUT = _abi.STATUS_GRANTED, _abi.STATUS_TIMEOUT
GiB = 1 << 30

# ---- the host thresholds (yadcc_b200/csrc/ydsched.cu unless noted) ------------------------------------------------
REQ_BLOCK = 1024  # NextPow2(N, 1024) (:1427) and the finals' 1024-thread blocks (nb = Nb / 1024, :1198)
RANK_TILE = 1024  # yd::kRankTile (parallel.cuh:23): request tiles of the fused kernel, :1510
LIST_TILE = 1024  # yd::kListTile (classes.cuh:345): tiles of the kept slot table, :1511
FUSED_MAX_NB = 262144  # fused_max_nb (:200): largest batch size class the fused kernel takes, :1509
FUSED_CELLS = 32768  # cls_bound * rank tiles and cls_bound * list tiles, :1510-1511
LOFF_CACHE_WORDS = 16384  # kFusedLoffCacheWords (:1093): solo offsets in shared memory iff they fit, :1151-1152
FINAL_FUSED_MAX_BLOCKS = 2048  # kFinalFusedMaxBlocks (:1181): k_final_fused up to here, else three passes, :1186
STATIC_SLOT_LIMIT = 1 << 26  # kStaticSlotLimit (:945): kept slot table up to here, :1434
NARROW_CAP_LIMIT = 8192  # yd::kNarrowCapLimit (common.cuh:36): 32-bit slot keys up to here, :370
DEFAULT_CLS_BOUND = 16  # cls_bound (:185); grows to the next power of two at or above classes + 1 on demand, :1637-1641


def _next_pow2(v: int, lo: int) -> int:
    r = lo
    while r < v:
        r <<= 1
    return r


def _sms() -> int:
    import torch

    return torch.cuda.get_device_properties(0).multi_processor_count  # fused grid: one block per SM (:600)


@dataclass
class Path:
    """Which branch each host threshold selects for a batch of `n` requests (solver: 0 auto, 1 row-scan)."""

    n: int
    caps: list[int]  # min(nproc, max_tasks) of every servant
    cls_bound: int = DEFAULT_CLS_BOUND
    solver: int = 0
    coupled: bool = False  # a component the solo kernel cannot decide: fused variant 1 instead of 2/3

    @property
    def Nb(self) -> int:
        return _next_pow2(self.n, REQ_BLOCK)

    @property
    def static(self) -> bool:  # :1433-1434
        return self.solver != 1 and sum(c + 1 for c in self.caps) <= STATIC_SLOT_LIMIT

    @property
    def slot_b(self) -> int:  # :1435-1441
        bound = sum(c + 1 for c in self.caps) if self.static else sum(min(c, self.n) + 1 for c in self.caps)
        return _next_pow2(max(bound, 1), 4096)

    @property
    def rank_cells(self) -> int:
        return self.cls_bound * -(-self.Nb // RANK_TILE)

    @property
    def list_cells(self) -> int:
        return self.cls_bound * -(-self.slot_b // LIST_TILE)

    @property
    def fused(self) -> bool:  # :1509-1511
        return (self.solver == 0 and self.static and self.Nb <= FUSED_MAX_NB and self.rank_cells <= FUSED_CELLS
                and self.list_cells <= FUSED_CELLS)

    @property
    def solo(self) -> bool:
        return self.fused and not self.coupled

    @property
    def offsets_in_hbm(self) -> bool:  # :1151-1152
        return self.solo and self.list_cells + self.cls_bound + 1 > LOFF_CACHE_WORDS

    @property
    def final_passes(self) -> int:  # FinalPasses, :1184-1187
        if self.solo:
            return 0
        return 1 if self.solver == 0 and self.Nb // REQ_BLOCK <= FINAL_FUSED_MAX_BLOCKS else 3

    @property
    def wide(self) -> bool:  # :365-370
        return max(self.caps) > NARROW_CAP_LIMIT

    def fused_rounds(self, sms: int) -> int:
        """Grid-stride rounds of the fused kernel over request tiles (grid = sms blocks)."""
        tiles = -(-self.n // RANK_TILE)
        return -(-tiles // sms)


_DEBUG_RE = re.compile(r"ydsched: solver (\d+) graph (\d+) .* variant (\d+) fused_dyn (\d+) lite (\d+) "
                       r"final_passes (\d+) wide (\d+) static (\d+)")
_PROF_RE = re.compile(r"ydsched: fused variant (\d+) n (\d+) ns:")


class Witness:
    """Reads what the library says about each CUDA solve: the YDSCHED_DEBUG line (written once per solve), the last
    YDSCHED_FUSED_PROF line and last_solve_stats()."""

    def __init__(self, monkeypatch, capfd):
        monkeypatch.setenv("YDSCHED_DEBUG", "1")  # (both read by yd_create)
        monkeypatch.setenv("YDSCHED_FUSED_PROF", "1")
        self.capfd = capfd
        self.solves: list[dict] = []

    def __call__(self, d, n):
        err = self.capfd.readouterr().err
        dbg = _DEBUG_RE.findall(err)
        assert len(dbg) == 1, f"expected one YDSCHED_DEBUG line per solve, got:\n{err}"
        solver, graph, variant, dyn, lite, passes, wide, static = map(int, dbg[0])
        prof = _PROF_RE.findall(err)
        st = d.last_solve_stats()
        self.solves.append(dict(n=n, solver=solver, graph=graph, variant=variant, dyn=dyn, lite=lite, passes=passes,
                                wide=wide, static=static, prof=[tuple(map(int, p)) for p in prof], stats=st))

    def check(self, p: Path, k: int = 0, *, lite: bool = True):
        """Solve k of the last run took the branches `p` predicts."""
        w = self.solves[k]
        assert w["n"] == p.n and w["stats"]["decisions"] == p.n
        assert w["solver"] == w["stats"]["solver"] == (1 if p.solver == 1 else 2)
        want_variant = {True: (2, 3), False: (1,)}[p.solo] if p.fused else (0,)
        assert w["variant"] in want_variant, (w, p)
        if p.fused:  # the fused kernel reports its own variant and batch size
            assert w["prof"] and w["prof"][-1] == (w["variant"], p.n), w
            assert w["lite"] == int(lite)
        assert (w["dyn"] == 0) == (not p.solo or p.offsets_in_hbm), w
        if p.solo and not p.offsets_in_hbm:
            assert w["dyn"] == 4 * (p.list_cells + p.cls_bound + 1), w
        assert w["passes"] == p.final_passes, (w, p.final_passes)
        assert w["wide"] == int(p.wide) and w["static"] == int(p.static), w
        assert w["stats"]["kernel_launches"] >= 1 + (p.final_passes if not p.fused else 0), w


# ---- event sequences ------------------------------------------------------------------------------------------------
# ("hb", now, [Servant])  heartbeats;  ("wait", now, build(d) -> REQ array)  one batch;  ("free", seed, frac)  free a
# seeded share of the outstanding grants;  ("state",)  servant_state(), num_tasks(), next_task_id()


def _solve(d, reqs, now, packed, pinned):
    n = len(reqs)
    if packed:
        if pinned:
            g = d.wait_for_starting_new_tasks_packed(pack_requests(reqs, d.alloc_requests16(n)), now,
                                                     out8=d.alloc_grants8(n))
        else:
            g = d.wait_for_starting_new_tasks_packed(pack_requests(reqs), now)
    elif pinned:
        buf = d.alloc_requests(n)
        buf[...] = reqs
        g = d.wait_for_starting_new_tasks(buf, now, out=d.alloc_grants(n))
    else:
        g = d.wait_for_starting_new_tasks(np.ascontiguousarray(reqs), now)
    return np.stack([g["status"].astype(np.uint64), g["servant_index"].astype(np.uint64), g["task_id"]], axis=1)


def _play(d, events, *, packed=False, pinned=False, witness=None):
    """Runs `events` on `d`; returns the trace: (kind, array) per solve and per state snapshot."""
    trace, held = [], []
    for ev in events:
        if ev[0] == "hb":
            d.keep_servants_alive(ev[2], 100.0, now=ev[1])
        elif ev[0] == "wait":
            reqs = ev[2](d)
            g = _solve(d, reqs, ev[1], packed, pinned)
            if witness is not None:
                witness(d, len(reqs))
            held.extend(g[g[:, 0] == GRANTED, 2].tolist())
            trace.append(("grants", g))
        elif ev[0] == "free":
            ids = np.asarray(sorted(held), dtype=np.uint64)
            pick = ids[np.random.default_rng(ev[1]).random(len(ids)) < ev[2]]
            d.free_tasks(pick)
            gone = set(pick.tolist())
            held = [t for t in held if t not in gone]
        elif ev[0] == "state":
            st = d.servant_state()
            trace.append(("state", np.stack([st[k].astype(np.uint64) for k in st.dtype.names], axis=1)))
            trace.append(("counts", np.asarray([d.num_tasks(), d.next_task_id()], dtype=np.uint64)))
    return trace


def _assert_same(got, want, what):
    assert len(got) == len(want), f"{what}: {len(got)} vs {len(want)} outputs"
    for k, ((kind, a), (_, b)) in enumerate(zip(got, want)):
        assert a.shape == b.shape, f"{what}: output {k} ({kind}) shape {a.shape} vs {b.shape}"
        bad = np.nonzero((a != b).reshape(len(a), -1).any(axis=1))[0] if a.ndim else np.nonzero(a != b)[0]
        assert not len(bad), (f"{what}: output {k} ({kind}), row {bad[0]}: cuda {a[bad[0]].tolist()} vs port "
                              f"{b[bad[0]].tolist()} ({len(bad)} rows differ)")


_port_traces: dict = {}


def _port_trace(make_dispatcher, key, events):
    """The port's trace of one event sequence (the same for every CUDA configuration it is compared with)."""
    if key not in _port_traces:
        _port_traces[key] = _play(make_dispatcher("port"), events)
    return _port_traces[key]


IFACES = [(False, False), (True, True)]  # (packed, pinned): the plain call from pageable memory, the packed one pinned
ALL_IFACES = [(False, False), (False, True), (True, False), (True, True)]


def _parity(make_dispatcher, monkeypatch, capfd, key, events, ifaces=IFACES, **cuda_kw):
    """Plays `events` into the port and into CUDA once per interface; returns (port trace, [Witness])."""
    want = _port_trace(make_dispatcher, key, events)
    witnesses = []
    for packed, pinned in ifaces:
        w = Witness(monkeypatch, capfd)
        got = _play(make_dispatcher("cuda", **cuda_kw), events, packed=packed, pinned=pinned, witness=w)
        _assert_same(got, want, f"{key} {cuda_kw} packed={packed} pinned={pinned}")
        witnesses.append(w)
    return want, witnesses


def _grants(trace):
    return [a for kind, a in trace if kind == "grants"]


def _servants(caps, digests_of, *, load=None, dedicated=(), nproc=None):
    out = []
    for i, c in enumerate(caps):
        out.append(Servant(f"{S.servant_ip(i)}:8335", None, digests_of(i), 8, nproc[i] if nproc else c,
                           load[i] if load else 0, 256 * GiB, 200 * GiB, c,
                           _abi.PRIORITY_DEDICATED if i in dedicated else _abi.PRIORITY_USER))
    return out


def _digests(n, seed):
    rng = np.random.default_rng(seed)
    return [S.hex_digest(rng) for _ in range(n)]


# ---- 1: three-pass final above 2^21 requests ---------------------------------------------------------------------
# 64 servants x 4000 slots, 4 digests; ~6 % of the requests ask a held digest (uniformly), the rest an unknown one, so
# every 1024-request block holds grants and a wrong carry in k_final_scan moves task ids.

BIG = [1 << 21, (1 << 21) + 1, 2_300_000]


def _sparse_events(n, layout="mod", zero_head=False, seed=11, n_servants=64, cap=4000):
    dgs = _digests(5, seed)
    held, unknown = dgs[:4], dgs[4]
    rng = np.random.default_rng(seed)
    if layout == "random":
        sets = [[held[j] for j in rng.choice(4, size=int(rng.integers(1, 4)), replace=False)] for _ in range(n_servants)]
    else:
        sets = [[held[i % 4]] for i in range(n_servants)]
    servants = _servants([cap] * n_servants, lambda i: sets[i])

    def build(d, n=n, salt=0):
        r = np.random.default_rng(seed + 1 + salt)
        env = np.asarray([d.intern_env(x) for x in held], dtype=np.uint32)
        miss = d.intern_env(unknown)
        outside = np.asarray([d.intern_ip(f"172.16.{i >> 8}.{i & 255}") for i in range(1024)], dtype=np.uint32)
        hit = r.random(n) < 0.06
        hit[-1] = True  # (the last block of 2^21 + 1 requests holds one request)
        if zero_head:
            hit[: 1 << 20] = False
        ips = outside[r.integers(0, len(outside), n)]
        if layout == "self":  # a third of the held-digest requests come from servants
            inside = np.asarray([d.intern_ip(S.servant_ip(i)) for i in range(n_servants)], dtype=np.uint32)
            ips = np.where(hit & (r.random(n) < 0.33), inside[r.integers(0, n_servants, n)], ips)
        return S._requests(d, np.where(hit, env[r.integers(0, 4, n)], miss).astype(np.uint32), ips, 8)

    return [("hb", 0.0, servants), ("wait", 0.001, build), ("state",), ("free", 5, 0.5),
            ("wait", 0.002, lambda d: build(d, n, 1)), ("state",)], [cap] * n_servants


def _every_block_granted(g, skip_blocks=0):
    granted = g[:, 0] == GRANTED
    per_block = np.add.reduceat(granted, np.arange(0, len(g), REQ_BLOCK))
    assert (per_block[skip_blocks:] > 0).all(), "a 1024-request block without grants"
    return per_block


@GPU
@pytest.mark.parametrize("solver", [0, 1], ids=["auto", "rowscan"])
@pytest.mark.parametrize("n", BIG)
def test_final_above_2_21_requests(make_dispatcher, monkeypatch, capfd, n, solver):
    events, caps = _sparse_events(n)
    want, ws = _parity(make_dispatcher, monkeypatch, capfd, ("sparse", n), events, solver=solver)
    p = Path(n, caps, solver=solver)
    assert p.final_passes == (1 if solver == 0 and n <= 1 << 21 else 3) and not p.fused
    for w in ws:
        w.check(p, 0)
        w.check(p, 1)
    for g in _grants(want):
        per_block = _every_block_granted(g)
        assert len(per_block) > 1024 or n <= 1 << 20  # the scan carries over more than one 1024-block round
        assert g[g[:, 0] == GRANTED, 2].max() == g[g[:, 0] == GRANTED, 2].min() + per_block.sum() - 1


@GPU
@pytest.mark.parametrize("variant", ["zero-head", "random", "self-merge", "self-sequential"])
def test_three_pass_final_layouts(make_dispatcher, monkeypatch, capfd, variant):
    """2^21 + 1 requests: the first 2^20 all unknown (the first scan round carries zero), a coupled component (the
    merge solver), requestors that are servants (merge solver, and the sequential solver with merge_self=False)."""
    n = (1 << 21) + 1
    layout = {"zero-head": "mod", "random": "random"}.get(variant, "self")
    events, caps = _sparse_events(n, layout=layout, zero_head=variant == "zero-head")
    kw = {"merge_self": False} if variant == "self-sequential" else {}
    want, ws = _parity(make_dispatcher, monkeypatch, capfd, ("sparse", n, variant), events, **kw)
    p = Path(n, caps)
    assert p.final_passes == 3
    for w in ws:
        w.check(p, 0)
        w.check(p, 1)
    for g in _grants(want):
        per_block = _every_block_granted(g, skip_blocks=(1 << 20) // REQ_BLOCK if variant == "zero-head" else 0)
        if variant == "zero-head":
            assert per_block[: (1 << 20) // REQ_BLOCK].sum() == 0
    if layout == "self":  # some grants went to the requestor's own machine or past it
        g = _grants(want)[0]
        assert (g[:, 0] == GRANTED).sum() > 100_000


# ---- 2: the fused kernel's second grid-stride round over request tiles -------------------------------------------

def _cfg2_events(n, variant, n_servants=256, cap=1100, seed=42):
    """config2's servants and first batch, then (after freeing half the grants) n / 2 more requests for its digests."""
    w = S.config2(n, n_servants, 8, seed=seed, variant=variant, max_tasks=cap, nproc=cap)

    def second(d):
        r = np.random.default_rng(seed + 7)
        env = np.asarray([d.intern_env(x) for x in w.digests], dtype=np.uint32)
        ips = np.asarray([d.intern_ip(f"172.16.{i >> 8}.{i & 255}") for i in range(4096)], dtype=np.uint32)
        return S._requests(d, env[r.integers(0, 8, n // 2)], ips[r.integers(0, 4096, n // 2)], 8)

    return [("hb", 0.0, w.servants), ("wait", 0.001, w.build_requests), ("state",), ("free", 3, 0.5),
            ("wait", 0.002, second), ("state",)], [cap] * n_servants


@GPU
@pytest.mark.parametrize("graphs", [True, False], ids=["graph", "eager"])
@pytest.mark.parametrize("n", [200_000, 262_144, 262_145])
@pytest.mark.parametrize("variant", ["mod", "random"])
def test_fused_second_round(make_dispatcher, monkeypatch, capfd, variant, n, graphs):
    """mod: data-parallel components, the solo kernel; random: one coupled component, the fused front + coupled
    solvers.  262 145 requests take the pipeline.  Pinned (zero-copy in and out) and pageable arrays."""
    events, caps = _cfg2_events(n, variant)
    want, ws = _parity(make_dispatcher, monkeypatch, capfd, ("cfg2", variant, n), events, ALL_IFACES, graphs=graphs)
    sms = _sms()
    p = Path(n, caps, coupled=variant == "random")
    assert p.fused == (n <= FUSED_MAX_NB)
    if p.fused:
        assert p.fused_rounds(sms) == 2
    for w in ws:
        w.check(p, 0)
        w.check(Path(n // 2, caps, coupled=variant == "random"), 1)
    g = _grants(want)[0]
    beyond = g[sms * RANK_TILE:]
    assert (beyond[:, 0] == GRANTED).sum() > 0.9 * len(beyond)  # requests in tiles >= SM count are granted
    if variant == "mod" and n == 200_000:
        assert (g[:, 0] == GRANTED).all()


# ---- 3: the solo kernel's list offsets in HBM (and in shared memory), NOLITE ---------------------------------------
# 8 data-parallel components, nproc = max_tasks = 8000: 64 servants keep 2^19 slots (offsets in shared memory),
# 100 -> 2^20 (one list tile too many for shared memory), 200 -> 2^21 (the last slot table the fused kernel takes),
# 300 -> 2^22 (the pipeline).

@GPU
@pytest.mark.parametrize("nolite", [False, True], ids=["lite", "nolite"])
@pytest.mark.parametrize("n_servants", [64, 100, 200, 300])
def test_solo_list_offsets(make_dispatcher, monkeypatch, capfd, n_servants, nolite):
    if nolite:
        monkeypatch.setenv("YDSCHED_FUSED_NOLITE", "1")
    n = 150_000
    events, caps = _cfg2_events(n, "mod", n_servants=n_servants, cap=8000, seed=21)
    want, ws = _parity(make_dispatcher, monkeypatch, capfd, ("offsets", n_servants), events)
    p = Path(n, caps)
    assert (p.fused, p.offsets_in_hbm) == {64: (True, False), 100: (True, True), 200: (True, True),
                                           300: (False, False)}[n_servants]
    for w in ws:
        w.check(p, 0, lite=not nolite)
        w.check(Path(n // 2, caps), 1, lite=not nolite)
    g = _grants(want)[0]
    assert (g[:, 0] == GRANTED).all()
    # every class's list is searched far past its first tile
    per_servant = np.bincount(g[:, 1].astype(np.int64), minlength=n_servants)
    per_class = np.bincount(np.arange(n_servants) % 8, weights=per_servant)
    assert (per_class > 8 * LIST_TILE).all()


# ---- 4: the per-solve slot table above 2^26 kept slots ------------------------------------------------------------

def _ordinary_caps(seed=31):
    return [int(c) for c in np.random.default_rng(seed).choice([16, 24, 48, 64, 96], 15)]


def _huge_events(big, seed=31):
    """One servant with nproc = max_tasks = `big` (its load leaves it 300 + r free cores: it competes on r/cap) among
    15 ordinary ones, four dedicated; requests from outside and from servants, four solves with frees in between."""
    dgs = _digests(2, seed)
    rng = np.random.default_rng(seed + 1)
    caps = [big] + _ordinary_caps(seed)
    load = [big - 300] + [int(rng.integers(0, 20)) for _ in range(15)]
    nproc = [big] + [c + int(rng.integers(0, 16)) for c in caps[1:]]
    servants = _servants(caps, lambda i: [dgs[i % 2]] if i % 5 == 4 else dgs, load=load, dedicated=(2, 5, 9, 13),
                         nproc=nproc)

    def build(k):
        def b(d):
            r = np.random.default_rng(seed + 10 + k)
            n = int(r.integers(1500, 4000))
            env = np.asarray([d.intern_env(x) for x in dgs], dtype=np.uint32)
            ips = np.asarray([d.intern_ip(f"172.16.0.{i}") for i in range(50)] +
                             [d.intern_ip(S.servant_ip(i)) for i in range(16)], dtype=np.uint32)
            return S._requests(d, env[r.integers(0, 2, n)], ips[r.integers(0, len(ips), n)], 8)
        return b

    ev = [("hb", 0.0, servants)]
    for k in range(4):
        ev += [("wait", 0.001 * (k + 1), build(k)), ("state",), ("free", 40 + k, 0.6)]
    return ev + [("state",)], caps


@GPU
@pytest.mark.parametrize("side", ["per-solve", "kept"])
def test_per_solve_slot_table(make_dispatcher, monkeypatch, capfd, side):
    """Static slot bound 2^26 + 1 (the table is rebuilt per solve, rows clamped to the batch) and exactly 2^26 (kept)."""
    big = STATIC_SLOT_LIMIT - sum(c + 1 for c in _ordinary_caps()) - 1 + (side == "per-solve")
    events, caps = _huge_events(big)
    want, ws = _parity(make_dispatcher, monkeypatch, capfd, ("huge", side), events)
    assert sum(c + 1 for c in caps) == STATIC_SLOT_LIMIT + (side == "per-solve")
    for w in ws:
        for k, s in enumerate(w.solves):
            p = Path(s["n"], caps)
            assert p.static == (side == "kept") and p.wide and not p.fused
            w.check(p, k)
    for g in _grants(want):  # the huge servant and the ordinary ones both win in every solve
        won = g[g[:, 0] == GRANTED, 1]
        assert (won == 0).sum() > 50 and (won != 0).sum() > 50
    states = [a for kind, a in want if kind == "state"]
    assert all(st[0, 0] > 0 for st in states)  # solves after the first start with the huge servant partly filled


# ---- 5: narrow slot keys where they are tightest --------------------------------------------------------------------

def _tight_servants(widen=False):
    """8 servants with min(nproc, max_tasks) in 8185..8192 (one at 8193 when widened), loads that make capacity vary
    with r, two dedicated with odd nproc."""
    caps = [8192, 8191, 8190, 8189, 8188, 8187, 8186, 8185]
    nproc = [8192, 8191, 8193, 8189, 8195, 8187, 8186, 8191]
    load = [0, 700, 0, 1500, 40, 0, 3001, 0]
    if widen:
        caps[3] = nproc[3] = 8193
    return caps, nproc, load, (2, 5)


def _tight_events(widen=False, seed=51):
    dg = _digests(1, seed)
    caps, nproc, load, dedicated = _tight_servants(widen)
    servants = _servants(caps, lambda i: dg, load=load, dedicated=dedicated, nproc=nproc)

    def build(k, n):
        def b(d):
            r = np.random.default_rng(seed + k)
            ips = np.asarray([d.intern_ip(f"172.16.1.{i}") for i in range(40)] +
                             [d.intern_ip(S.servant_ip(i)) for i in range(8)], dtype=np.uint32)
            return S._requests(d, np.full(n, d.intern_env(dg[0]), np.uint32), ips[r.integers(0, len(ips), n)], 8)
        return b

    ev = [("hb", 0.0, servants)]
    for k, (n, frac) in enumerate([(64_000, 0.97)] * 5):  # fill to (nearly) full, free almost all, five times
        ev += [("wait", 0.001 * (k + 1), build(k, n)), ("state",), ("free", 60 + k, frac)]
    return ev, caps


class RationalModel:
    """WaitForStartingNewTask (task_dispatcher.cc:93-140 as restated in oracle/port.cc:144-192) with r/cap compared
    exactly by integer cross-multiplication.  Memory is ample and every servant holds the one digest, so
    eligibility is `max_tasks != 0`.  Records, per grant, the gap between the winner's and the runner-up's ratio."""

    def __init__(self, servants):
        self.sv = servants
        self.host = [s.observed_location.rsplit(":", 1)[0] for s in servants]
        self.run = [0] * len(servants)
        self.ever = [0] * len(servants)
        self.tasks: dict[int, int] = {}
        self.next_id = 0
        self.gaps: list[Fraction] = []
        self.envs: dict[str, int] = {}
        self.ips: dict[str, int] = {"": 0}

    # request arrays are built against the model as against a dispatcher: ids in first-seen order, "" is ip 0
    def intern_env(self, x):
        return self.envs.setdefault(x, len(self.envs))

    def intern_ip(self, x):
        return self.ips.setdefault(x, len(self.ips))

    def cap(self, i):
        s = self.sv[i]
        foreign = max(s.current_load - self.run[i], 0)
        return min(s.max_tasks, max(s.num_processors - foreign, 0))

    def _less(self, a, b):
        """(run/cap, position) of a below b's: run_a * cap_b < run_b * cap_a, first position on a tie."""
        x, y = self.run[a] * self.cap(b), self.run[b] * self.cap(a)
        return x < y or (x == y and a < b)

    def decide(self, ip):
        free, self_i = [], -1
        for i, s in enumerate(self.sv):
            if s.max_tasks == 0 or self.run[i] >= self.cap(i):
                continue
            if self_i < 0 and self.host[i] == ip:
                self_i = i
                continue
            free.append(i)
        if not free and self_i < 0:
            return (TIMEOUT, _abi.NO_SERVANT, 0)
        tier = [i for i in free if self.sv[i].priority == _abi.PRIORITY_DEDICATED
                and 2 * self.run[i] < self.sv[i].num_processors]
        pool = tier or free
        if pool:
            best = second = None
            for i in pool:
                if best is None or self._less(i, best):
                    best, second = i, best
                elif second is None or self._less(i, second):
                    second = i
            pick = best
            if second is not None:
                self.gaps.append(Fraction(self.run[second], self.cap(second)) - Fraction(self.run[best], self.cap(best)))
        else:
            pick = self_i
        self.run[pick] += 1
        self.ever[pick] += 1
        tid = self.next_id
        self.next_id += 1
        self.tasks[tid] = pick
        return (GRANTED, pick, tid)

    def play(self, events):
        trace, held = [], []
        ip_name = None
        for ev in events:
            if ev[0] == "wait":
                reqs = ev[2](self)
                ip_name = {v: k for k, v in self.ips.items()}
                g = np.asarray([self.decide(ip_name[int(ip)]) for ip in reqs["requestor_ip"]], dtype=np.uint64)
                held.extend(g[g[:, 0] == GRANTED, 2].tolist())
                trace.append(("grants", g))
            elif ev[0] == "free":
                ids = np.asarray(sorted(held), dtype=np.uint64)
                pick = ids[np.random.default_rng(ev[1]).random(len(ids)) < ev[2]]
                for t in pick.tolist():
                    self.run[self.tasks.pop(t)] -= 1
                gone = set(pick.tolist())
                held = [t for t in held if t not in gone]
            elif ev[0] == "state":
                trace.append(("state", np.asarray([self.run, self.ever, [self.cap(i) for i in range(len(self.sv))]],
                                                  dtype=np.uint64).T))
                trace.append(("counts", np.asarray([len(self.tasks), self.next_id], dtype=np.uint64)))
        return trace


@pytest.mark.parametrize("widen", [False, True], ids=["narrow", "wide"])
def test_rational_model_equals_port_on_tight_keys(make_dispatcher, widen):
    """CPU: the exact-rational decision rule and the port agree on the tight-key workload, and that workload puts the
    runner-up within 2^-25 of the winner's ratio (two narrow-key units) in hundreds of decisions."""
    events, caps = _tight_events(widen)
    model = RationalModel(events[0][2])
    mt = model.play(events)
    pt = _play(make_dispatcher("port"), events)
    # the port's state rows are (running, ever, capacity); the model's too
    _assert_same([(k, a[:, :3] if k == "state" else a) for k, a in pt], mt, "port vs exact-rational model")
    close = sum(1 for gap in model.gaps if gap <= Fraction(1, 1 << 25))
    distinct = sum(1 for gap in model.gaps if 0 < gap <= Fraction(1, 1 << 25))
    assert close >= 200 and distinct >= 120, (close, distinct)
    assert max(_tight_servants(widen)[0]) == (8193 if widen else 8192)


@GPU
@pytest.mark.parametrize("solver", [0, 1], ids=["auto", "rowscan"])
@pytest.mark.parametrize("widen", [False, True], ids=["narrow", "wide"])
def test_tight_narrow_keys(make_dispatcher, monkeypatch, capfd, widen, solver):
    """Capacities 8185..8192 (32-bit keys at their limit) and the twin with one servant at 8193 (64-bit keys)."""
    events, caps = _tight_events(widen)
    want, ws = _parity(make_dispatcher, monkeypatch, capfd, ("tight", widen), events, solver=solver)
    for w in ws:
        for k, s in enumerate(w.solves):
            p = Path(s["n"], caps, solver=solver, coupled=True)  # (requestors that are servants: fused variant 1)
            assert p.wide == widen
            w.check(p, k)
    running = [a[:, 0] for kind, a in want if kind == "state"]
    assert max(r.min() for r in running) > 2000  # running counts reach thousands on every servant


# ---- 6: the rank-tile limit with 128 classes ---------------------------------------------------------------------
# 512 servants, digest i mod 128, 254 slots each: 130 560 kept slots (128 list tiles), cls_bound grows to 256, so
# cls_bound * list tiles = 32768 exactly and the batch size alone decides: 1024 / 1025 requests (one / two rank tiles,
# both fused), 131 072 (128 rank tiles: fused) / 131 073 (256: the pipeline).  20 % of the requests ask a 129th,
# unknown digest, so that capacity lasts to the batch's last rank tile.

@GPU
@pytest.mark.parametrize("n", [1024, 1025, 131_072, 131_073])
def test_rank_tile_limit_with_many_classes(make_dispatcher, monkeypatch, capfd, n):
    dgs = _digests(129, 61)
    caps = [254] * 512
    servants = _servants(caps, lambda i: [dgs[i % 128]])

    def build(d, n=n, seed=62):
        r = np.random.default_rng(seed)
        env = np.asarray([d.intern_env(x) for x in dgs], dtype=np.uint32)
        ips = np.asarray([d.intern_ip(f"172.17.{i >> 8}.{i & 255}") for i in range(2048)], dtype=np.uint32)
        pick = np.where(r.random(n) < 0.2, 128, r.integers(0, 128, n))
        pick[-1] = 0  # (the last rank tile of 131 073 requests holds one request)
        return S._requests(d, env[pick], ips[r.integers(0, 2048, n)], 8)

    events = [("hb", 0.0, servants), ("wait", 0.001, build), ("state",), ("free", 9, 0.9),
              ("wait", 0.002, lambda d: build(d, n, 63)), ("state",)]
    want, ws = _parity(make_dispatcher, monkeypatch, capfd, ("classes", n), events)
    p = Path(n, caps, cls_bound=256)
    assert p.list_cells == FUSED_CELLS and p.fused == (n <= 131_072)
    for w in ws:
        w.check(p, 0)
        w.check(p, 1)
    for g in _grants(want):
        last = g[(n - 1) // RANK_TILE * RANK_TILE:]  # the last rank tile
        assert (last[:, 0] == GRANTED).any()
        if n > RANK_TILE * 2:  # every class wins somewhere
            assert len(np.unique(g[g[:, 0] == GRANTED, 1] % 128)) == 128
