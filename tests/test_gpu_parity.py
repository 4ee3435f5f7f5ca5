"""Parity of the CUDA backend (through the C ABI) against the CPU checkers and
the committed golden vectors generated from the reference.  Bit-exact: statuses,
task ids, servant indices, per-servant bookkeeping, unknown-id lists."""
import json
import os
from pathlib import Path

import numpy as np
import pytest

from golden_cases import ALL_CASES
from yadcc_b200 import streams as S
from yadcc_b200 import STATUS_GRANTED

pytestmark = pytest.mark.gpu
GOLDEN = Path(__file__).parent / "golden"


@pytest.mark.parametrize("case", ALL_CASES, ids=lambda f: f.__name__)
def test_reference_golden_cases_on_cuda(make_dispatcher, case):
    case(make_dispatcher("cuda"))


SOLVERS = {0: "auto", 1: "rowscan", 2: "stream"}  # auto = slot streams + the one-launch path for batches of <= 8


def _parity(make_dispatcher, name_or_builder, kinds=("port",), solver=0):
    traces = {}
    for kind in ("cuda",) + tuple(kinds):
        d = make_dispatcher(kind, solver=solver) if kind == "cuda" else make_dispatcher(kind)
        st = name_or_builder(d) if callable(name_or_builder) else S.named_stream(name_or_builder, d)
        traces[kind] = S.Replayer(d, pinned=(kind == "cuda")).run(st)
        d.close()
    for kind in kinds:
        assert S.traces_equal(traces["cuda"], traces[kind]), f"cuda vs {kind}: " + S.first_mismatch(
            traces["cuda"], traces[kind]
        )
    return traces["cuda"]


@pytest.mark.parametrize("solver", [0, 1, 2], ids=SOLVERS.get)
@pytest.mark.parametrize("seed", range(150))
def test_fuzz_cuda_equals_oracle(make_dispatcher, seed, solver):
    kinds = ("port", "ref") if seed % 3 == 0 else ("port",)
    _parity(make_dispatcher, lambda d: S.fuzz_stream(d, seed, n_servants=8 + seed % 30, wide=(seed % 5 == 0)), kinds,
            solver)


@pytest.mark.parametrize("seed", range(60))
def test_fuzz_packed_interface(make_dispatcher, seed):
    """yd_wait_for_starting_new_tasks_packed (16-byte requests up, 8-byte grants down, unpacked / packed by the
    fused kernel itself or by the conversion kernels around the pipeline) against the checkers' plain call."""
    traces = {}
    for kind in ("cuda", "port"):
        d = make_dispatcher(kind)
        st = S.fuzz_stream(d, seed, n_servants=8 + seed % 30, wide=(seed % 5 == 0))
        traces[kind] = S.Replayer(d, pinned=(kind == "cuda"), packed=(kind == "cuda")).run(st)
        d.close()
    assert S.traces_equal(traces["cuda"], traces["port"]), S.first_mismatch(traces["cuda"], traces["port"])


@pytest.mark.parametrize("fused", [True, False], ids=["fused", "pipeline"])
@pytest.mark.parametrize("packed", [True, False], ids=["packed", "plain"])
@pytest.mark.parametrize("name", ["cfg2-mod-small", "cfg2-random-small", "cfg3-small", "cfg-self-small", "cfg2-mod",
                                  "cfg2-random", "cfg-self"])
def test_fused_front_and_packed_interface_match_reference_digest(make_dispatcher, name, packed, fused):
    """The one-launch solve (fused.cuh; solo for cfg2-mod, fused front + coupled solvers for the others), with and
    without the packed interface, and the kernel-by-kernel pipeline behind the same interfaces: reference digests."""
    d = make_dispatcher("cuda", fused=fused)
    tr = S.Replayer(d, pinned=True, packed=packed).run(S.named_stream(name, d))
    golden = json.loads((GOLDEN / "digests.json").read_text())["streams"][name]
    assert S.trace_digest(tr) == golden["sha256"]


def _flip_stream(d, seed=7, n_servants=96, n_digests=4):
    """Batches that alternate between 'data-parallel components only' (the fused kernel finishes the solve alone) and
    'a requestor is a servant of its component' (it must stand down, flag 4, and the general sequence runs), with
    frees in between so that slots come back."""
    rng = np.random.default_rng(seed)
    w = S.config2(4000, n_servants, n_digests, seed=seed, variant="mod", max_tasks=24, nproc=64)
    ev = [("hb", 0.0, sv, 100.0) for sv in w.servants]
    env = np.asarray([d.intern_env(x) for x in w.digests], dtype=np.uint32)
    outside = np.asarray([d.intern_ip(f"172.16.0.{i}") for i in range(200)], dtype=np.uint32)
    inside = np.asarray([d.intern_ip(S.servant_ip(i)) for i in range(n_servants)], dtype=np.uint32)
    now = 0.001
    for k, kind in enumerate(["dp", "dp", "self", "dp", "dp", "self", "self", "dp", "tiny", "dp"]):
        n = int(rng.integers(300, 900)) if kind != "tiny" else 5
        ips = outside[rng.integers(0, len(outside), n)]
        if kind == "self":
            ips = np.where(rng.random(n) < 0.3, inside[rng.integers(0, n_servants, n)], ips)
        ev.append(("wait", now, S._requests(d, env[rng.integers(0, n_digests, n)], ips, 8,
                                            expires_in_s=float(rng.choice([0.5, 15.0])), prefetch=rng.random(n) < 0.2)))
        ev.append(("state",))
        ev.append(("free_frac", seed + k, 0.6))
        now += 0.01
    return S.Stream("flip", ev)


@pytest.mark.parametrize("packed", [True, False], ids=["packed", "plain"])
@pytest.mark.parametrize("graphs", [True, False], ids=["graph", "eager"])
def test_solo_kernel_stands_down_for_coupled_batches(make_dispatcher, packed, graphs):
    traces = {}
    for kind in ("cuda", "port"):
        d = make_dispatcher(kind, graphs=graphs) if kind == "cuda" else make_dispatcher(kind)
        traces[kind] = S.Replayer(d, pinned=(kind == "cuda"), packed=(packed and kind == "cuda")).run(_flip_stream(d))
        d.close()
    assert S.traces_equal(traces["cuda"], traces["port"]), S.first_mismatch(traces["cuda"], traces["port"])


@pytest.mark.parametrize("solver", [1, 2], ids=SOLVERS.get)
@pytest.mark.parametrize("seed", range(1000, 1012))
def test_fuzz_large_components(make_dispatcher, seed, solver):
    """Components above 256 servants use the multi-warp path of the row-scan solver."""
    _parity(make_dispatcher,
            lambda d: S.fuzz_stream(d, seed, n_servants=300 + 150 * (seed % 4), n_events=40, max_batch=600),
            solver=solver)


@pytest.mark.parametrize("seed", range(2000, 2000 + int(os.environ.get("YD_SOAK_SEEDS", "0"))))
def test_fuzz_soak(make_dispatcher, seed):
    """Opt-in soak (YD_SOAK_SEEDS=n): more large-component / many-class streams through the
    slot-stream solver than the default suite runs."""
    _parity(make_dispatcher,
            lambda d: S.fuzz_stream(d, seed, n_servants=40 + 97 * (seed % 9), n_events=50, max_batch=200 + 300 * (seed % 4),
                                    wide=(seed % 7 == 0)), solver=2)


@pytest.mark.parametrize("solver", [1, 2], ids=SOLVERS.get)
@pytest.mark.parametrize("name", ["cfg1", "cfg2-mod-small", "cfg2-random-small", "cfg3-small", "cfg3-mod-small",
                                  "cfg-self-small", "cfg-self"])
def test_small_configs(make_dispatcher, name, solver):
    tr = _parity(make_dispatcher, name, solver=solver)
    golden = json.loads((GOLDEN / "digests.json").read_text())["streams"]
    assert S.trace_digest(tr) == golden[name]["sha256"]


@pytest.mark.parametrize("solver", [1, 2], ids=SOLVERS.get)
@pytest.mark.parametrize("name", ["cfg2-mod", "cfg2-random"])
def test_full_size_configs_match_reference_digest(make_dispatcher, name, solver):
    """BASELINE.json configs[1] at full size against the digest produced by the
    reference itself (tests/golden/make_golden.py)."""
    d = make_dispatcher("cuda", solver=solver)
    tr = S.Replayer(d, pinned=True).run(S.named_stream(name, d))
    golden = json.loads((GOLDEN / "digests.json").read_text())["streams"][name]
    g = tr[0]
    assert int((g["status"] == STATUS_GRANTED).sum()) == golden["granted"]
    assert S.trace_digest(tr) == golden["sha256"]


@pytest.mark.parametrize("merge_self", [True, False], ids=["merge", "sequential"])
@pytest.mark.parametrize("name", ["cfg3", "cfg5-1m"])
def test_million_request_configs_match_reference_digest(make_dispatcher, name, merge_self):
    """BASELINE configs[2] at FULL size through its whole multi-round stream (1 M x 4 k; solve, free a
    seeded half, renew, re-heartbeat, tick, re-offer: 2.7 M decisions) and configs[4]'s 8 k-servant
    pool on the first 1 M requests of its queue, against the digests the reference itself produced
    (tests/golden/make_golden.py HUGE) -- once with the merge solver deciding the coupled component
    (20 % of the requestors are servants of it) and once with the sequential solver."""
    golden = json.loads((GOLDEN / "digests.json").read_text())["streams"]
    if name not in golden:
        pytest.skip(f"no reference digest for {name}")
    d = make_dispatcher("cuda", merge_self=merge_self)
    r = S.Replayer(d, pinned=True)
    tr = r.run(S.named_stream(name, d))
    assert (r.decisions, r.granted) == (golden[name]["decisions"], golden[name]["granted"])
    assert S.trace_digest(tr) == golden[name]["sha256"]


@pytest.mark.parametrize("merge_self", [True, False], ids=["merge", "sequential"])
@pytest.mark.parametrize("seed", range(3000, 3060))
def test_fuzz_one_daemon_per_machine(make_dispatcher, seed, merge_self):
    """Every servant on its own IP and many requestors that are servants: the merge solver's own-servant
    rule, passed-over (pending) requests and -- capacity is tiny here -- the last-resort hand-back to the
    sequential solver all get exercised; every third seed also against the reference itself."""
    kinds = ("port", "ref") if seed % 3 == 0 else ("port",)
    traces = {}
    for kind in ("cuda",) + kinds:
        d = make_dispatcher(kind, merge_self=merge_self) if kind == "cuda" else make_dispatcher(kind)
        st = S.fuzz_stream(d, seed, n_servants=6 + seed % 40, n_events=50, max_batch=30 + 40 * (seed % 5), unique_hosts=True)
        traces[kind] = S.Replayer(d).run(st)
        d.close()
    for kind in kinds:
        assert S.traces_equal(traces["cuda"], traces[kind]), f"cuda vs {kind}: " + S.first_mismatch(traces["cuda"], traces[kind])


@pytest.mark.parametrize("chunk,rounds", [(32, 2), (64, 3), (256, 8)])
@pytest.mark.parametrize("name", ["cfg2-random-small", "cfg-self-small", "cfg3-small"])
def test_merge_solver_tiny_chunks_and_round_escalation(make_dispatcher, monkeypatch, name, chunk, rounds):
    """Chunks far shorter than the healing length and too few rounds in the graph: the boundary states do
    not settle, the solve stands down, reruns with more rounds and finally with the sequential solver --
    the answers never change."""
    monkeypatch.setenv("YDSCHED_MERGE_CHUNK", str(chunk))
    monkeypatch.setenv("YDSCHED_MERGE_ROUNDS", str(rounds))
    tr = _parity(make_dispatcher, name)
    golden = json.loads((GOLDEN / "digests.json").read_text())["streams"]
    assert S.trace_digest(tr) == golden[name]["sha256"]


@pytest.mark.parametrize("burst", [3, 40, 400])
def test_merge_solver_bursts_from_one_servant(make_dispatcher, burst):
    """`make -j` on a machine that is itself a servant: long runs of consecutive requests from ONE servant's
    IP.  Its own slots pass the whole run over (a pending run), other servants' slots then serve it."""
    from yadcc_b200 import Servant, PRIORITY_USER

    results = []
    for kind in ("cuda", "port"):
        d = make_dispatcher(kind)
        dg = "ab" * 32
        for i in range(60):
            d.keep_servant_alive(Servant(f"10.9.0.{i}:8335", None, [dg], 8, 16, i % 3, 0, 64 << 30, 6 + i % 5, PRIORITY_USER),
                                 10.0, now=0.0)
        rng = np.random.default_rng(burst)
        who = []
        while len(who) < 500:
            who += [int(rng.integers(0, 60))] * int(rng.integers(1, burst + 1))
        ips = [f"10.9.0.{j}" if k % 7 else "172.16.0.1" for k, j in enumerate(who[:500])]
        reqs = d.make_requests(500, [dg] * 500, ips, np.full(500, 8, np.uint32))
        results.append(d.wait_for_starting_new_tasks(reqs, 0.5).copy())
        results.append(d.servant_state()["running_tasks"].copy())
    assert (results[0] == results[2]).all()
    assert (results[1] == results[3]).all()


@pytest.mark.parametrize("seed", range(0, 60, 2))
def test_batched_heartbeats_on_cuda(make_dispatcher, seed):
    """One tick's heartbeats as two calls (yd_keep_servants_alive, yd_notify_servants_running_tasks: one upload,
    one sweep + one check kernel, one sync) against the reference's one-call-per-servant sequence."""
    traces = {}
    for kind in ("cuda", "port"):
        d = make_dispatcher(kind)
        st = S.fuzz_stream(d, seed, n_servants=8 + seed % 30, n_events=80)
        # lengthen the notify runs: every servant reports after every tick
        ev = []
        for e in st.events:
            ev.append(e)
            if e[0] == "tick":
                ev += [("notify_own", i, 17 * seed + i, [i, 10_000 + i]) for i in range(8 + seed % 30)]
                ev += [("notify_own", 0, 5, []), ("notify", "203.0.113.9:1", [(1, 3, "aa")])]  # a repeat and a stranger
        traces[kind] = S.Replayer(d, batch_heartbeats=(kind == "cuda")).run(S.Stream(st.name, ev))
        d.close()
    assert S.traces_equal(traces["cuda"], traces["port"]), S.first_mismatch(traces["cuda"], traces["port"])


def test_heartbeat_reporting_ten_thousand_tasks(make_dispatcher):
    """A heartbeat may list any number of running tasks (the reference takes whatever arrives,
    task_dispatcher.cc:222-277), zombies or not: 10 000 ids, most of them bogus, with zombies present."""
    from yadcc_b200 import PRIORITY_USER, RunningTask, Servant

    out = []
    for kind in ("cuda", "port"):
        d = make_dispatcher(kind)
        dg = "cd" * 32
        for i in range(4):
            d.keep_servant_alive(Servant(f"10.8.0.{i}:8335", None, [dg], 8, 64, 0, 0, 64 << 30, 40, PRIORITY_USER), 100.0, now=0.0)
        g = d.wait_for_starting_new_tasks(d.make_requests(120, dg, "172.16.0.1", 8, expires_in=1.0), 0.0)
        d.on_expiration_timer(now=5.0)  # every lease expired: 120 zombies
        mine = [int(t) for t, sidx in zip(g["task_id"], g["servant_index"]) if sidx == 1]
        ids = mine[::2] + list(range(1000, 1000 + 10_000))
        loc = "10.8.0.1:8335"
        unknown = d.notify_servant_running_tasks(loc, [RunningTask(k, t, loc, f"{t:064x}") for k, t in enumerate(ids)])
        st = d.servant_state()
        out.append((unknown, st["running_tasks"].tolist(), d.num_tasks()))
    assert out[0] == out[1]


@pytest.mark.parametrize("seed", [3, 11])
def test_dump_internals_on_cuda(make_dispatcher, seed):
    """DumpInternals (task_dispatcher.cc:538-614): per-servant rows and summary of the CUDA backend against the
    reference's own function after the same stream."""
    dumps = []
    for kind in ("cuda", "ref"):
        d = make_dispatcher(kind)
        S.Replayer(d).run(S.fuzz_stream(d, seed, n_servants=12 + seed))
        dumps.append(d.dump_internals())
    assert dumps[0] == dumps[1]


def test_thirty_thousand_servants_behind_one_digest(make_dispatcher):
    """One compiler digest on 30 000 servants is ONE component: the merge solver has no per-component size limit and
    the sequential solver keeps running_tasks of such a component in HBM instead of shared memory (no abort).  Every
    requestor is a servant (self rule live); then the same with two servants behind one requestor IP, which forces the
    sequential solver."""
    from yadcc_b200 import PRIORITY_DEDICATED, PRIORITY_USER, Servant

    dg = "ef" * 32
    for twin in (False, True):
        results = []
        for kind in ("cuda", "port"):
            d = make_dispatcher(kind)
            r = np.random.default_rng(5)
            svs = [Servant(f"10.{i >> 16}.{(i >> 8) & 255}.{i & 255}:8335", None, [dg], 8, int(r.choice([8, 16, 32])), int(r.integers(0, 4)),
                           0, 64 << 30, int(r.integers(1, 5)), PRIORITY_DEDICATED if i % 9 == 0 else PRIORITY_USER) for i in range(30_000)]
            if twin:
                svs.append(Servant("10.0.0.7:9000", None, [dg], 8, 16, 0, 0, 64 << 30, 3, PRIORITY_USER))
            d.keep_servants_alive(svs, 10.0, now=0.0)
            n = 40_000
            who = r.integers(0, 30_000, n)
            ips = [f"10.{j >> 16}.{(j >> 8) & 255}.{j & 255}" for j in who]
            if twin:
                ips[::50] = ["10.0.0.7"] * len(ips[::50])
            reqs = d.make_requests(n, dg, ips, 8)
            results.append(d.wait_for_starting_new_tasks(reqs, 0.5).copy())
            results.append(d.servant_state()["running_tasks"].copy())
        assert (results[0] == results[2]).all()
        assert (results[1] == results[3]).all()


def test_cfg1_vectors(make_dispatcher):
    z = np.load(GOLDEN / "cfg1_reference.npz")
    d = make_dispatcher("cuda")
    g = S.Replayer(d).run(S.named_stream("cfg1", d))[0]
    for k in ("status", "task_id", "servant_index"):
        assert (g[k] == z[k]).all(), k


def test_cfg3_million_properties(make_dispatcher):
    """1 M x 4 k (BASELINE configs[2]) through size-independent properties: ids are
    the grant ordinals, per-servant running counts equal the grants they received
    and never exceed capacity, a second offer of the same queue grants nothing,
    and the oracle agrees on a 50 k-request prefix."""
    w = S.config3(1_000_000, 4000, 8)
    d = make_dispatcher("cuda")
    w.register(d)
    reqs = w.build_requests(d)
    g = d.wait_for_starting_new_tasks(reqs, 0.001)
    ok = g["status"] == STATUS_GRANTED
    n_ok = int(ok.sum())
    assert (g["task_id"][ok] == np.arange(n_ok, dtype=np.uint64)).all()
    st = d.servant_state()
    counts = np.bincount(g["servant_index"][ok], minlength=len(st))
    assert (st["running_tasks"] == counts).all()
    assert (st["ever_assigned_tasks"] == counts).all()
    assert d.num_tasks() == n_ok and d.next_task_id() == n_ok
    # every servant that got work stayed within its capacity model
    assert (st["running_tasks"][counts > 0] <= st["capacity_available"][counts > 0]).all()
    # idempotence: the queue that timed out times out again (nothing was freed)
    pend = reqs[g["status"] == 1]
    g2 = d.wait_for_starting_new_tasks(pend[:200_000], 0.002)
    assert not (g2["status"] == STATUS_GRANTED).any()
    # prefix against the oracle
    d2, o = make_dispatcher("cuda"), make_dispatcher("port")
    for x in (d2, o):
        w.register(x)
    r2, ro = w.build_requests(d2)[:50_000], w.build_requests(o)[:50_000]
    a, b = d2.wait_for_starting_new_tasks(r2, 0.001), o.wait_for_starting_new_tasks(ro, 0.001)
    assert (a == b).all()


def test_lease_ring_growth_and_window(make_dispatcher):
    """More leases than the initial ring (65536) and a sliding window."""
    traces = []
    for kind in ("cuda", "port"):
        d = make_dispatcher(kind)
        w = S.config2(150_000, 2500, 4, variant="mod", max_tasks=64, nproc=128)
        ev = [("hb", 0.0, sv, 30.0) for sv in w.servants]
        ev += [("enqueue", w.build_requests(d)), ("solve", 0.001), ("free_frac", 7, 0.9), ("tick", 1.0),
               ("enqueue", w.build_requests(d)), ("solve", 1.5), ("keepalive", 2.0, None, 1.0), ("tick", 20.0),
               ("state",), ("free_frac", 8, 0.5), ("tick", 21.0), ("state",)]
        traces.append(S.Replayer(d).run(S.Stream("ring", ev)))
        d.close()
    assert S.traces_equal(*traces), S.first_mismatch(*traces)


def test_native_library_is_what_ran(make_dispatcher):
    d = make_dispatcher("cuda")
    assert d.backend == "cuda-sm100a"
    w = S.config1()
    w.register(d)
    d.wait_for_starting_new_tasks(w.build_requests(d), 0.0)
    st = d.last_solve_stats()
    assert st["kernel_launches"] >= 4 and st["solver"] in (1, 2) and st["decisions"] == 1000
    maps = Path("/proc/self/maps").read_text()
    assert "libydsched.so" in maps


@pytest.mark.parametrize("n_classes", [40, 300])
def test_many_classes(make_dispatcher, n_classes):
    """More (digest, min_version) classes than the solver provisions for: 40 grows the
    class bound and retries; 300 exceeds the class table and falls back to the row-scan
    solver.  Either way the answers are the reference's."""
    import numpy as np
    from yadcc_b200 import Servant, PRIORITY_USER, PRIORITY_DEDICATED

    rng = np.random.default_rng(n_classes)
    digests = [f"{i:064x}" for i in range(n_classes // 2)]
    results = []
    for kind in ("cuda", "port"):
        d = make_dispatcher(kind)
        r = np.random.default_rng(7)
        for i in range(400):
            envs = [digests[j] for j in r.choice(len(digests), size=int(r.integers(1, 4)), replace=False)]
            d.keep_servant_alive(
                Servant(f"10.3.{i >> 8}.{i & 255}:8335", None, envs, int(r.choice([7, 8])), 16, int(r.integers(0, 6)),
                        0, 64 << 30, int(r.integers(0, 9)), PRIORITY_DEDICATED if i % 7 == 0 else PRIORITY_USER),
                10.0, now=0.0)
        n = 6000
        reqs = d.make_requests(n, [digests[j] for j in r.integers(0, len(digests), n)],
                               [f"10.3.{j >> 8}.{j & 255}" if k % 5 == 0 else "172.16.0.9"
                                for k, j in enumerate(r.integers(0, 400, n))],
                               r.choice([7, 8], n).astype(np.uint32))
        results.append(d.wait_for_starting_new_tasks(reqs, 0.5).copy())
        results.append(d.servant_state()["running_tasks"].copy())
    assert (results[0] == results[2]).all()
    assert (results[1] == results[3]).all()


@pytest.mark.parametrize("packed", [False, True], ids=["plain", "packed"])
def test_many_classes_on_a_component_beyond_the_rowscan_solver(make_dispatcher, packed):
    """300 (digest, min_version) classes overflow the class table while one component has 9000 servants, more than
    the row-scan fallback holds: the batch is decided as consecutive halves (sequential decisions compose)."""
    import numpy as np
    from yadcc_b200 import Servant, PRIORITY_USER, pack_requests

    dg = "ab" * 32
    results = []
    for kind in ("cuda", "port"):
        d = make_dispatcher(kind)
        r = np.random.default_rng(3)
        d.keep_servants_alive(
            [Servant(f"10.{i >> 16}.{(i >> 8) & 255}.{i & 255}:8335", None, [dg], int(r.integers(1, 300)), 8, int(r.integers(0, 4)),
                     0, 64 << 30, int(r.integers(0, 3)), PRIORITY_USER) for i in range(9000)], 10.0, now=0.0)
        n = 3000
        reqs = d.make_requests(n, dg, [f"10.0.{j >> 8}.{j & 255}" if k % 7 == 0 else "172.16.0.9"
                                       for k, j in enumerate(r.integers(0, 9000, n))],
                               r.integers(1, 301, n).astype(np.uint32))
        if packed and kind == "cuda":
            results.append(d.wait_for_starting_new_tasks_packed(pack_requests(reqs), 0.5).copy())
        else:
            results.append(d.wait_for_starting_new_tasks(reqs, 0.5).copy())
        results.append(d.servant_state()["running_tasks"].copy())
    assert (results[0] == results[2]).all()
    assert (results[1] == results[3]).all()


@pytest.mark.parametrize("seed", range(8))
def test_merge_solver_coupled_no_self(make_dispatcher, seed):
    """Coupled components whose requestors are NOT servants take the merge solver
    (slots pick the earliest unserved compatible request).  Mixed versions, dedicated
    servants, low memory, capacity below demand (Timeouts), a digest nobody can serve
    (EnvironmentNotFound), several independent coupled components, and a component with
    more than 32 classes (falls back to the sequential solver)."""
    import numpy as np
    from yadcc_b200 import Servant, PRIORITY_USER, PRIORITY_DEDICATED

    rng = np.random.default_rng(100 + seed)
    n_groups = 1 + seed % 3                     # independent coupled components
    digs = [[f"{g:02x}{i:062x}" for i in range(int(rng.integers(2, 7)))] for g in range(n_groups)]
    many_versions = seed == 5                   # > 32 (digest, min_version) classes in one component
    results = []
    for kind in ("cuda", "port"):
        d = make_dispatcher(kind)
        r = np.random.default_rng(200 + seed)
        k = 0
        for g in range(n_groups):
            for _ in range(int(r.integers(30, 400))):
                envs = [digs[g][j] for j in r.choice(len(digs[g]), size=int(r.integers(1, len(digs[g]) + 1)), replace=False)]
                nproc = int(r.choice([8, 16, 32]))
                d.keep_servant_alive(
                    Servant(f"10.5.{k >> 8}.{k & 255}:8335", None, envs, int(r.choice([6, 7, 8, 9])), nproc,
                            int(r.integers(0, nproc + 2)), int(r.choice([0, 64 << 30])),
                            int(r.choice([5 << 30, 40 << 30, 40 << 30])), int(r.integers(0, nproc)),
                            PRIORITY_DEDICATED if r.random() < 0.15 else PRIORITY_USER), 10.0, now=0.0)
                k += 1
        n = int(r.integers(500, 6000))
        all_d = [x for g in digs for x in g] + ["ee" * 32]
        mv = r.integers(0, 40, n).astype(np.uint32) if many_versions else r.choice([0, 7, 8, 9], n).astype(np.uint32)
        reqs = d.make_requests(n, [all_d[j] for j in r.integers(0, len(all_d), n)],
                               [f"172.20.{j >> 8}.{j & 255}" for j in r.integers(0, 3000, n)], mv)
        results.append(d.wait_for_starting_new_tasks(reqs, 0.5).copy())
        # a second batch continues from the state the first one left
        results.append(d.wait_for_starting_new_tasks(reqs[: n // 2], 0.6).copy())
        st = d.servant_state()
        results.append(np.stack([st["running_tasks"], st["ever_assigned_tasks"]], 1))
    for a, b in zip(results[:3], results[3:]):
        assert (a == b).all()


@pytest.mark.parametrize("seed", range(12))
def test_rpc_expansion_cuda_equals_oracle(make_dispatcher, seed):
    """yd_wait_for_starting_task_rpcs (the caller's request expansion,
    scheduler_service_impl.cc:209-271) on the CUDA backend against the oracle."""
    from rpc_cases import run_rpc_stream

    a = run_rpc_stream(make_dispatcher("cuda"), seed)
    b = run_rpc_stream(make_dispatcher("ref"), seed)
    for x, y in zip(a, b):
        assert x.shape == y.shape and (x == y).all()


def test_strided_task_ids(make_dispatcher):
    """Sharded deployments: yd_config.id_stride / id_offset make a handle hand out and accept
    ids of the form local * stride + offset, so shards share one id space without talking.
    Everything except the numbering must equal an unsharded handle."""
    import numpy as np

    w = S.config2(3000, 60, 4, variant="random", max_tasks=8, nproc=16)
    plain = make_dispatcher("cuda")
    shard = [make_dispatcher("cuda", id_stride=4, id_offset=k) for k in (1, 3)]
    for d in [plain] + shard:
        w.register(d)
    base = plain.wait_for_starting_new_tasks(w.build_requests(plain), 0.1).copy()
    ok = base["status"] == STATUS_GRANTED
    outs = []
    for k, d in zip((1, 3), shard):
        g = d.wait_for_starting_new_tasks(w.build_requests(d), 0.1).copy()
        assert (g["status"] == base["status"]).all() and (g["servant_index"] == base["servant_index"]).all()
        assert (g["task_id"][ok] == base["task_id"][ok] * 4 + k).all()
        assert d.next_task_id() == plain.next_task_id() * 4 + k
        outs.append(g)
    # each shard ignores the other's ids (and plain garbage) in FreeTask / KeepTaskAlive / heartbeats
    mixed = np.concatenate([outs[0]["task_id"][ok][:50], outs[1]["task_id"][ok][:70], [7, 8, 2**40]]).astype(np.uint64)
    for d in shard:
        alive = d.keep_tasks_alive(mixed, 5.0, now=0.2)
        d.free_tasks(mixed)
    assert shard[0].num_tasks() == int(ok.sum()) - 50 and shard[1].num_tasks() == int(ok.sum()) - 70
    plain.free_tasks(base["task_id"][ok][:50])
    assert (shard[0].servant_state()["running_tasks"] == plain.servant_state()["running_tasks"]).all()
    loc = shard[0].servant_location(int(outs[0]["servant_index"][ok][60]))
    from yadcc_b200 import RunningTask
    mine = int(outs[0]["task_id"][ok][60])
    other = int(outs[1]["task_id"][ok][60])
    unknown = shard[0].notify_servant_running_tasks(loc, [RunningTask(1, mine, loc, "a"), RunningTask(2, other, loc, "b")])
    assert unknown == [other]
    # the CPU restatement implements the same option: identical ids, answers and state
    twin = make_dispatcher("port", id_stride=4, id_offset=1)
    w.register(twin)
    g = twin.wait_for_starting_new_tasks(w.build_requests(twin), 0.1)
    assert (g == outs[0]).all()
    assert (twin.keep_tasks_alive(mixed, 5.0, now=0.2) == np.concatenate([np.ones(50, bool), np.zeros(73, bool)])).all()
    twin.free_tasks(mixed)
    assert twin.notify_servant_running_tasks(loc, [RunningTask(1, mine, loc, "a"), RunningTask(2, other, loc, "b")]) == [other]
    assert (twin.servant_state() == shard[0].servant_state()).all() and twin.next_task_id() == shard[0].next_task_id()


@pytest.mark.parametrize("seed", range(2))
def test_bloom_prefilter_cuda_equals_oracle(make_dispatcher, seed):
    """SURVEY 8(f) row 1: flare's SaltedBloomFilter (10 x XXH64(salt || key), 2^25 bits) on
    the GPU: identical filter bytes after Add, identical lookups (false positives included),
    all key lengths, tiny geometries, imported filters."""
    from bloom_cases import run_bloom_suite

    a = run_bloom_suite(make_dispatcher("cuda"), seed)
    b = run_bloom_suite(make_dispatcher("ref"), seed)
    assert len(a) == len(b)
    for k, (x, y) in enumerate(zip(a, b)):
        assert x.shape == y.shape and (x == y).all(), k


def test_cfg4_trace_with_bloom_prefilter(make_dispatcher):
    """BASELINE configs[3]: 100 k requests replaying 6124 TU keys, cache bloom filter on.
    Requests whose cache key may be in the cache are dropped before the solver (the delegate
    daemon does this, distributed_cache_reader.cc:70-77), requests whose task digest is
    already being compiled somewhere join that task instead (running_task_keeper.cc:67-75,
    distributed_task_dispatcher.cc:257); the rest is solved as config 2."""
    import numpy as np
    from bloom_cases import tu_keys
    from running_index_cases import task_digests
    from yadcc_b200 import RunningTask

    keys = tu_keys(6124)
    digests = task_digests(6124, 11)  # the task digest of TU i (task_digest.cc:25-31)
    rng = np.random.default_rng(4)
    cached = [k for k, m in zip(keys, rng.random(len(keys)) < 0.3) if m]
    n = 100_000
    tu = np.arange(n) % len(keys)
    trace = [keys[i] for i in tu]
    trace_digests = [digests[i] for i in tu]
    results = []
    for kind in ("cuda", "port"):
        d = make_dispatcher(kind)
        w = S.config2(n, 2000, 8, variant="mod")
        w.register(d)
        d.bloom_reset()
        d.bloom_add(cached)
        # an earlier wave is still compiling: its servants list those tasks in their heartbeats
        all_reqs = w.build_requests(d)
        early = d.wait_for_starting_new_tasks(all_reqs[:1500].copy(), 0.25)
        locs = [d.servant_location(i) for i in range(2000)]
        by_servant = {}
        for j, gr in enumerate(early):
            assert gr["status"] == 2
            by_servant.setdefault(int(gr["servant_index"]), []).append(
                RunningTask(j + 1, int(gr["task_id"]), locs[int(gr["servant_index"])], digests[5000 - j]))
        for si, tasks in by_servant.items():
            d.notify_servant_running_tasks(locs[si], tasks)
        d.running_index_refresh()
        hit = d.bloom_possibly_contains(trace)
        joined = d.find_running_tasks(trace_digests)
        keep = ~hit & (joined["found"] == 0)
        g = d.wait_for_starting_new_tasks(all_reqs[keep], 0.5)
        results.append((hit.copy(), joined.copy(), g.copy()))
    assert (results[0][0] == results[1][0]).all()
    assert (results[0][1] == results[1][1]).all()
    assert (results[0][2] == results[1][2]).all()
    assert 0.25 < results[0][0].mean() < 0.35
    assert 0.15 < results[0][1]["found"].mean() < 0.35


@pytest.mark.parametrize("stages", ["both", "bloom", "dedupe", "none"])
def test_cfg4_prefiltered_solve_in_one_call(make_dispatcher, stages):
    """yd_filter_and_wait_for_starting_new_tasks (bloom probes, in-flight index probes, compaction and solve with the
    queue resident in HBM) against the checker, whose version of the call is its definition: the three calls in order."""
    import numpy as np
    from bloom_cases import tu_keys
    from running_index_cases import task_digests
    from yadcc_b200 import RunningTask

    keys = tu_keys(6124)
    digests = task_digests(6124, 11)
    rng = np.random.default_rng(4)
    cached = [k for k, m in zip(keys, rng.random(len(keys)) < 0.3) if m]
    n = 30_000
    tu = np.arange(n) % len(keys)
    trace = [keys[i] for i in tu] if stages in ("both", "bloom") else None
    trace_digests = [digests[i] for i in tu] if stages in ("both", "dedupe") else None
    results = []
    for kind in ("cuda", "port"):
        d = make_dispatcher(kind)
        w = S.config2(n, 600, 8, variant="mod", max_tasks=24)
        w.register(d)
        d.bloom_reset()
        d.bloom_add(cached)
        all_reqs = w.build_requests(d)
        early = d.wait_for_starting_new_tasks(all_reqs[:900].copy(), 0.25)
        locs = [d.servant_location(i) for i in range(600)]
        by_servant = {}
        for j, gr in enumerate(early):
            by_servant.setdefault(int(gr["servant_index"]), []).append(
                RunningTask(j + 1, int(gr["task_id"]), locs[int(gr["servant_index"])], digests[5000 - j]))
        d.notify_servants_running_tasks([(locs[si], tasks) for si, tasks in by_servant.items()])
        d.running_index_refresh()
        verdict, hits, g = d.filter_and_wait_for_starting_new_tasks(all_reqs, trace, trace_digests, 0.5)
        results.append((verdict.copy(), hits.copy(), g.copy(), d.servant_state()["running_tasks"].copy()))
    for a, b in zip(results[0], results[1]):
        assert a.shape == b.shape and (a == b).all()
    v = results[0][0]
    assert (v == 0).sum() == len(results[0][2])
    if stages == "both":
        assert (v == 1).any() and (v == 2).any()


@pytest.mark.gpu
@pytest.mark.parametrize("seed", range(3))
def test_running_index_matches_oracle(make_dispatcher, seed):
    """In-flight task index (RunningTaskKeeper): device hash table vs the CPU restatement."""
    from running_index_cases import run_suite

    a = run_suite(make_dispatcher("cuda"), seed)
    b = run_suite(make_dispatcher("port"), seed)
    assert len(a) == len(b)
    for k, (x, y) in enumerate(zip(a, b)):
        assert x.shape == y.shape and (x == y).all(), k


@pytest.mark.gpu
def test_running_index_reference_test_and_scale(make_dispatcher):
    """running_task_keeper_test.cc's own scenario, then a 2000-servant cluster with ~30 k
    in-flight tasks (many duplicate digests) probed by a 100 k-entry queue."""
    import numpy as np
    from running_index_cases import populate, reference_test_case, task_digests

    first, second = reference_test_case(make_dispatcher("cuda"))
    assert first["found"].all() and list(first["servant_task_id"]) == [0, 1, 2]
    assert not second["found"].any()

    pool = task_digests(12000, 3)
    queue = [pool[i % len(pool)] for i in range(60_000)] + task_digests(40_000, 4)
    res = []
    for kind in ("cuda", "port"):
        d = make_dispatcher(kind)
        populate(d, 2000, 8, pool, seed=1)  # 2000 servants, 8000 grants
        n = d.running_index_refresh()
        res.append((n, d.running_index_size(), d.find_running_tasks(queue)))
    assert res[0][0] == res[1][0] > 7000 and res[0][1] == res[1][1]
    assert (res[0][2] == res[1][2]).all()
    assert 0.1 < res[0][2]["found"].mean() < 0.6


@pytest.mark.gpu
def test_service_layer_over_cuda_backend(make_dispatcher):
    """SchedulerServiceImpl's handlers (include/ydservice.h) over the CUDA dispatcher give the
    same answers as over the CPU restatement, for every case of tests/service_cases.py."""
    import service_cases as SC
    from test_service import CASES, _same

    for case in CASES:
        assert _same(case(make_dispatcher("cuda")), case(make_dispatcher("port"))), case.__name__


@pytest.mark.gpu
def test_staged_queue_equals_direct_call(make_dispatcher):
    """yd_stage_requests + yd_wait_for_staged_tasks == yd_wait_for_starting_new_tasks, also for a
    prefix of the staged queue and after an un-staged call in between."""
    import numpy as np

    w = S.config2(30_000, 600, 8, variant="random")
    outs = []
    for mode in ("direct", "staged"):
        d = make_dispatcher("cuda")
        w.register(d)
        reqs = w.build_requests(d)
        res = []
        if mode == "direct":
            res.append(d.wait_for_starting_new_tasks(reqs[:20_000].copy(), 0.5).copy())
            res.append(d.wait_for_starting_new_tasks(reqs[20_000:].copy(), 0.6).copy())
            res.append(d.wait_for_starting_new_tasks(reqs[:5_000].copy(), 0.7).copy())
        else:
            d.stage_requests(reqs)
            res.append(d.wait_for_staged_tasks(20_000, 0.5).copy())          # a prefix of the staged queue
            res.append(d.wait_for_starting_new_tasks(reqs[20_000:].copy(), 0.6).copy())  # un-staged call in between
            d.stage_requests(reqs[:5_000].copy())
            res.append(d.wait_for_staged_tasks(5_000, 0.7).copy())
        outs.append(res)
    for a, b in zip(*outs):
        assert (a == b).all()


@pytest.mark.gpu
def test_late_class_bound_overflow_leaves_no_trace(make_dispatcher):
    """16 classes fit the initial class bound, but three merge-mode components need three more
    list slots: the overflow is only noticed after the single-class components were marked
    data-parallel.  The aborted attempt must not count anything (running_tasks, task ids):
    the retry with a bigger bound has to give the reference's answers and state."""
    import numpy as np
    from yadcc_b200 import Servant

    digests = [f"{i:064x}" for i in range(16)]
    results = []
    for kind in ("cuda", "port"):
        d = make_dispatcher(kind)
        k = 0
        for c in range(10):  # ten single-digest components
            for _ in range(6):
                d.keep_servant_alive(Servant(f"10.5.{k >> 8}.{k & 255}:8335", None, [digests[c]], 8, 16, 0, 0, 64 << 30, 8),
                                     10.0, now=0.0)
                k += 1
        for c in range(3):  # three components coupling two digests each
            for j in range(8):
                envs = [digests[10 + 2 * c], digests[11 + 2 * c]] if j % 2 else [digests[10 + 2 * c + j // 4 % 2]]
                d.keep_servant_alive(Servant(f"10.5.{k >> 8}.{k & 255}:8335", None, envs, 8, 16, 0, 0, 64 << 30, 8),
                                     10.0, now=0.0)
                k += 1
        rng = np.random.default_rng(3)
        n = 4000
        for rnd in range(2):
            reqs = d.make_requests(n, [digests[j] for j in rng.integers(0, 16, n)], "172.16.0.9", 8)
            results.append(d.wait_for_starting_new_tasks(reqs, 0.5 + rnd).copy())
            results.append(d.servant_state()["running_tasks"].copy())
    h = len(results) // 2
    for a, b in zip(results[:h], results[h:]):
        assert (a == b).all()


@pytest.mark.gpu
def test_wire_front_end_over_cuda_backend(make_dispatcher):
    """FlareStd frames in, frames out (include/ydwire.h) over the CUDA dispatcher: every response
    frame equals, byte for byte, the one produced over the CPU restatement."""
    pytest.importorskip("google.protobuf")
    from wire_cases import run_wire_scenario

    assert run_wire_scenario(make_dispatcher, "cuda") == run_wire_scenario(make_dispatcher, "port")


@pytest.mark.gpu
def test_c_example_against_cuda_library(tmp_path):
    """examples/minimal.c linked against the product library."""
    import subprocess

    from conftest import CUDA_LIB, ROOT

    exe = tmp_path / "minimal"
    r = subprocess.run(["gcc", "-std=c99", "-Wall", "-Werror", f"-I{ROOT / 'include'}", str(ROOT / "examples" / "minimal.c"), "-o",
                        str(exe), str(CUDA_LIB), f"-Wl,-rpath,{CUDA_LIB.parent}"], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    r = subprocess.run([str(exe)], capture_output=True, text=True, timeout=120)
    assert r.returncode == 0, r.stdout + r.stderr
    assert r.stdout.strip().endswith("ok") and "request 4 -> timeout" in r.stdout
