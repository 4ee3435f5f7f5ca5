"""SchedulerServiceImpl restatement over the C ABI, on the CPU backends.  The handlers need
flare's RPC controller and protobuf, so scheduler_service_impl.cc is not compilable here: the
rules are pinned on the reference's own test (scheduler_service_impl_test.cc) and on the
handler source line by line; the dispatcher underneath is the verbatim reference (`ref`) or the
restatement (`port`), and both must agree on everything observable."""
import numpy as np
import pytest

import service_cases as SC

CASES = [SC.token_case, SC.token_with_intersection_case, SC.token_without_intersection_case, SC.heartbeat_rules_case,
         SC.lease_flow_case, SC.token_rollout_case]


def _same(a, b):
    if isinstance(a, np.ndarray):
        return a.shape == b.shape and a.dtype == b.dtype and (a == b).all()
    if isinstance(a, (list, tuple)):
        return len(a) == len(b) and all(_same(x, y) for x, y in zip(a, b))
    return a == b


@pytest.mark.parametrize("case", CASES, ids=lambda c: c.__name__)
def test_service_case(make_dispatcher, reference, case):
    a = case(make_dispatcher("ref"))
    reference.observe(a)
    b = case(make_dispatcher("port"))
    assert _same(a, b)


def test_service_needs_both_token_lists(make_dispatcher):
    from yadcc_b200.service import SchedulerService

    d = make_dispatcher("port")
    with pytest.raises(ValueError):
        SchedulerService(d, acceptable_user_tokens="", acceptable_servant_tokens="x")
    with pytest.raises(ValueError):
        SchedulerService(d, acceptable_user_tokens="x", acceptable_servant_tokens="")
    # "a," keeps the empty entry: the empty token is then acceptable (token_verifier.cc:61, keep_empty)
    svc = SchedulerService(d, acceptable_user_tokens="a,", acceptable_servant_tokens="s")
    assert svc.get_config("")[0] == 0 and svc.get_config("b")[0] == 1003


# ---- the C restatement against a second, independent restatement (tests/service_model.py) ----------------------

def _service_fuzz(make_dispatcher, kind_c: str, kind_model: str, seed: int, n_ops: int = 260):
    """Random request stream through (a) include/ydservice_impl.inc over backend `kind_c` and (b) the Python model of
    scheduler_service_impl.cc over backend `kind_model`; everything observable must agree, step by step."""
    from service_model import ServiceModel
    from yadcc_b200 import RunningTask, _abi
    from yadcc_b200.service import HeartbeatRequest, SchedulerService

    rng = np.random.default_rng(seed)
    user_flag, servant_flag = [("u1,u2", "s1,u2"), ("u1", "s1"), ("u1,", "s1,s2")][seed % 3]
    interval = int(rng.choice([2, 5, 3600]))
    min_version = int(rng.choice([0, 3]))
    da, db = make_dispatcher(kind_c), make_dispatcher(kind_model)
    svc = SchedulerService(da, acceptable_user_tokens=user_flag, acceptable_servant_tokens=servant_flag,
                           min_daemon_version=min_version, serving_daemon_token_rollout_interval=interval, token_seed=seed + 1)
    model = ServiceModel(db, acceptable_user_tokens=user_flag, acceptable_servant_tokens=servant_flag,
                         min_daemon_version=min_version, serving_daemon_token_rollout_interval=interval)
    tokens = ["u1", "u2", "s1", "s2", "", "bad"]
    digests = [f"{i:02x}" * 32 for i in range(4)]
    seen_tokens: dict[int, str] = {}  # serving-daemon tokens of the C side by generation: window after k rolls = generations k, k+1, k+2
    granted: list[int] = []
    now = 0.0

    def check_window(rolls, triple=None, middle=None):
        if triple is not None:
            for j, t in enumerate(triple):
                assert seen_tokens.setdefault(rolls + j, t) == t, "serving-daemon token window rolled differently"
            assert len(set(triple)) == 3
        if middle is not None:
            assert seen_tokens.setdefault(rolls + 1, middle) == middle, "serving-daemon token window rolled differently"
        assert len(set(seen_tokens.values())) == len(seen_tokens)  # (every generation is a fresh token)

    def servant_ip(k):
        return f"10.7.{k >> 8}.{k & 255}"

    for step in range(n_ops):
        now += float(rng.choice([0.0, 0.05, 0.4, 1.1, 2.6]))
        op = rng.choice(["hb", "hb", "hb", "wait", "wait", "batch", "keep", "free", "config", "running", "tick"])
        if op == "hb":
            k = int(rng.integers(0, 12))
            ip = servant_ip(k)
            loc = rng.choice([f"{ip}:8335", f"{ip}:8335", f"{ip}:8335", f"192.168.1.{k}:8335", "nonsense", f"{ip}:99999", f"{ip}",
                              f"0{ip}:80", "[::1]:8335", f"{ip}:"])
            v6 = bool(loc.startswith("[") and rng.random() < 0.7)
            running = []
            if granted and rng.random() < 0.5:
                for t in rng.choice(granted, size=min(len(granted), 3), replace=False):
                    running.append(RunningTask(int(rng.integers(1, 99)), int(t), str(loc), f"{int(t):064x}"))
            if rng.random() < 0.3:
                running.append(RunningTask(7, int(rng.integers(10**6, 10**7)), str(loc), "ee" * 32))
            req = HeartbeatRequest(
                token=str(rng.choice(tokens)), location=str(loc), remote_ip="::1" if v6 else ip, remote_is_ipv6=v6,
                next_heartbeat_in_ms=int(rng.choice([0, 1000, 5000, 30000, 30001])), version=int(rng.integers(0, 8)),
                num_processors=int(rng.choice([0, 4, 16])), current_load=int(rng.integers(0, 6)),
                servant_priority=int(rng.choice([0, 1, 2, 9])), not_accepting_task_reason=int(rng.choice([0, 1, 3])),
                capacity=int(rng.choice([0, 2, 8])), total_memory_in_bytes=int(rng.choice([0, 64 << 30])),
                memory_available_in_bytes=int(rng.choice([1 << 30, 32 << 30])),
                env_digests=[digests[j] for j in rng.choice(4, size=int(rng.integers(0, 4)), replace=False)],
                running_tasks=running)
            a, b = svc.heartbeat(req, now=now), model.heartbeat(req, now=now)
            assert a.status == b.status, (step, req)
            if a.status == 0:
                assert a.expired_tasks == b.expired_tasks, (step, req)
                check_window(b.rolls, triple=a.acceptable_tokens)
        elif op in ("wait", "batch"):
            n_rpc = 1 if op == "wait" else int(rng.integers(2, 6))
            toks, rows = [], []
            for _ in range(n_rpc):
                toks.append(str(rng.choice(["u1", "u1", "u2", "s1", "bad"])))
                dg = digests[int(rng.integers(0, 4))] if rng.random() < 0.9 else "77" * 32
                ip = servant_ip(int(rng.integers(0, 12))) if rng.random() < 0.4 else "172.16.3.3"
                rows.append((dg, int(rng.integers(0, 8)), ip, int(rng.choice([0, 1, 1, 2, 5])), int(rng.choice([0, 0, 1, 3])),
                             int(rng.choice([0, 100, 10000, 10001])), int(rng.choice([1, 15, 30, 31])) * 1_000_000_000))
            per = []
            for d in (da, db):
                r = np.zeros(n_rpc, dtype=_abi.RPC_WAIT_DTYPE)
                for i, (dg, mv, ip, imm, pre, wait_ms, ka) in enumerate(rows):
                    r[i] = (d.intern_env(dg), mv, d.intern_ip(ip), imm, pre, wait_ms, ka)
                per.append(r)
            results, grants = svc.wait_for_starting_tasks(toks, per[0], now=now)  # ONE batched solve
            for i in range(n_rpc):  # the model: RPC after RPC, decision after decision
                st, gl = model.wait_for_starting_task(toks[i], per[1][i], now=now)
                assert int(results[i]["status"]) == st, (step, i, rows[i], toks[i])
                mine = grants[int(results[i]["first_grant"]): int(results[i]["first_grant"]) + int(results[i]["n_grants"])]
                assert [(int(g["task_id"]), int(g["servant_index"])) for g in mine] == gl, (step, i, rows[i])
                granted.extend(t for t, _ in gl)
        elif op == "keep" and granted:
            ids = [int(x) for x in rng.choice(granted, size=min(len(granted), 4), replace=False)] + [10**9]
            tok, ms = str(rng.choice(["u1", "s1", "bad"])), int(rng.choice([1000, 30000, 30001]))
            sa, oka = svc.keep_task_alive(tok, ids, ms, now=now)
            sb, okb = model.keep_task_alive(tok, ids, ms, now=now)
            assert sa == sb and (sa != 0 or list(oka) == okb), (step, tok, ms)
        elif op == "free" and granted:
            ids = [int(x) for x in rng.choice(granted, size=min(len(granted), 5), replace=False)]
            tok = str(rng.choice(["u1", "u1", "bad"]))
            assert svc.free_task(tok, ids) == model.free_task(tok, ids)
        elif op == "config":
            tok = str(rng.choice(["u1", "u2", "s1", ""]))
            (sa, ta), (sb, rolls) = svc.get_config(tok, now=now), model.get_config(tok, now=now)
            assert sa == sb
            if sa == 0:
                check_window(rolls, middle=ta)
        elif op == "running":
            assert svc.get_running_tasks() == model.get_running_tasks()
        elif op == "tick":
            da.on_expiration_timer(now=now)
            db.on_expiration_timer(now=now)
        if step % 40 == 39:
            sa, sb = da.servant_state(), db.servant_state()
            assert sa.shape == sb.shape and (sa == sb).all()
    svc.close()


@pytest.mark.parametrize("kind", ["port", "ref"])
@pytest.mark.parametrize("seed", range(24))
def test_service_layer_against_independent_python_model(make_dispatcher, kind, seed):
    _service_fuzz(make_dispatcher, kind, kind, seed)


@pytest.mark.gpu
@pytest.mark.parametrize("seed", range(6))
def test_service_layer_over_cuda_against_python_model_over_checker(make_dispatcher, seed):
    """The C handlers over the CUDA backend (batched WaitForStartingTask -> one solve) against the Python model of the
    reference's handlers over the CPU checker (one decision per call)."""
    _service_fuzz(make_dispatcher, "cuda", "port", seed)
