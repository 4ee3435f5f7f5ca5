"""FlareStd wire front end on the CPU backends: frames encoded/decoded by the google.protobuf
runtime against the hand-written codec, handlers checked against direct calls, and the verbatim
reference dispatcher (`ref`) against the restatement (`port`) frame by frame."""
import pytest

pytest.importorskip("google.protobuf")

from wire_cases import run_wire_scenario


def test_wire_scenario_port_equals_reference(make_dispatcher, reference):
    a = run_wire_scenario(make_dispatcher, "ref")
    reference.observe(a)
    b = run_wire_scenario(make_dispatcher, "port")
    assert a == b


def test_wire_parser_survives_mutated_frames(make_dispatcher):
    """A network-facing parser must not crash or over-read on garbage: 6 000 mutated frames
    (bit flips, truncations, length-field corruption, random tails) only ever yield a verdict in
    {-1, 0, 1}; handled frames produce a well-formed response frame."""
    import struct

    import numpy as np

    import wire_protos as W
    from yadcc_b200.service import SchedulerService

    PB = W.PB
    svc = SchedulerService(make_dispatcher("port"), acceptable_user_tokens="usr", acceptable_servant_tokens="srv", token_seed=2)
    hb = PB["HeartbeatRequest"](token="srv", next_heartbeat_in_ms=1000, version=3, location="10.0.0.1:8335", num_processors=8,
                                capacity=4, servant_priority=2, total_memory_in_bytes=1 << 36, memory_available_in_bytes=1 << 35)
    hb.env_descs.add().compiler_digest = "d" * 64
    t = hb.running_tasks.add()
    t.servant_task_id, t.task_grant_id, t.servant_location, t.task_digest = 5, 6, "10.0.0.1:8335", "e" * 64
    wq = PB["WaitForStartingTaskRequest"](token="usr", immediate_reqs=2, prefetch_reqs=1, next_keep_alive_in_ms=1000, min_version=1)
    wq.env_desc.compiler_digest = "d" * 64
    ka = PB["KeepTaskAliveRequest"](token="usr", next_keep_alive_in_ms=1000)
    ka.task_grant_ids.extend(range(40))
    seeds = [W.request_frame("Heartbeat", hb, 1), W.request_frame("WaitForStartingTask", wq, 2),
             W.request_frame("KeepTaskAlive", ka, 3), W.request_frame("GetRunningTasks", None, 4, flags=4),
             W.request_frame("FreeTask", PB["FreeTaskRequest"](token="usr", task_grant_ids=[1, 2, 3]), 5)]
    rng = np.random.default_rng(0)
    batch, verdicts = [], {-1: 0, 0: 0, 1: 0}
    for it in range(6000):
        f = bytearray(seeds[it % len(seeds)])
        kind = it % 6
        if kind == 0:  # bit flips anywhere
            for _ in range(int(rng.integers(1, 6))):
                f[int(rng.integers(0, len(f)))] ^= 1 << int(rng.integers(0, 8))
        elif kind == 1:  # truncation
            f = f[: int(rng.integers(0, len(f)))]
        elif kind == 2:  # corrupt a header length
            struct.pack_into("<I", f, 4 * int(rng.integers(1, 4)), int(rng.integers(0, 1 << 32)))
        elif kind == 3:  # random bytes in the body
            lo = 16 + struct.unpack_from("<I", f, 4)[0]
            for k in range(lo, len(f)):
                if rng.random() < 0.2:
                    f[k] = int(rng.integers(0, 256))
        elif kind == 4:  # random bytes in the meta
            for k in range(16, min(len(f), 16 + struct.unpack_from("<I", f, 4)[0])):
                if rng.random() < 0.2:
                    f[k] = int(rng.integers(0, 256))
        else:  # junk appended
            f += bytes(rng.integers(0, 256, int(rng.integers(1, 40)), dtype=np.uint8))
        batch.append((bytes(f), "10.0.0.%d" % (it % 200)))
        if len(batch) == 64:
            for (verdict, consumed, status, frame), (data, _) in zip(svc.handle_frames(batch, now=1.0 + it * 1e-3), batch):
                assert verdict in (-1, 0, 1)
                verdicts[verdict] += 1
                if verdict == 1:
                    assert 16 <= consumed <= len(data)
                    magic, ms, bs, att = struct.unpack("<IIII", frame[:16])
                    assert magic == W.MAGIC and att == 0 and len(frame) == 16 + ms + bs
                    meta = PB["RpcMeta"]()
                    meta.ParseFromString(frame[16:16 + ms])
                    assert meta.response_meta.status == status
                else:
                    assert consumed == 0 and frame == b""
            batch = []
    assert min(verdicts.values()) > 100  # all three outcomes really occurred


def test_wire_request_counts_are_not_trusted(make_dispatcher, reference):
    """immediate_reqs / prefetch_reqs are uint32s off the wire.  A caller with a BAD token and
    immediate_reqs = 0xFFFFFFFF gets ACCESS_DENIED (scheduler_service_impl.cc:216-219) before
    anything is sized for it; a caller with a good token gets exactly what the reference's loop
    would hand out -- every free slot, then it stops at the first failure (:247-251)."""
    import wire_protos as W
    from yadcc_b200 import PRIORITY_USER, Servant
    from yadcc_b200.service import SchedulerService

    PB = W.PB
    results = []
    for kind in ("port", "ref"):
        d = make_dispatcher(kind)
        svc = SchedulerService(d, acceptable_user_tokens="usr", acceptable_servant_tokens="srv", token_seed=2)
        dg = "d" * 64
        for i in range(5):
            d.keep_servant_alive(Servant(f"10.0.0.{i}:8335", None, [dg], 8, 16, 0, 0, 64 << 30, 4, PRIORITY_USER), 10.0, now=0.0)
        bad = PB["WaitForStartingTaskRequest"](token="nope", immediate_reqs=0xFFFFFFFF, prefetch_reqs=0xFFFFFFFF,
                                               next_keep_alive_in_ms=1000, min_version=1)
        bad.env_desc.compiler_digest = dg
        st, _, body = svc.call(W.SERVICE + "WaitForStartingTask", bad.SerializeToString(), "172.16.0.1", now=1.0)
        assert st == 1003 and body == b""
        good = PB["WaitForStartingTaskRequest"](token="usr", immediate_reqs=0xFFFFFFFF, prefetch_reqs=0xFFFFFFF0,
                                                next_keep_alive_in_ms=1000, min_version=1)
        good.env_desc.compiler_digest = dg
        st, _, body = svc.call(W.SERVICE + "WaitForStartingTask", good.SerializeToString(), "172.16.0.1", now=1.0)
        resp = PB["WaitForStartingTaskResponse"]()
        resp.ParseFromString(body)
        assert st == 0 and len(resp.grants) == 20  # 5 servants x max_tasks 4
        results.append([(g.task_grant_id, g.servant_location) for g in resp.grants])
        # and the same two as frames in one batch
        frames = [(W.request_frame("WaitForStartingTask", bad, 7), "172.16.0.1"),
                  (W.request_frame("WaitForStartingTask", good, 8), "172.16.0.1")]
        out = svc.handle_frames(frames, now=1.5)
        assert [o[2] for o in out] == [1003, 1001]  # the pool is full now: NO_QUOTA for the good caller
        svc.close()
    reference.observe(results[1])
    assert results[0] == results[1]
