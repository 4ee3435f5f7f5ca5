"""Shared fixtures.  Backends:

  port  oracle/libydoracle.so      CPU restatement (always buildable: g++ only)
  ref   oracle/_ref/libydref.so    reference sources compiled verbatim (built only
                                   where the reference sources are present)
  cuda  yadcc_b200/libydsched.so   the product; needs a B200 -> @pytest.mark.gpu

What a test's `ref` dispatchers return (every public method's result, in call order,
plus whatever the test hands to `reference.observe`) is digested and compared with
tests/golden/reference_results.json, which was recorded from the reference build.
Without that build, `ref` runs the CPU restatement under the same check, so every
comparison with the reference still runs.  To re-record, where the reference is
built:  YD_RECORD_REFERENCE=tests/golden/reference_results.json pytest tests
"""
import hashlib
import json
import os
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))

PORT_LIB = ROOT / "oracle" / "libydoracle.so"
REF_LIB = ROOT / "oracle" / "_ref" / "libydref.so"
CUDA_LIB = ROOT / "yadcc_b200" / "libydsched.so"
REF_RESULTS = ROOT / "tests" / "golden" / "reference_results.json"
RECORD_REF = os.environ.get("YD_RECORD_REFERENCE")
_recorded: dict = {}


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a real B200 (run with -m gpu on the GPU box)")


def _ensure_port():
    if not PORT_LIB.exists():
        subprocess.check_call(["make", "-C", str(ROOT / "oracle"), "libydoracle.so"])
    return PORT_LIB


def have_gpu() -> bool:
    if os.environ.get("YD_FORCE_NO_GPU"):
        return False
    try:
        import torch

        return torch.cuda.is_available()
    except Exception:
        return False


@pytest.fixture(scope="session")
def port_lib():
    return str(_ensure_port())


@pytest.fixture(scope="session")
def ref_lib():
    if not REF_LIB.exists():
        pytest.skip("oracle/_ref/libydref.so not built (needs the reference sources)")
    return str(REF_LIB)


@pytest.fixture(scope="session")
def cuda_lib():
    assert CUDA_LIB.exists(), "yadcc_b200/libydsched.so missing: run `make` / __graft_entry__.build()"
    return str(CUDA_LIB)


def cpu_backends():
    out = [pytest.param("port", id="port")]
    out.append(pytest.param("ref", id="ref"))
    return out


def _feed(h, v) -> None:
    """Canonical bytes of a result (arrays field by field, so struct padding never counts)."""
    if isinstance(v, np.ndarray):
        h.update(f"a{v.dtype.descr}{v.shape}".encode())
        for k in v.dtype.names or [None]:
            h.update(np.ascontiguousarray(v if k is None else v[k]).tobytes())
    elif isinstance(v, np.generic):
        _feed(h, v.item())
    elif isinstance(v, (bytes, bytearray)):
        h.update(b"b%d:" % len(v) + bytes(v))
    elif isinstance(v, dict):
        h.update(b"d%d" % len(v))
        for k in sorted(v, key=repr):
            _feed(h, k)
            _feed(h, v[k])
    elif isinstance(v, (list, tuple)):
        h.update(b"l%d" % len(v))
        for x in v:
            _feed(h, x)
    else:
        h.update(repr(v).encode() + b";")


class ReferenceResults:
    """Running SHA-256 over what the reference returned in one test."""

    def __init__(self):
        self.sha = hashlib.sha256()
        self.count = 0

    def observe(self, value, what: str = "value") -> None:
        self.sha.update(what.encode())
        _feed(self.sha, value)
        self.count += 1


class _Observed:
    """Forwards to a dispatcher and hands every public method's result to `results`."""

    UNOBSERVED = {"close", "alloc_requests", "alloc_grants", "alloc_requests16", "alloc_grants8", "last_solve_stats"}

    def __init__(self, d, results: ReferenceResults):
        self._d, self._results = d, results

    def __getattr__(self, name):
        attr = getattr(self._d, name)
        if name.startswith("_") or name in self.UNOBSERVED or not callable(attr):
            return attr

        def observed(*a, **kw):
            out = attr(*a, **kw)
            self._results.observe(out, name)
            return out

        return observed


@pytest.fixture
def reference(request):
    """This test's ReferenceResults; checked against the recorded ones when the test body returns."""
    request.node._reference_results = ReferenceResults()
    return request.node._reference_results


@pytest.hookimpl(wrapper=True)
def pytest_runtest_call(item):
    out = yield
    rec = getattr(item, "_reference_results", None)
    if rec is not None and rec.count:
        key = f"{item.path.name}::{item.name}"
        got = {"results": rec.count, "sha256": rec.sha.hexdigest()}
        if RECORD_REF:
            _recorded[key] = got
        else:
            want = json.loads(REF_RESULTS.read_text()).get(key) if REF_RESULTS.exists() else None
            assert want is not None, f"no recorded reference results for {key} in {REF_RESULTS.name}"
            assert got == want, (f"{key}: results differ from the reference's recorded ones "
                                 f"({'reference build' if REF_LIB.exists() else 'CPU restatement'} gave {got}, recorded {want})")
    return out


def pytest_sessionfinish(session):
    if RECORD_REF and _recorded:
        stored = json.loads(REF_RESULTS.read_text()) if REF_RESULTS.exists() else {}
        stored.update(_recorded)
        Path(RECORD_REF).write_text(json.dumps(dict(sorted(stored.items())), indent=1) + "\n")


@pytest.fixture
def make_dispatcher(request, reference):
    """Factory: make_dispatcher('port'|'ref'|'cuda', **kw) -> TaskDispatcher."""
    from yadcc_b200 import TaskDispatcher

    made = []

    def factory(kind: str, **kw):
        if kind == "port":
            lib = str(_ensure_port())
        elif kind == "ref":
            assert REF_LIB.exists() or not RECORD_REF, "recording reference results needs oracle/_ref/libydref.so"
            lib = str(REF_LIB) if REF_LIB.exists() else str(_ensure_port())
        elif kind == "cuda":
            assert CUDA_LIB.exists(), "yadcc_b200/libydsched.so missing"
            lib = str(CUDA_LIB)
        else:
            raise ValueError(kind)
        d = TaskDispatcher(lib, **kw)
        if kind == "ref":
            d = _Observed(d, reference)
        made.append(d)
        return d

    yield factory
    for d in made:
        d.close()
