"""The oracle (C and Python restatements) against the reference's own golden vectors.

Vectors: tests/golden/go_filter_test_vectors.json, extracted from the reference's
pkg/ext-proc/scheduling/filter_test.go (TestFilter :12-215, TestFilterFunc :217-409) and
pkg/ext-proc/test/hermetic_test.go (:27-139) by tests/golden/extract_go_vectors.py.
"""
import hashlib
import os

from helpers import golden_to_py, pod_key
from oracle import lig_oracle_py as PY

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GO_FILTER_TEST_VECTORS_SHA256 = "76726ceef9370a712ec7e1c46ac74ea31668804514a670d731de786d140871e0"


def _func_of(case):
    """(which, q_thr, kv_thr) of a TestFilterFunc case's `f` field."""
    f = case["f"]
    if f["name"] == "toFilterFunc":
        inner = f["args"][0]
        if inner["name"] == "noQueueAndLessThanKVCacheThresholdPredicate":
            return inner["name"], inner["args"][0], inner["args"][1]
        return inner["name"], 0, 0.0
    return f["name"], 0, 0.0


def test_fixture_has_every_reference_case(golden):
    assert [c["name"] for c in golden["TestFilter"]] == [
        "simple filter without successor, failure", "default filter, critical request",
        "default filter, sheddable request, accepted", "default filter, sheddable request, dropped"]
    assert len(golden["TestFilterFunc"]) == 6
    assert len(golden["TestHandleRequestBody"]) == 1


def test_fixture_is_fresh():
    """The fixture is byte for byte what extract_go_vectors.py extracts from the reference at the
    commit BASELINE.md names; the digest was taken from that extraction."""
    path = os.path.join(ROOT, "tests", "golden", "go_filter_test_vectors.json")
    assert hashlib.sha256(open(path, "rb").read()).hexdigest() == GO_FILTER_TEST_VECTORS_SHA256


# ---- TestFilter (filter_test.go:12-215) -------------------------------------------------------
def test_c_oracle_TestFilter(golden, oracle):
    for case in golden["TestFilter"]:
        pool = oracle.Pool(case["input"])
        if case["filter"]["name"] == "$filter_literal":       # filter_test.go:21-27
            rc, idx = pool.filter_error_leaf()
            assert rc == oracle.LIGO_ERROR and idx == [] and case["err"] and case["output"] is None
            continue
        req = case["req"]
        rc, idx = pool.filter(req["resolved_target_model"], req["critical"])
        assert (rc in (oracle.LIGO_DROP, oracle.LIGO_ERROR)) == case["err"], case["name"]
        got = [pod_key(case["input"][i]) for i in idx]
        assert got == [pod_key(p) for p in case["output"]], case["name"]   # order-sensitive cmp.Diff


def test_py_oracle_TestFilter(golden):
    for case in golden["TestFilter"]:
        if case["filter"]["name"] == "$filter_literal":
            node = PY.Filter("", lambda req, pods: (None, PY.FilterError("filter error")))
            out, err = node.Filter(None, [])
            assert out is None and err is not None
            continue
        pods = [golden_to_py(p) for p in case["input"]]
        req = PY.LLMRequest(model=case["req"]["model"],
                            resolved_target_model=case["req"]["resolved_target_model"],
                            critical=case["req"]["critical"])
        out, err = PY.Tree().default_filter.Filter(req, pods)
        assert (err is not None) == case["err"], case["name"]
        assert [p.pod.name for p in (out or [])] == [p["name"] for p in case["output"]], case["name"]


# ---- TestFilterFunc (filter_test.go:217-409) --------------------------------------------------
def test_c_oracle_TestFilterFunc(golden, oracle):
    for case in golden["TestFilterFunc"]:
        which, q_thr, kv_thr = _func_of(case)
        pool = oracle.Pool(case["input"])
        model = case["req"]["resolved_target_model"] if case["req"] else None
        rc, idx = pool.filter_func(which, model, False, q_thr, kv_thr)
        assert (rc != 0) == case["err"], case["name"]
        got = [pod_key(case["input"][i]) for i in idx]
        assert got == [pod_key(p) for p in case["output"]], case["name"]


def test_py_oracle_TestFilterFunc(golden):
    tree = PY.Tree()
    for case in golden["TestFilterFunc"]:
        which, q_thr, kv_thr = _func_of(case)
        pods = [golden_to_py(p) for p in case["input"]]
        req = PY.LLMRequest(resolved_target_model=case["req"]["resolved_target_model"]) if case["req"] else None
        if which == "leastQueuingFilterFunc":
            out, err = PY.least_queuing_filter_func(req, pods)
        elif which == "leastKVCacheFilterFunc":
            out, err = PY.least_kv_cache_filter_func(req, pods)
        elif which == "noQueueAndLessThanKVCacheThresholdPredicate":
            out, err = PY.to_filter_func(
                PY.no_queue_and_less_than_kv_cache_threshold_predicate(q_thr, kv_thr))(req, pods)
        else:
            out, err = PY.to_filter_func(tree.predicates[which])(req, pods)
        assert (err is not None) == case["err"], case["name"]
        got = [pod_key(case["input"][pods.index(p)]) for p in (out or [])]
        assert got == [pod_key(p) for p in case["output"]], case["name"]


# ---- hermetic (test/hermetic_test.go:27-139) --------------------------------------------------
def test_oracles_hermetic_target_pod(golden, oracle):
    case = golden["TestHandleRequestBody"][0]
    model_obj = case["models"][case["request_model"]]
    # RandomWeightedDraw with a single target of weight 100 is deterministic (datastore.go:78-98)
    assert len(model_obj["target_models"]) == 1
    resolved = model_obj["target_models"][0]["name"]
    critical = False                       # no Criticality in the spec => IsCritical false (datastore.go:100-105)
    assert model_obj["criticality"] is None
    want_address = next(h["raw_value"] for h in case["want_headers"] if h["key"] == "target-pod")
    pool = oracle.Pool(case["pods"])
    for rand_key in range(8):              # singleton survivor set: every draw picks it
        rc, pod, n = pool.schedule(resolved, critical, 1234, rand_key)
        assert (rc, n) == (oracle.LIGO_OK, 1)
        assert case["pods"][pod]["address"] == want_address
    sched = PY.Scheduler(PY.StaticProvider([golden_to_py(p) for p in case["pods"]]))
    st, idx, n, _ = sched.Schedule(PY.LLMRequest(model=case["request_model"],
                                                 resolved_target_model=resolved, critical=critical))
    assert (st, n) == (PY.LIGO_OK, 1) and case["pods"][idx]["address"] == want_address
    # the body rewrite the handler performs around the path (request.go:62-70): Content-Length
    import json
    body = json.dumps({"max_tokens": 100, "model": resolved, "prompt": "hello", "temperature": 0},
                      separators=(",", ":"), sort_keys=True)
    assert body == case["want_body"]
    assert str(len(body)) == next(h["raw_value"] for h in case["want_headers"] if h["key"] == "Content-Length")
