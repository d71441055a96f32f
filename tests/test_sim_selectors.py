"""oracle/sim_selectors.py against vectors produced by the reference simulator's own method bodies
(tests/golden/make_sim_selector_vectors.py).  CPU only; candidate index lists must match exactly,
order included, and the float64 ratios bit for bit."""
import hashlib
import json
import os

from oracle import sim_selectors as S

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PATH = os.path.join(ROOT, "tests", "golden", "sim_selector_vectors.json")
SIM_SELECTOR_VECTORS_SHA256 = "0370a020bbb83b9ab992c301b8c95d298c974761ab6c3fbb1dd64c8e2039e1e5"


def load_case(c):
    return [S.PodState(lora_loaded=set(p["lora_loaded"]), max_num_tokens_allowed=p["max_num_tokens_allowed"],
                       decode=[S.Item(*x) for x in p["decode"]], prefill=[S.Item(*x) for x in p["prefill"]],
                       recompute=[S.Item(*x) for x in p["recompute"]]) for p in c["pods"]]


def test_restatement_matches_the_reference_method_bodies():
    data = json.load(open(PATH))
    assert data["loras"] == list(S.LORA_DICT) and len(data["cases"]) == 200
    n_multi = 0
    for c in data["cases"]:
        pods = load_case(c)
        assert [S.pending_tokens_perc(p) for p in pods] == c["pending_perc"]           # same float64 division
        assert [S.expected_kv_after_prefill(p) for p in pods] == c["expected_kv"]
        for lora, want in c["lora_affinity"].items():
            aff = S.lora_affinity(pods, lora)
            assert aff == want
            sub = [pods[i] for i in aff]
            for safe in (False, True):
                w = c["min_pending"][f"{lora}|{int(safe)}"]
                cand = S.min_pending_candidates(sub, safe)
                assert cand == w["candidates"]
                if cand:      # the quirk: the drawn index addresses the FULL actor list
                    assert S.resolve_quirk(cand[0]) == w["returned_actor"]
                else:
                    assert w["returned_actor"] is None
                n_multi += len(cand) > 1
            w = c["min_kv"][lora]
            cand = S.min_kv_candidates(sub)
            assert cand == w["candidates"] and (S.resolve_quirk(cand[0]) == w["returned_actor"] if cand else True)
            n_multi += len(cand) > 1
    assert n_multi > 100          # ties (the part random.choice then decides) are exercised


def test_c1_shape_is_covered():
    """BASELINE.json configs[0]: 8 pods, the 4 LoRA adapters of constants.py:21."""
    data = json.load(open(PATH))
    assert sum(len(c["pods"]) == 8 for c in data["cases"]) >= 150
    assert set(data["loras"]) == {"tweet", "sql", "dummy-1", "dummy-2"}


def test_fixture_is_fresh():
    """The fixture is byte for byte what make_sim_selector_vectors.py wrote from the reference source
    at the commit BASELINE.md names; the digest was taken from that run."""
    assert hashlib.sha256(open(PATH, "rb").read()).hexdigest() == SIM_SELECTOR_VECTORS_SHA256
