"""Mechanical cross-check of the hand-transcribed fixtures (tests/golden/*.json) against the Go test sources they cite.

tests/golden/transcribe.py was written by hand.  tests/golden/extract_go_tables.py regex-parses the
table-driven Go tests of the reference and stores their cases in tests/golden/go_test_tables.json; these tests assert that the
literals in the hand-written fixtures equal the literals parsed out of the Go source, case by case and in order:
  Test_ShouldDeletePod                  raycluster_controller_unit_test.go:2380-2503
  TestCalculateMaxReplicasOverflow      utils/util_test.go:802-894
  TestInconsistentRayClusterStatus      utils/consistency_test.go:16-146
  TestShouldRecreatePodsForUpgrade      raycluster_controller_unit_test.go:3680-3814
  TestGetWorkerGroupDesiredReplicas     utils/util_test.go:555-601"""
import json
import os

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def gold(name):
    with open(os.path.join(GOLD, name + ".json")) as f:
        return json.load(f)


GO = gold("go_test_tables")


def test_should_delete_pod_table_matches_the_go_source():
    assert GO["should_delete_pod"] == gold("should_delete_pod")["cases"]


def test_max_replicas_overflow_table_matches_the_go_source():
    cases = GO["max_overflow"]
    want = gold("replica_arithmetic")["max_overflow"]["cases"]
    assert len(cases) == len(want)
    for c, w in zip(cases, want):
        assert c["expected"] == w["want_max"], w["name"]
        assert c["groups"] == [{k: v for k, v in g.items() if k in ("hosts", "replicas", "min", "max")} for g in w["groups"]], w["name"]


def test_desired_replicas_table_matches_the_go_source():
    """The Go test mutates one WorkerGroupSpec step by step and asserts after each step: at every assert the spec's state and
    the expected value must equal the fixture's case."""
    want = gold("replica_arithmetic")["desired_replicas"]["cases"]
    for seen, (state, w) in enumerate(zip(GO["desired_replicas"], want)):
        assert state["expected"] == w["want"], (seen, state, w)
        assert state["hosts"] == w["hosts"] and state["min"] == w["min"] and state["max"] == w["max"], (seen, state, w)
        assert state["replicas"] == w["replicas"] and state["suspend"] == w["suspend"], (seen, state, w)
    assert len(GO["desired_replicas"]) == len(want) == 6


def test_inconsistent_status_table_matches_the_go_source():
    go = GO["inconsistent_status"]
    g = gold("inconsistent_status")
    old = g["old"]
    for key in ("readyWorkerReplicas", "availableWorkerReplicas", "desiredWorkerReplicas", "minWorkerReplicas", "maxWorkerReplicas", "observedGeneration"):
        assert go["old"][key] == old[key], key
    assert go["old"]["head"]["podIP"] == old["head"]["podIP"]
    assert go["old"]["head"]["serviceIP"] == old["head"]["serviceIP"]
    assert go["old"]["reason"] == old["reason"]
    assert go["old"]["state"] == "ready" and old["state"] == "ready"
    assert len(go["cases"]) == len(g["cases"])
    for c, w in zip(go["cases"], g["cases"]):
        name = c["name"]
        assert name.startswith(w["name"].split(" ")[0].split(".")[0]) or w["name"].split(" ")[0] in name, (name, w["name"])
        assert c["want"] == w["want"], name


def test_recreate_upgrade_table_matches_the_go_source():
    cases = GO["recreate_upgrade"]
    want = gold("recreate_upgrade")["cases"]
    assert len(cases) == len(want)
    for c, w in zip(cases, want):
        assert c["want"] == w["want"], w["name"]
        assert c["upgradeStrategy"] == w["upgradeStrategy"], w["name"]
        assert (c["head"] is not None) == (w["head"] is not None), w["name"]
        if c["head"] is not None:
            assert c["head"]["hash_is_current"] == (w["head"]["hash"] == "<current>"), w["name"]
            assert c["head"]["version_is_current"] == (w["head"]["version"] == "<current>"), w["name"]
