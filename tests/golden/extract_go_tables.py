#!/usr/bin/env python
"""Extracts the case tables of five table-driven Go tests of the reference mechanically (regex parsing of the Go source) and
writes them to go_test_tables.json, which tests/test_golden_pin.py holds the hand-written fixtures of transcribe.py to:
  Test_ShouldDeletePod                  raycluster_controller_unit_test.go:2380-2503
  TestCalculateMaxReplicasOverflow      utils/util_test.go:802-894
  TestInconsistentRayClusterStatus      utils/consistency_test.go:16-146
  TestShouldRecreatePodsForUpgrade      raycluster_controller_unit_test.go:3680-3814
  TestGetWorkerGroupDesiredReplicas     utils/util_test.go:555-601

usage: extract_go_tables.py <kuberay checkout>      (the JSON is committed; rerun it when the reference moves)"""
import json
import os
import re
import sys

HERE = os.path.dirname(os.path.abspath(__file__))


def go_func(ref: str, path: str, name: str) -> str:
    src = open(os.path.join(ref, path)).read()
    start = src.index(f"func {name}(")
    nxt = src.find("\nfunc ", start + 1)
    return src[start:nxt if nxt > 0 else len(src)]


def table_cases(body: str) -> list[str]:
    """The `{ ... },` literals of the first table-driven slice in a Go test body (brace matching, comments stripped)."""
    body = re.sub(r"//[^\n]*", "", body)
    m = re.search(r":= \[\]struct \{.*?\n\t\}\{\n", body, re.S)
    assert m, "no table found"
    i, depth, cases, cur = m.end(), 0, [], None
    while i < len(body):
        ch = body[i]
        if ch == "{":
            if depth == 0:
                cur = i
            depth += 1
        elif ch == "}":
            depth -= 1
            if depth == 0:
                cases.append(body[cur:i + 1])
            if depth < 0:
                break
        i += 1
    return cases


def should_delete_pod(ref: str) -> list[dict]:
    out = []
    for c in table_cases(go_func(ref, "raycluster_controller_unit_test.go", "Test_ShouldDeletePod")):
        out.append({
            "restartPolicy": re.search(r"restartPolicy:\s*corev1\.RestartPolicy(\w+)", c).group(1),
            "phase": re.search(r"phase:\s*corev1\.Pod(\w+)", c).group(1),
            "terminated": "Terminated: &corev1.ContainerStateTerminated" in c,
            "want": re.search(r"shouldDelete:\s*(true|false)", c).group(1) == "true",
        })
    return out


def _groups(case: str) -> list[dict]:
    out = []
    for g in re.findall(r"\{[^{}]*?NumOfHosts[^{}]*?\}", case, re.S):
        d = {"hosts": int(re.search(r"NumOfHosts:\s*(\d+)", g).group(1))}
        for key, fld in (("replicas", "Replicas"), ("min", "MinReplicas"), ("max", "MaxReplicas")):
            m = re.search(rf"\b{fld}:\s*ptr\.To\[int32\]\((-?\d+)\)", g)
            if m:
                d[key] = int(m.group(1))
        out.append(d)
    return out


def max_overflow(ref: str) -> list[dict]:
    return [{"expected": int(re.search(r"expected:\s*(-?\d+)", c).group(1)), "groups": _groups(c)}
            for c in table_cases(go_func(ref, "utils/util_test.go", "TestCalculateMaxReplicasOverflow"))]


def desired_replicas(ref: str) -> list[dict]:
    """The Go test mutates one WorkerGroupSpec step by step (fields bound to local variables through pointers) and asserts after
    each step: replay the assignments and record, at every assert, the spec's state and the expected value."""
    body = re.sub(r"//[^\n]*", "", go_func(ref, "utils/util_test.go", "TestGetWorkerGroupDesiredReplicas"))
    var: dict[str, object] = {}
    bind: dict[str, tuple[str, bool]] = {}   # struct field -> (variable, bound by pointer)
    fields = {"NumOfHosts": "hosts", "MinReplicas": "min", "MaxReplicas": "max", "Replicas": "replicas", "Suspend": "suspend"}
    frozen: dict[str, object] = {}           # value fields copy at assignment time
    out = []
    for line in body.splitlines():
        line = line.strip().rstrip(",")
        m = re.fullmatch(r"(\w+)\s*:?=\s*int32\((-?\d+)\)", line)
        if m:
            var[m.group(1)] = int(m.group(2)); continue
        m = re.fullmatch(r"(\w+)\s*:?=\s*(true|false)", line)
        if m:
            var[m.group(1)] = m.group(2) == "true"; continue
        m = re.fullmatch(r"(?:workerGroupSpec\.)?(\w+)\s*[:=]\s*(&?)(\w+)", line)
        if m and m.group(1) in fields:
            if m.group(2):
                bind[m.group(1)] = (m.group(3), True); frozen.pop(m.group(1), None)
            else:
                bind.pop(m.group(1), None); frozen[m.group(1)] = var[m.group(3)]
            continue
        m = re.fullmatch(r"assert\.(Equal|Zero)\(t, GetWorkerGroupDesiredReplicas\(workerGroupSpec\)(?:, (.+))?\)", line)
        if m:
            state = {key: var[bind[f][0]] if f in bind else frozen.get(f) for f, key in fields.items()}
            state["suspend"] = bool(state["suspend"])
            state["expected"] = 0 if m.group(1) == "Zero" else eval(m.group(2), {}, dict(var))  # noqa: S307 - a product of two test locals at most
            out.append(state)
    return out


def inconsistent_status(ref: str) -> dict:
    body = go_func(ref, "utils/consistency_test.go", "TestInconsistentRayClusterStatus")
    lit = re.search(r"oldStatus := rayv1\.RayClusterStatus\{(.*?)\n\t\}\n", body, re.S).group(1)
    old = {key: int(re.search(rf"\b{go_name}:\s*(\d+)", lit).group(1))
           for go_name, key in (("ReadyWorkerReplicas", "readyWorkerReplicas"), ("AvailableWorkerReplicas", "availableWorkerReplicas"),
                                ("DesiredWorkerReplicas", "desiredWorkerReplicas"), ("MinWorkerReplicas", "minWorkerReplicas"),
                                ("MaxWorkerReplicas", "maxWorkerReplicas"), ("ObservedGeneration", "observedGeneration"))}
    old["head"] = {"podIP": re.search(r'PodIP:\s*"([^"]+)"', lit).group(1), "serviceIP": re.search(r'ServiceIP:\s*"([^"]+)"', lit).group(1)}
    old["reason"] = re.search(r'Reason:\s*"([^"]+)"', lit).group(1)
    old["state"] = "ready" if "State:                   rayv1.Ready" in lit else None
    cases = [{"name": re.search(r'name:\s*"([^"]+)"', c).group(1), "want": re.search(r"expectResult:\s*(true|false)", c).group(1) == "true"}
             for c in table_cases(body[body.index("testCases :="):])]
    return {"old": old, "cases": cases}


def recreate_upgrade(ref: str) -> list[dict]:
    out = []
    for c in table_cases(go_func(ref, "raycluster_controller_unit_test.go", "TestShouldRecreatePodsForUpgrade")):
        if "upgradeStrategy:  nil" in c or re.search(r"upgradeStrategy:\s*nil", c):
            strategy = None
        elif "Type: nil" in c:
            strategy = {"type": None}
        elif "RayClusterUpgradeNone" in c:
            strategy = {"type": "None"}
        else:
            assert "RayClusterRecreate" in c, c
            strategy = {"type": "Recreate"}
        d = {"want": re.search(r"expectedRecreate:\s*(true|false)", c).group(1) == "true", "upgradeStrategy": strategy,
             "head": None}
        m = re.search(r"createPodWithHash\(([^)]*)\)", c)
        if m:
            hash_arg, ver_arg = [a.strip() for a in m.group(1).split(",")][-2:]
            d["head"] = {"hash_is_current": hash_arg == "RayClusterHash", "version_is_current": ver_arg == "utils.KUBERAY_VERSION"}
        out.append(d)
    return out


def main(checkout: str):
    ref = os.path.join(checkout, "ray-operator", "controllers", "ray")
    doc = {"_source": "ray-operator/controllers/ray/ of ray-project/kuberay, parsed by extract_go_tables.py",
           "should_delete_pod": should_delete_pod(ref), "max_overflow": max_overflow(ref), "desired_replicas": desired_replicas(ref),
           "inconsistent_status": inconsistent_status(ref), "recreate_upgrade": recreate_upgrade(ref)}
    with open(os.path.join(HERE, "go_test_tables.json"), "w") as f:
        json.dump(doc, f, indent=1)
        f.write("\n")


if __name__ == "__main__":
    main(sys.argv[1])
