#!/usr/bin/env python3
"""TEST INFRASTRUCTURE -- records what the differential tests compare against, from the UNMODIFIED reference, into
tests/golden/live_ticks.json.gz and tests/golden/template_fixtures.json.xz.

These tests used to run the reference live next to the product; recorded, they run wherever the suite runs:
* tests/test_reference_live_cpu.py: the reference's constructors on synthetic kube objects (KubePod.resources,
  create_kube_node capacity, count_pod sums) and one D = 8 / T = 8 tick (ReferenceTick.run);
* tests/test_host_layer_live_cpu.py: four ticks recorded with node assignments, used_capacity key sets and every
  node's get_node_state;
* tests/test_template_processing_cpu.py: the reference's ARM template fixtures (test/data) and what its
  template_processing functions return on them.
Each synthetic case stores a digest of the generator's arrays and of the kube objects the reference was given, so
that generator drift is caught instead of compared against stale answers.

    python oracle/make_golden_live.py        (needs the reference tree: $ACSFIT_REFERENCE_ROOT or oracle/_ref)
"""
import gzip
import hashlib
import importlib
import json
import lzma
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
sys.path.insert(0, os.path.dirname(HERE))

import make_golden_mid as mid  # noqa: E402
import ref_bench  # noqa: E402
import ref_shim  # noqa: E402
from kubernetes_acs_engine_autoscaler_b200 import synthetic as syn  # noqa: E402

GOLDEN = os.path.join(os.path.dirname(HERE), "tests", "golden")
CONSTRUCTOR_CASES = [{"P": 400, "N": 40, "D": 4, "T": 1, "seed": 77}, {"P": 400, "N": 40, "D": 8, "T": 8, "seed": 77}]
ORACLE_CASE = {"P": 700, "N": 90, "D": 8, "T": 8, "seed": 78, "over_provision": 1}
HOST_LAYER_CASES = [{"P": 1500, "N": 200, "D": 4, "T": 2, "seed": 901, "max_size": None},
                    {"P": 900, "N": 120, "D": 4, "T": 1, "seed": 902, "max_size": None},
                    {"P": 1200, "N": 150, "D": 4, "T": 2, "seed": 903, "max_size": 40},
                    {"P": 1200, "N": 160, "D": 8, "T": 8, "seed": 904, "max_size": None}]
TEMPLATE_FIXTURES = ["azuredeploy.original.json", "azuredeploy.expected_nic.json", "azuredeploy.expected_vm.json",
                     "azuredeploy.cluster.json"]


def kube_digest(c):
    return hashlib.sha256(json.dumps(syn.kube_objects(c), sort_keys=True).encode()).hexdigest()


def make(case):
    c = syn.make_cluster(case["P"], case["N"], case["D"], case["T"], seed=case["seed"],
                         **({"over_provision": case["over_provision"]} if "over_provision" in case else {}))
    return c, dict(case, digest=mid.digest(c), kube_digest=kube_digest(c))


def rows(objs, attr, names):
    """float64 rows of a KubeResource attribute, and each object's key set as a bit mask over `names`."""
    vals = np.array([[float(getattr(o, attr).raw.get(k, 0.0)) for k in names] for o in objs], dtype=np.float64)
    keys = []
    for o in objs:
        raw = getattr(o, attr).raw
        assert set(raw) <= set(names), sorted(raw)
        keys.append(sum(1 << i for i, k in enumerate(names) if k in raw))
    return vals.reshape(len(objs), len(names)), np.array(keys, dtype=np.uint8)


def ids(uids):
    return np.array([int(u.split("-")[1]) for u in uids], dtype=np.int32)


def constructors(case):
    c, rec = make(case)
    tick = ref_bench.ReferenceTick(c)
    names = c["dim_names"]
    pending = [p for p in tick.pods if p.status == "Pending"]
    req, req_keys = rows(pending, "resources", names)
    run, _ = rows(tick.running, "resources", names)
    cap, _ = rows(tick.nodes, "capacity", names)
    tick.occupancy()
    used, _ = rows(tick.nodes, "used_capacity", names)
    rec.update({"n_pending": len(pending), "n_running": len(tick.running), "req_bits": mid.pack(req.view(np.uint64)),
                "req_keys": mid.pack(req_keys), "run_bits": mid.pack(run.view(np.uint64)),
                "cap_bits": mid.pack(cap.view(np.uint64)), "used_bits": mid.pack(used.view(np.uint64))})
    return rec


def tick_record(res):
    return {"to_schedule": mid.pack(ids(res["to_schedule"])), "pending": mid.pack(ids(res["pending"])),
            "used_bits": mid.pack(res["used"].view(np.uint64)), "scale_pools": res["scale_calls"],
            "exception": res["exception"]}


def host_layer(case):
    c, rec = make(dict(case, over_provision=1))
    cap = int(case["max_size"] if case["max_size"] is not None else c["pool_max"][0])
    tick = ref_bench.ReferenceTick(c, max_size=cap)
    res = tick.run(record=True)
    _, keys = rows(tick.nodes, "used_capacity", c["dim_names"])
    rec.update(tick_record(res))
    rec.update({"node_names": [n.name for n in tick.nodes], "used_keys": mid.pack(keys),
                "states": mid.pack(np.array([mid.STATE_CODES[str(s)] for s in res["states"]], dtype=np.uint8))})
    return rec


def templates():
    """the fixtures verbatim, and the reference's template_processing results on them (the calls the test makes)."""
    data = os.path.join(ref_shim.REFERENCE_ROOT, "test", "data")
    fixtures = {}
    for name in TEMPLATE_FIXTURES:
        with open(os.path.join(data, name)) as f:
            fixtures[name] = json.load(f)
    ref_shim.load_reference()
    sys.path.insert(0, ref_shim.REFERENCE_ROOT)
    try:
        ref_tp = importlib.import_module("autoscaler.template_processing")
    finally:
        sys.path.remove(ref_shim.REFERENCE_ROOT)
    sys.path.insert(0, os.path.join(os.path.dirname(HERE), "tests"))
    import test_template_processing_cpu as t
    calls = t.differential_calls(fixtures["azuredeploy.cluster.json"])
    return {"fixtures": fixtures, "results": {key: getattr(ref_tp, fn)(*args()) for key, (fn, args) in calls.items()}}


def main():
    import oracle
    oracle.build()
    out = {"source": "unmodified reference via oracle/ref_bench.py",
           "constructors": [constructors(case) for case in CONSTRUCTOR_CASES]}
    c, rec = make(ORACLE_CASE)
    res = ref_bench.ReferenceTick(c).run()
    assert ref_bench.compare(c, res, ref_bench.dense_answer(oracle, c)) == []
    rec.update(tick_record(res))
    out["oracle_tick"] = rec
    out["host_layer"] = [host_layer(case) for case in HOST_LAYER_CASES]
    path = os.path.join(GOLDEN, "live_ticks.json.gz")
    with gzip.GzipFile(path, "wb", mtime=0) as f:
        f.write(json.dumps(out, sort_keys=True).encode())
    print(path, os.path.getsize(path), "bytes")
    path = os.path.join(GOLDEN, "template_fixtures.json.xz")
    with lzma.open(path, "wb", preset=9 | lzma.PRESET_EXTREME) as f:
        f.write(json.dumps(dict(templates(), source="unmodified reference, test/data and autoscaler/template_processing.py"),
                           sort_keys=True).encode())
    print(path, os.path.getsize(path), "bytes")


if __name__ == "__main__":
    main()
