"""Shared loader of tests/golden/live_ticks.json.gz (recorded from the unmodified reference by
oracle/make_golden_live.py): regenerates a case's snapshot from its make_cluster arguments, verifies the digests of
the generated arrays and of the kube objects the reference was given, and unpacks what the reference computed."""
import functools
import gzip
import hashlib
import json
import os

import numpy as np

from kubernetes_acs_engine_autoscaler_b200 import synthetic as syn
from make_golden_mid import STATE_CODES
from mid_golden import _unpack

PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "live_ticks.json.gz")
STATE_NAMES = {code: name for name, code in STATE_CODES.items()}  # the reference's state strings by code


@functools.lru_cache(maxsize=1)
def load():
    with gzip.open(PATH, "rb") as f:
        return json.loads(f.read().decode())


def find(section, **match):
    hits = [r for r in load()[section] if all(r[k] == v for k, v in match.items())]
    assert len(hits) == 1, (section, match)
    return hits[0]


def cluster_of(rec):
    kw = {"over_provision": rec["over_provision"]} if "over_provision" in rec else {}
    c = syn.make_cluster(rec["P"], rec["N"], rec["D"], rec["T"], seed=rec["seed"], **kw)
    h = hashlib.sha256()
    for k in ("req", "cap_type", "node_type", "row_ptr", "run_idx", "req_run", "flags_run", "node_flags", "node_age"):
        h.update(np.ascontiguousarray(c[k]).tobytes())
    assert h.hexdigest() == rec["digest"], "synthetic generator drifted: regenerate the recorded ticks"
    kube = hashlib.sha256(json.dumps(syn.kube_objects(c), sort_keys=True).encode()).hexdigest()
    assert kube == rec["kube_digest"], "kube objects of the snapshot drifted: regenerate the recorded ticks"
    return c


def f64(rec, key, shape):
    return _unpack(rec[key], np.uint64).view(np.float64).reshape(shape)


def key_sets(masks, names):
    return [{k for i, k in enumerate(names) if int(m) >> i & 1} for m in masks]


def tick_result(rec):
    """the recorded tick in the form of ref_bench.ReferenceTick.run()'s result."""
    return {"to_schedule": ["pend-%d" % i for i in _unpack(rec["to_schedule"], np.int32)],
            "pending": ["pend-%d" % i for i in _unpack(rec["pending"], np.int32)],
            "used": f64(rec, "used_bits", (rec["N"], rec["D"])), "scale_calls": rec["scale_pools"],
            "exception": rec["exception"]}
