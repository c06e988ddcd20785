"""`-m "not gpu"`: the reference's own constructors give the synthetic dense rows back bit for bit (SURVEY.md
section 7), and the C oracle equals the reference on a mid-size tick.  What the unmodified reference computed on the
same kube objects is recorded in tests/golden/live_ticks.json.gz (oracle/make_golden_live.py)."""
import os
import sys

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(os.path.dirname(HERE), "oracle"))
import live_golden  # noqa: E402


@pytest.mark.parametrize("D,T", [(4, 1), (8, 8)])
def test_synthetic_rows_equal_reference_constructors(D, T):
    from kubernetes_acs_engine_autoscaler_b200 import synthetic as syn
    rec = live_golden.find("constructors", P=400, N=40, D=D, T=T, seed=77)
    c = live_golden.cluster_of(rec)
    names, P, N = c["dim_names"], c["P"], c["N"]
    R = c["req_run"].shape[0]
    assert rec["n_pending"] == P and rec["n_running"] == R
    # KubePod.resources (kube.py:41-49) == the dense request row; its keys: what the requests name, plus pods = 1
    np.testing.assert_array_equal(live_golden.f64(rec, "req_bits", (P, D)).view(np.uint64), c["req"].view(np.uint64))
    keys = live_golden.key_sets(live_golden._unpack(rec["req_keys"], np.uint8), names)
    assert keys == [set(syn.requests_of(row, names)) | {"pods"} for row in c["req"]]
    np.testing.assert_array_equal(live_golden.f64(rec, "run_bits", (R, D)).view(np.uint64),
                                  c["req_run"][c["run_idx"]].view(np.uint64))
    # create_kube_node capacity (cluster.py:130-133) == cap_type row
    np.testing.assert_array_equal(live_golden.f64(rec, "cap_bits", (N, D)).view(np.uint64),
                                  c["cap_type"][c["node_type"]].view(np.uint64))
    # count_pod sums (cluster.py:165-168) == initial_used
    np.testing.assert_array_equal(live_golden.f64(rec, "used_bits", (N, D)).view(np.uint64),
                                  syn.initial_used(c).view(np.uint64))


def test_oracle_equals_live_reference(oracle_mod):
    import ref_bench
    rec = live_golden.load()["oracle_tick"]
    c = live_golden.cluster_of(rec)
    assert (c["P"], c["N"], c["D"], c["T"], c["over_provision"]) == (700, 90, 8, 8, 1)
    assert ref_bench.compare(c, live_golden.tick_result(rec), ref_bench.dense_answer(oracle_mod, c)) == []
