"""`-m "not gpu"`: the HOST LAYER of this package (Cluster.loop_logic: object construction incl. the C helper,
flattening, hand-off, write-back of `used_capacity`, maintain) on mid-size synthetic clusters against the unmodified
reference run on the same kube-style objects, as recorded in tests/golden/live_ticks.json.gz
(oracle/make_golden_live.py).  The device work is done by the plain-C oracle here (tests/oracle_engine.py); the CUDA
engine behind the same layer is checked by the GPU suite."""
import logging
import os
import re
import sys

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(os.path.dirname(HERE), "oracle"))
import live_golden  # noqa: E402


class Raw(object):
    __slots__ = ("obj",)

    def __init__(self, o):
        self.obj = o

    @property
    def name(self):
        return self.obj["metadata"]["name"]


class Lines(logging.Handler):
    def __init__(self):
        logging.Handler.__init__(self)
        self.lines = []

    def emit(self, record):
        self.lines.append(record.getMessage())


@pytest.mark.parametrize("P,N,D,T,seed,max_size", [(1500, 200, 4, 2, 901, None), (900, 120, 4, 1, 902, None),
                                                     (1200, 150, 4, 2, 903, 40), (1200, 160, 8, 8, 904, None)])
def test_loop_logic_equals_the_live_reference(oracle_mod, tmp_path, monkeypatch, P, N, D, T, seed, max_size):
    import ref_bench
    from oracle_engine import OracleEngine
    from kubernetes_acs_engine_autoscaler_b200 import agent_pool, capacity, engine_scaler, snapshot, utils
    from kubernetes_acs_engine_autoscaler_b200 import synthetic as syn
    from kubernetes_acs_engine_autoscaler_b200.cluster import Cluster

    rec = live_golden.find("host_layer", P=P, N=N, D=D, T=T, seed=seed, max_size=max_size)
    c = live_golden.cluster_of(rec)
    assert c["over_provision"] == 1
    cap = int(max_size if max_size is not None else c["pool_max"][0])

    # ---- the reference, as recorded on the same objects ------------------------------------------
    ref = live_golden.tick_result(rec)
    ref_names = rec["node_names"]
    ref_keys = live_golden.key_sets(live_golden._unpack(rec["used_keys"], np.uint8), c["dim_names"])
    ref_state = {name: live_golden.STATE_NAMES[int(s)]
                 for name, s in zip(ref_names, live_golden._unpack(rec["states"], np.uint8))}

    # ---- this package's host layer on the same objects -----------------------------------------
    st = syn.kube_objects(c)
    nodes, pods = [Raw(o) for o in st["nodes"]], [Raw(o) for o in st["pods"]]
    cl = Cluster(None, 1800, 1, "a", "b", "c", "d", "e", "f", 600, "rg", None, "", over_provision=c["over_provision"], dry_run=True)
    cl.list_nodes, cl.list_pods = (lambda: nodes), (lambda: pods)
    cl.arm_template, cl.arm_parameters = {}, st["arm_parameters"]
    kube_nodes = []
    orig_create = cl.create_kube_node

    def create(node):
        kn = orig_create(node)
        kube_nodes.append(kn)
        return kn
    cl.create_kube_node = create
    orig_init = agent_pool.AgentPool.__init__

    def pool_init(self, *a, **k):
        orig_init(self, *a, **k)
        self.max_size = cap
    monkeypatch.setattr(agent_pool.AgentPool, "__init__", pool_init)
    scale_calls = []
    monkeypatch.setattr(engine_scaler.EngineScaler, "scale_pools", lambda self, sizes: scale_calls.append(dict(sizes)))
    monkeypatch.setattr(utils, "now", lambda tz=None: syn.NOW if tz is None else syn.NOW.astimezone(tz))
    prev = snapshot._engine
    snapshot.set_engine(OracleEngine())
    capacity.load(ref_bench.capacity_file(c, str(tmp_path)))  # the table the reference was given (D = 8: generated)
    handler = Lines()
    log = logging.getLogger("autoscaler")
    log.addHandler(handler)
    old_level = log.level
    log.setLevel(logging.INFO)
    exc = None
    try:
        try:
            cl.loop_logic()
        except Exception as e:  # the raise path of fulfill_pending (scaler.py:179-181) leaves loop_logic, as upstream
            exc = [type(e).__name__, str(e)]
    finally:
        log.removeHandler(handler)
        log.setLevel(old_level)
        snapshot._engine = prev
        capacity.load()

    # ---- compare ---------------------------------------------------------------------------------
    assert (exc is None) == (ref["exception"] is None)
    if exc is not None:
        assert exc[0] == ref["exception"][0]
    assert scale_calls == ref["scale_calls"]
    names = c["dim_names"]
    assert [n.name for n in kube_nodes] == ref_names
    used = np.array([[float(n.used_capacity.raw.get(k, 0.0)) for k in names] for n in kube_nodes], dtype=np.float64)
    assert np.array_equal(used.view(np.uint64), ref["used"].view(np.uint64))
    assert [set(n.used_capacity.raw) for n in kube_nodes] == ref_keys      # KubeResource.__add__ unions the key sets
    text = "\n".join(handler.lines)
    assert "Pods to schedule: %d" % len(ref["to_schedule"]) in text
    assert "Pending pods: %d" % len(ref["pending"]) in text
    if exc is None:  # maintain ran: one state line per node of a scalable pool, the reference's state strings
        got_state = {}
        for line in handler.lines:
            m = re.match(r"node: (.*\S)\s+state: (\S+)$", line)
            if m:
                got_state[re.search(r"(k8s-[a-z0-9]+-\d+-\d+)", m.group(1)).group(1)] = m.group(2)
        assert len(got_state) == len(kube_nodes)
        assert got_state == ref_state
