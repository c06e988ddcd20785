"""ARM template unrolling (SURVEY.md section 8(f)3): the reference's own known-answer tests
(test/test_template_processing.py:34-89) and a differential run of every function on the reference's fixture
templates.  The fixtures and what the unmodified reference returned on them are recorded in
tests/golden/template_fixtures.json.xz (oracle/make_golden_live.py)."""
import copy
import json
import lzma
import os

import pytest

from kubernetes_acs_engine_autoscaler_b200 import template_processing as tp

HERE = os.path.dirname(os.path.abspath(__file__))
FIXTURES = os.path.join(HERE, "golden", "template_fixtures.json.xz")


class Node(object):
    def __init__(self, index):
        self.index = index
        self.unschedulable = False


class Pool(object):
    def __init__(self, name, indexes):
        self.name = name
        self.nodes = [Node(i) for i in indexes]

    @property
    def actual_capacity(self):
        return len(self.nodes)

    def has_node_with_index(self, index):
        return any(n.index == index for n in self.nodes)


def test_get_new_node_indexes_kat():
    """reference test/test_template_processing.py:58-89"""
    assert tp.get_new_nodes_indexes(Pool("agentpool1", [0]), 2) == [1]
    assert tp.get_new_nodes_indexes(Pool("agentpool1", [0, 2]), 3) == [1]
    assert tp.get_new_nodes_indexes(Pool("agentpool1", [0, 1, 2]), 3) == []
    assert tp.get_new_nodes_indexes(Pool("agentpool1", [4]), 5) == [0, 1, 2, 3]
    assert tp.get_new_nodes_indexes(Pool("agentpool1", [2]), 5) == [0, 1, 3, 4]
    assert tp.get_new_nodes_indexes(Pool("agentpool1", [0, 1]), 1) == []   # shrinking asks for nothing


def mini_template():
    def res(name, kind, deps=(), counted=True, body=None):
        r = {"name": name, "type": kind, "dependsOn": list(deps), "properties": body or {}}
        if counted:
            r["copy"] = {"count": "[variables('xCount')]", "name": "loop"}
        return r
    resources = [res("[variables('nsgName')]", "Microsoft.Network/networkSecurityGroups", counted=False),
                 res("[variables('virtualNetworkName')]", "Microsoft.Network/virtualNetworks",
                     ["[concat('Microsoft.Network/networkSecurityGroups/', variables('nsgName'))]", "other"], counted=False)]
    for p in ("a", "b"):
        resources += [
            res(tp._NIC.format(p=p), "Microsoft.Network/networkInterfaces", ["[variables('nsgID')]", "[variables('vnetID')]"]),
            res(tp._STORAGE.format(p=p), "Microsoft.Storage/storageAccounts"),
            res(tp._AVSET.format(p=p), "Microsoft.Compute/availabilitySets", counted=False),
            res(tp._VM.format(p=p), "Microsoft.Compute/virtualMachines",
                ["[concat('nic-', copyIndex(variables('%sOffset')))]" % p],
                body={"osProfile": {"computerName": "[concat(variables('%sVMNamePrefix'), copyIndex(variables('%sOffset')))]" % (p, p)}}),
            res(tp._EXT.format(p=p), "Microsoft.Compute/virtualMachines/extensions",
                ["[concat(variables('%sVMNamePrefix'), copyIndex(variables('%sOffset')))]" % (p, p)]),
        ]
    resources.append(res(tp._EXT.format(p="master"), "Microsoft.Compute/virtualMachines/extensions"))
    return {"resources": resources, "outputs": {"x": 1}, "variables": {}}


def test_scale_out_template_shape():
    t = mini_template()
    before = copy.deepcopy(t)
    out = tp.prepare_template_for_scale_out(t, [Pool("a", [0, 2]), Pool("b", [0])], {"a": 4, "b": 1})
    assert t == before                                   # the argument is not modified
    names = [r["name"] for r in out["resources"]]
    assert "outputs" not in out and "[variables('nsgName')]" not in names
    assert not any("variables('b" in n for n in names)   # the unchanged pool is gone entirely
    # pool a grows from {0, 2} to 4 nodes: indexes 1 and 3, highest first, extension / vm / nic groups
    assert names[:6] == ["[concat(variables('aVMNamePrefix'), 3,'/cse', 3)]", "[concat(variables('aVMNamePrefix'), 1,'/cse', 1)]",
                         "[concat(variables('aVMNamePrefix'), 3)]", "[concat(variables('aVMNamePrefix'), 1)]",
                         "[concat(variables('aVMNamePrefix'), 'nic-', 3)]", "[concat(variables('aVMNamePrefix'), 'nic-', 1)]"]
    vm3 = out["resources"][2]
    assert "copy" not in vm3 and vm3["dependsOn"] == ["[concat('nic-', 3)]"]
    assert vm3["properties"]["osProfile"]["computerName"] == "[concat(variables('aVMNamePrefix'), 3)]"
    nic = out["resources"][4]
    assert nic["dependsOn"] == ["[variables('vnetID')]"]  # NSG dependency dropped, copyIndex left alone in NICs
    vnet = [r for r in out["resources"] if r["type"] == "Microsoft.Network/virtualNetworks"][0]
    assert vnet["dependsOn"] == ["other"]
    with pytest.raises(ValueError, match="NIC resource"):
        tp.unroll_nic({"resources": []}, Pool("a", []), 1)
    assert len(tp.delete_master_vm_extension(mini_template())["resources"]) == len(mini_template()["resources"]) - 1


def differential_calls(cluster):
    """the calls compared with the reference on its cluster fixture: key -> (function name, fresh arguments)."""
    pool_names = sorted({r["name"].split("variables('")[1].split("VMNamePrefix")[0] for r in cluster["resources"]
                         if "VMNamePrefix'), copyIndex" in r["name"] and "master" not in r["name"]})
    assert pool_names
    calls = {}
    for k, (sizes, held) in enumerate([({n: 3 for n in pool_names}, [0]), ({n: 1 for n in pool_names}, [0]),
                                       ({n: (5 if i == 0 else 2) for i, n in enumerate(pool_names)}, [1, 3])]):
        calls["prepare_template_for_scale_out/%d" % k] = (
            "prepare_template_for_scale_out",
            lambda sizes=sizes, held=held: (copy.deepcopy(cluster), [Pool(n, held) for n in pool_names], dict(sizes)))
    for fn in ("unroll_vm_extension", "unroll_nic", "unroll_vm"):
        calls[fn] = (fn, lambda: (copy.deepcopy(cluster), Pool(pool_names[0], [0, 2]), 5))
    for fn in ("delete_master_vm_extension", "delete_nsg"):
        calls[fn] = (fn, lambda: (copy.deepcopy(cluster),))
    calls["delete_unchanged_pools"] = ("delete_unchanged_pools",
                                       lambda: (copy.deepcopy(cluster), [Pool(pool_names[0], [0])]))
    return calls


def test_every_function_equals_the_reference_on_its_fixtures():
    with lzma.open(FIXTURES, "rb") as f:
        golden = json.loads(f.read().decode())
    fixtures = golden["fixtures"]
    original = fixtures["azuredeploy.original.json"]
    pool = Pool("agentpool1", [0])
    # the reference's two fixture KATs (test/test_template_processing.py:34-56)
    assert tp.unroll_nic(copy.deepcopy(original), pool, 3) == fixtures["azuredeploy.expected_nic.json"]
    assert tp.unroll_vm(copy.deepcopy(original), pool, 3) == fixtures["azuredeploy.expected_vm.json"]
    calls = differential_calls(fixtures["azuredeploy.cluster.json"])
    assert sorted(calls) == sorted(golden["results"])
    for key, (fn, args) in calls.items():
        assert getattr(tp, fn)(*args()) == golden["results"][key], key
