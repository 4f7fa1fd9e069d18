"""Unit tests for the node agent's pure logic: config defaulting, XID_CONFIG, MPS env maths, NUMA topology, sharing
validation, MIG table. Table-test shape follows the reference (pkg/gpu/nvidia/manager_test.go:30-310,
gpusharing/gpusharing_test.go:24-119)."""
import json

import os

import pytest

from container_engine_accelerators_b200.agent import config as cfgmod
from container_engine_accelerators_b200.agent import manager as mgr
from container_engine_accelerators_b200.agent import mig, nvml, protos, sharing, testing, util, version_visibility
from container_engine_accelerators_b200.agent.config import GPUConfig, GPUSharingConfig


@pytest.mark.parametrize("raw,want,err", [
    ({}, ("", 0), None),
    ({"MaxTimeSharedClientsPerGPU": 10}, ("time-sharing", 10), None),
    ({"MaxTimeSharedClientsPerGPU": 4, "GPUSharingConfig": {"GPUSharingStrategy": "mps", "MaxSharedClientsPerGPU": 2}}, ("time-sharing", 4), None),
    ({"GPUSharingConfig": {"GPUSharingStrategy": "mps", "MaxSharedClientsPerGPU": 8}}, ("mps", 8), None),
    ({"GPUSharingConfig": {"GPUSharingStrategy": "time-sharing"}}, None, "MaxSharedClientsPerGPU should be > 0"),
    ({"GPUSharingConfig": {"MaxSharedClientsPerGPU": 3}}, None, "GPU sharing strategy needs to be specified"),
    ({"GPUSharingConfig": {"GPUSharingStrategy": "bogus", "MaxSharedClientsPerGPU": 3}}, None, "invalid GPU Sharing strategy"),
])
def test_add_defaults_and_validate(raw, want, err):
    cfg = GPUConfig.from_json(json.dumps(raw))
    if err:
        with pytest.raises(cfgmod.ConfigError, match=err):
            cfg.add_defaults_and_validate()
    else:
        cfg.add_defaults_and_validate()
        assert (cfg.sharing.strategy, cfg.sharing.max_shared_clients_per_gpu) == want


def test_parse_gpu_config_falls_back_to_empty_on_garbage(tmp_path):
    p = tmp_path / "gpu_config.json"
    p.write_text("{not json")
    assert cfgmod.parse_gpu_config(str(p)) == GPUConfig()
    p.write_text(json.dumps({"GPUSharingConfig": {"GPUSharingStrategy": "bogus", "MaxSharedClientsPerGPU": 1}}))
    assert cfgmod.parse_gpu_config(str(p)) == GPUConfig()
    p.write_text(json.dumps({"GPUPartitionSize": "1g.23gb", "Transport": "b200coll"}))
    cfg = cfgmod.parse_gpu_config(str(p))
    assert cfg.gpu_partition_size == "1g.23gb" and cfg.transport.name == "b200coll"
    assert cfgmod.parse_gpu_config(str(tmp_path / "missing.json")) == GPUConfig()


@pytest.mark.parametrize("env,want,err", [("", [], None), ("61", [61], None), ("61, 74 ,79", [61, 74, 79], None), ("61,abc", None, "Invalid HealthCriticalXid input")])
def test_xid_config(env, want, err):
    cfg = GPUConfig()
    if err:
        with pytest.raises(cfgmod.ConfigError, match=err):
            cfg.add_health_critical_xid({"XID_CONFIG": env})
    else:
        cfg.add_health_critical_xid({"XID_CONFIG": env})
        assert cfg.health_critical_xid == want


@pytest.mark.parametrize("max_clients,total_gb,requested,thread,mem", [(10, 80, 1, "10", "0=8192M"), (2, 80, 1, "50", "0=40960M"), (4, 180, 2, "50", "0=92160M")])
def test_mps_envs(tmp_path, max_clients, total_gb, requested, thread, mem):
    # expected strings: reference manager_test.go:188-207
    cfg = GPUConfig(sharing=GPUSharingConfig(sharing.MPS, max_clients))
    ngm = mgr.GPUManager(str(tmp_path), str(tmp_path), [], cfg, nvml=nvml.MockNvml(str(tmp_path)))
    ngm.total_mem_per_gpu = total_gb << 30
    assert ngm.envs(requested) == {"CUDA_MPS_ACTIVE_THREAD_PERCENTAGE": thread, "CUDA_MPS_PINNED_DEVICE_MEM_LIMIT": mem}
    assert mgr.GPUManager(str(tmp_path), str(tmp_path), [], GPUConfig(), nvml=nvml.MockNvml(str(tmp_path))).envs(1) == {}


def test_mps_start_requires_control_daemon(tmp_path):
    dev = testing.make_fake_dev(str(tmp_path), 1)
    cfg = GPUConfig(sharing=GPUSharingConfig(sharing.MPS, 4)); cfg.add_defaults_and_validate()
    ok = tmp_path / "mps-ok"; ok.write_text("#!/bin/sh\ncat >/dev/null\necho 100.0\n"); ok.chmod(0o755)
    ngm = mgr.GPUManager(dev, str(tmp_path / "proc"), [], cfg, nvml=nvml.MockNvml(dev, mem_total=180 << 30), mps_control_bin=str(ok))
    ngm.start()
    assert ngm.total_mem_per_gpu == 180 << 30 and any(m.host_path == "/tmp/nvidia-mps" and not m.read_only for m in ngm.mount_paths)
    bad = mgr.GPUManager(dev, str(tmp_path / "proc"), [], cfg, nvml=nvml.MockNvml(dev), mps_control_bin=str(tmp_path / "absent"))
    with pytest.raises(RuntimeError, match="NVIDIA MPS is not running on this node"):
        bad.start()


@pytest.mark.parametrize("bus,sysfs_name,node,want", [("00000000:1B:00.0", "0000:1b:00.0", 1, 1), ("00000000:1B:00.0", "0000:1b:00.0", -1, None), ("0000:AF:00.0", "0000:af:00.0", 0, 0)])
def test_numa_topology(tmp_path, bus, sysfs_name, node, want):
    root = testing.make_fake_pci(str(tmp_path), sysfs_name, node)
    assert nvml.numa_topology(bus, root) == want


def test_numa_topology_missing_file_raises(tmp_path):
    with pytest.raises(nvml.NvmlError, match="failed to read NUMA information"):
        nvml.numa_topology("00000000:1B:00.0", str(tmp_path))


def test_discovery_sets_topology(tmp_path):
    dev = testing.make_fake_dev(str(tmp_path), 2)
    pci = testing.make_fake_pci(str(tmp_path), "0000:1b:00.0", 1)
    ngm = mgr.GPUManager(dev, str(tmp_path / "proc"), [], GPUConfig(), nvml=nvml.MockNvml(dev, bus_id="00000000:1B:00.0"), pci_root=pci)
    ngm.start()
    assert {k: v.numa_node for k, v in ngm.list_devices().items()} == {"nvidia0": 1, "nvidia1": 1}
    assert len(ngm.default_devices) == 4


@pytest.mark.parametrize("ids,count,strategy,err", [
    (["nvidia0/vgpu0"], 1, sharing.TIME_SHARING, None),
    (["nvidia0/vgpu0", "nvidia0/vgpu1"], 1, sharing.TIME_SHARING, sharing.ERR_TIME_SHARING),
    (["nvidia0/vgpu0", "nvidia0/vgpu1"], 1, sharing.MPS, None),
    (["nvidia0/vgpu0", "nvidia1/vgpu0"], 2, sharing.MPS, sharing.ERR_MPS),
    (["nvidia0/gi0/vgpu0", "nvidia0/gi1/vgpu0"], 2, sharing.MPS, sharing.ERR_MPS),
    (["nvidia0", "nvidia1"], 2, sharing.TIME_SHARING, None),
])
def test_validate_request(ids, count, strategy, err):
    if err:
        with pytest.raises(sharing.SharingError) as ei:
            sharing.validate_request(ids, count, strategy)
        assert str(ei.value) == err
    else:
        sharing.validate_request(ids, count, strategy)


@pytest.mark.parametrize("vid,want", [("nvidia0/vgpu0", "nvidia0"), ("nvidia12/vgpu3", "nvidia12"), ("nvidia0/gi3/vgpu1", "nvidia0/gi3"), ("nvidia0", None), ("vgpu0", None)])
def test_virtual_to_physical(vid, want):
    if want is None:
        with pytest.raises(sharing.SharingError, match="is not valid"):
            sharing.virtual_to_physical_device_id(vid)
    else:
        assert sharing.virtual_to_physical_device_id(vid) == want


def test_mig_table_b200_rows():
    # reference: partition_gpu/partition_gpu.go:61-68,113-120; mig.go:56-63
    want = {"1g.23gb": (19, 7), "1g.45gb": (15, 4), "2g.45gb": (14, 3), "3g.90gb": (9, 2), "4g.90gb": (5, 1), "7g.180gb": (0, 1)}
    for size, (pid, cnt) in want.items():
        p = mig.PROFILES[size]
        assert (p.profile_id, p.max_count) == (pid, cnt) and "b200" in p.families
    assert "4g.40gb" in mig.PROFILES          # the plugin table now has the 4g sizes the reference's lacked


def test_mig_bad_size(tmp_path):
    m = mig.MigDeviceManager(str(tmp_path), str(tmp_path))
    with pytest.raises(mig.MigError, match="9g.999gb is not a valid GPU partition size"):
        m.start("9g.999gb")


def test_mig_unpartitioned_gpu_detected(tmp_path):
    dev = testing.make_fake_dev(str(tmp_path), 2)
    proc = testing.make_fake_mig(str(tmp_path), dev, 1, 7)
    m = mig.MigDeviceManager(dev, proc)
    with pytest.raises(mig.MigError, match="Not all GPUs are partitioned as expected. Total number of GPUs: 2, number of partitioned GPUs: 1"):
        m.start("1g.23gb")


def test_device_name_from_path():
    assert util.device_name_from_path("/dev/nvidia3") == "nvidia3"
    with pytest.raises(ValueError):
        util.device_name_from_path("/dev/nvidiactl")


def test_driver_version_annotations_preserve_others():
    from container_engine_accelerators_b200.agent import kube
    api = testing.FakeKubeApi().start()
    try:
        api.add_node("n1", annotations={"keep": "me"})
        ann = version_visibility.publish_driver_version_annotations(kube.KubeClient(api.url), "n1", "580.159.03")
        assert ann[version_visibility.MAJOR] == "580" and ann[version_visibility.MINOR] == "159" and ann[version_visibility.REVISION] == "03"
        got = api.nodes["n1"]["metadata"]["annotations"]
        assert got["keep"] == "me" and got[version_visibility.FULL] == "580.159.03"
        method, path, ctype = api.requests[-1]
        assert method == "PATCH" and "apply-patch" in ctype
        with pytest.raises(ValueError):
            version_visibility.parse_driver_annotations("not.a.version.x")
    finally:
        api.stop()


# ------------------------------------------------------------------------------------------------- wire schemas vs upstream .proto files
# What the upstream sources say is stored in tests/golden/reference_facts.json (oracle/reference_facts.py regenerates it), so these
# comparisons run everywhere, not only next to an upstream checkout.
def _reference_facts(section):
    with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_facts.json")) as f:
        return json.load(f)[section]


_SCALARS = {9: "string", 8: "bool", 3: "int64", 5: "int32", 13: "uint32", 4: "uint64", 12: "bytes", 1: "double", 2: "float"}


def _our_fields(msg_cls):
    fields = {}
    for f in msg_cls.DESCRIPTOR.fields:
        if f.message_type is not None and f.message_type.GetOptions().map_entry:
            k, v = f.message_type.fields_by_name["key"], f.message_type.fields_by_name["value"]
            vt = v.message_type.name if v.message_type is not None else _SCALARS[v.type]
            fields[f.name] = (f.number, f"map<{_SCALARS[k.type]},{vt}>", False)
        else:
            typ = f.message_type.name if f.message_type is not None else (f.enum_type.name if f.enum_type is not None else _SCALARS[f.type])
            fields[f.name] = (f.number, typ, bool(f.is_repeated) if hasattr(f, "is_repeated") else f.label == f.LABEL_REPEATED)
    return fields


@pytest.mark.parametrize("ours,upstream", [
    ("deviceplugin", "k8s.io/kubelet/pkg/apis/deviceplugin/v1beta1/api.proto"),
    ("podresources", "k8s.io/kubelet/pkg/apis/podresources/v1alpha1/api.proto"),
    ("nri", "github.com/containerd/nri/pkg/api/api.proto"),
])
def test_kubelet_schemas_match_the_upstream_proto_files(ours, upstream):
    """protos.py builds descriptors at run time from a hand-written table (the image has no protoc); every message and field in that
    table must agree — name, number, type, repeated — with the schema the kubelet is compiled from. Fields we do not model are fine
    (proto3 skips unknown fields); a wrong number or type is not."""
    assert _reference_facts("proto_sources")[ours].endswith(upstream)
    theirs = {name: {f: tuple(spec) for f, spec in fields.items()} if name != "__enums__" else set(fields)
              for name, fields in _reference_facts("proto_schemas")[ours].items()}
    ns = getattr(protos, ours)
    checked = 0
    for name, cls in vars(ns).items():
        if not hasattr(cls, "DESCRIPTOR"):
            continue
        assert name in theirs, f"{name} is not a message of {upstream}"
        for fname, spec in _our_fields(cls).items():
            assert fname in theirs[name], f"{name}.{fname} does not exist upstream (has {sorted(theirs[name])})"
            up = theirs[name][fname]
            if up[1] in theirs.get("__enums__", ()) and spec[1] == "int32":
                up = (up[0], "int32", up[2])                  # an enum travels as an int32 varint: modelling it as int32 is wire-exact
            assert up == spec, f"{name}.{fname}: ours {spec}, upstream {theirs[name][fname]}"
            checked += 1
    assert checked >= {"deviceplugin": 30, "podresources": 6, "nri": 15}[ours]


def test_contract_constants_match_the_reference_sources():
    """Names that other systems key on (Prometheus queries, node-problem-detector, the kubelet, job templates) must be the reference's
    exactly, in the Python agent AND in the native binary: monitored Xids, gauge names, annotation keys, condition / event strings,
    resource name, topology labels, NRI annotation prefix."""
    from container_engine_accelerators_b200.agent import health, metrics, nri as nrimod
    from container_engine_accelerators_b200.scheduler import topology as topo
    ref = _reference_facts("contract_constants")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    native = open(os.path.join(root, "agent", "native", "dp", "device_plugin.cc")).read()
    xids = tuple(ref["monitor_xids"])
    assert health.MONITOR_XIDS == xids and "kMonitorXids[] = {" + ", ".join(map(str, xids)) + "}" in native
    assert ref["xid_condition_type"] == "XidCriticalError"
    assert health.XID_CONDITION_TYPE == "XidCriticalError" and 'kXidCondition = "XidCriticalError"' in native
    assert ref["event_source"] == "nvidia-gpu-device-plugin" and health.EVENT_SOURCE == "nvidia-gpu-device-plugin" and 'kEventSource = "nvidia-gpu-device-plugin"' in native
    gauges = ref["gauges"]
    assert sorted(gauges) == sorted(["duty_cycle_gpu_node", "memory_total_gpu_node", "memory_used_gpu_node", "duty_cycle", "memory_total", "memory_used", "request"])
    ours = {m._name for m in metrics.MetricServer(nvml.MockNvml("/nonexistent"))._all}
    assert set(gauges) <= ours
    for g in gauges:
        assert f'"{g}"' in native or f'"{g.replace("_gpu_node", "")}"' in native, g
    prefix = ref["driver_version_prefix"]
    assert version_visibility.PREFIX == prefix + "." and f'"{prefix}."' in native
    assert ref["field_manager"] == "gpu-device-plugin"
    assert version_visibility.FIELD_MANAGER == "gpu-device-plugin" and '"gpu-device-plugin"' in native
    assert ref["resource_name"] == "nvidia.com/gpu"
    assert mgr.RESOURCE_NAME == "nvidia.com/gpu" and 'kResourceName = "nvidia.com/gpu"' in native
    assert topo.PRERELEASE_LABELS == tuple(ref["topology_labels"]["prerelease"])
    assert topo.GA_LABELS == tuple(ref["topology_labels"]["ga"])
    assert nrimod.CTR_DEVICE_KEY_PREFIX == ref["nri_container_device_key_prefix"]
    assert nrimod.CTR_DEVICE_KEY_PREFIX == "devices.gke.io/container." and "devices.gke.io/container." in open(os.path.join(root, "agent", "native", "dp", "nri_injector.cc")).read()
