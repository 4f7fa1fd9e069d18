"""Health checker, metrics server and the native NVML binding (against the scripted fake libnvidia-ml).
Shapes follow the reference's tests: hand-built events and a fake API server with injected GET failures
(health_check/health_checker_test.go:44-462), a swappable collector with gauge assertions (metrics/metrics_test.go:26-209)."""
import json
import os
import time
from concurrent import futures

import grpc
import pytest
from prometheus_client import CollectorRegistry

from container_engine_accelerators_b200.agent import health, kube, metrics, nvml, protos, testing
from container_engine_accelerators_b200.agent.mig import Device


@pytest.fixture
def api():
    a = testing.FakeKubeApi().start()
    yield a
    a.stop()
    import yaml                                   # whatever the agent did to the API server must be allowed by the role it ships with
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    role = next(d for d in yaml.safe_load_all(open(os.path.join(root, "deploy", "device-plugin", "rbac.yaml"))) if d["kind"] == "ClusterRole")
    assert testing.rbac_violations(role, a.requests) == []


def make_checker(api, tmp_path, devices, xids=(), mock=None, sleep=lambda s: None):
    dev = testing.make_fake_dev(str(tmp_path), 2)
    m = mock or nvml.MockNvml(dev, uuids=["GPU-aaa", "GPU-bbb"])
    reported = []
    hc = health.GPUHealthChecker(devices, lambda d: reported.append(d) or True, list(xids), kube.KubeClient(api.url) if api else None, m, "node-1", sleep=sleep, wait_ms=1)
    return hc, m, reported


PLAIN = {"nvidia0": Device("nvidia0", "Healthy"), "nvidia1": Device("nvidia1", "Healthy")}


def test_xid48_marks_matching_device_unhealthy_and_sets_condition(api, tmp_path):
    api.add_node("node-1", boot_id="boot-A")
    hc, m, reported = make_checker(api, tmp_path, PLAIN)
    hc.start(background=False)
    m.events.append(nvml.XidEvent("GPU-bbb", 48))
    assert hc.poll_once()
    assert [(d.id, d.health) for d in reported] == [("nvidia1", "Unhealthy")]
    ev = api.events[-1]
    assert (ev["type"], ev["reason"], ev["message"], ev["source"]["component"]) == ("Warning", "XIDError", "Caught XID error, XID=48", "nvidia-gpu-device-plugin")
    cond = [c for c in api.nodes["node-1"]["status"]["conditions"] if c["type"] == "XidCriticalError"][0]
    assert (cond["status"], cond["reason"], cond["message"]) == ("True", '{"48":true}', "boot-A")


def test_monitor_only_xid_sets_condition_but_keeps_device_healthy(api, tmp_path):
    api.add_node("node-1", boot_id="boot-A")
    hc, m, reported = make_checker(api, tmp_path, PLAIN)
    hc.start(background=False)
    for xid in (79, 79, 63):
        m.events.append(nvml.XidEvent("GPU-aaa", xid))
        hc.poll_once()
    assert reported == []
    cond = [c for c in api.nodes["node-1"]["status"]["conditions"] if c["type"] == "XidCriticalError"][0]
    assert cond["reason"] == '{"63":true,"79":true}'                                     # sorted keys, duplicate wrote nothing
    puts = [r for r in api.requests if r[0] == "PUT" and r[1].endswith("/status")]
    assert len(puts) == 2


def test_configured_xid_is_critical_and_unknown_xid_is_ignored(api, tmp_path):
    api.add_node("node-1")
    hc, m, reported = make_checker(api, tmp_path, PLAIN, xids=[31])
    hc.start(background=False)
    m.events.append(nvml.XidEvent("GPU-aaa", 13)); hc.poll_once()
    assert reported == []
    m.events.append(nvml.XidEvent("GPU-aaa", 31)); hc.poll_once()
    assert [d.id for d in reported] == ["nvidia0"]
    assert not any(c["type"] == "XidCriticalError" for c in api.nodes["node-1"]["status"]["conditions"])   # 31 is not in the monitor set


def test_event_without_uuid_marks_all_devices(api, tmp_path):
    api.add_node("node-1")
    hc, m, reported = make_checker(api, tmp_path, PLAIN)
    hc.start(background=False)
    m.events.append(nvml.XidEvent("", 48)); hc.poll_once()
    assert sorted(d.id for d in reported) == ["nvidia0", "nvidia1"] and all(d.health == "Unhealthy" for d in reported)


def test_mig_device_matching(api, tmp_path):
    api.add_node("node-1")
    devs = {f"nvidia0/gi{i}": Device(f"nvidia0/gi{i}", "Healthy") for i in (1, 2, 3)}
    hc, m, reported = make_checker(api, tmp_path, devs)
    hc.start(background=False)
    m.events.append(nvml.XidEvent("GPU-aaa", 48, gpu_instance_id=2, compute_instance_id=0)); hc.poll_once()
    assert [d.id for d in reported] == ["nvidia0/gi2"]
    m.events.append(nvml.XidEvent("GPU-aaa", 48)); hc.poll_once()        # full-GPU event does not match any slice
    assert len(reported) == 1


def test_not_supported_registration_is_tolerated(api, tmp_path):
    api.add_node("node-1")
    hc, m, reported = make_checker(api, tmp_path, PLAIN)
    m.events_supported = False
    hc.start(background=False)          # must not raise: such GPUs are always healthy
    assert not hc.poll_once()


def test_reset_condition_depends_on_boot_id(api, tmp_path):
    xid_cond = {"type": "XidCriticalError", "status": "True", "reason": '{"48":true}', "message": "boot-OLD"}
    api.add_node("node-1", boot_id="boot-NEW", conditions=[{"type": "Ready", "status": "True"}, dict(xid_cond)])
    hc, _, _ = make_checker(api, tmp_path, PLAIN)
    assert hc.reset_xid_condition() is True
    assert [c["type"] for c in api.nodes["node-1"]["status"]["conditions"]] == ["Ready"]
    api.add_node("node-1", boot_id="boot-OLD", conditions=[dict(xid_cond)])     # plugin restart, same boot: keep
    assert hc.reset_xid_condition() is False
    assert len(api.nodes["node-1"]["status"]["conditions"]) == 1


def test_reset_retries_with_backoff(api, tmp_path):
    api.add_node("node-1")
    api.fail_next_gets = 2
    sleeps = []
    hc, _, _ = make_checker(api, tmp_path, PLAIN, sleep=sleeps.append)
    assert hc.reset_xid_condition_with_backoff() is True
    assert sleeps == [1.0, 2.0]                       # >= 3 s of backoff before the third GET succeeds


def test_heartbeat_only_touches_true_condition(api, tmp_path):
    api.add_node("node-1", conditions=[{"type": "XidCriticalError", "status": "True", "reason": "{}", "message": "b", "lastHeartbeatTime": "old"}])
    hc, _, _ = make_checker(api, tmp_path, PLAIN)
    assert hc.update_last_heartbeat() is True
    assert api.nodes["node-1"]["status"]["conditions"][0]["lastHeartbeatTime"] != "old"
    api.add_node("node-1")
    assert hc.update_last_heartbeat() is False


# ------------------------------------------------------------------------------------------------- metrics
class PodResourcesStub:
    def __init__(self, sock, pods, service=None):
        pr = protos.podresources
        resp = pr.ListPodResourcesResponse()
        for ns, pod, ctr, resource, ids in pods:
            p = resp.pod_resources.add(name=pod, namespace=ns)
            c = p.containers.add(name=ctr)
            c.devices.add(resource_name=resource, device_ids=ids)
        self.server = grpc.server(futures.ThreadPoolExecutor(max_workers=2))
        h = grpc.method_handlers_generic_handler(service or protos.POD_RESOURCES_SERVICE, {"List": grpc.unary_unary_rpc_method_handler(
            lambda req, ctx: resp, pr.ListPodResourcesRequest.FromString, pr.ListPodResourcesResponse.SerializeToString)})
        self.server.add_generic_rpc_handlers((h,))
        self.server.add_insecure_port(f"unix:{sock}")
        self.server.start()


@pytest.mark.parametrize("service", [protos.POD_RESOURCES_SERVICE, protos.POD_RESOURCES_SERVICE_V1])
def test_pod_resources_v1_and_v1alpha1_kubelets(tmp_path, service):
    """A kubelet that serves only one of the two API versions is understood either way (v1 is tried first)."""
    sock = str(tmp_path / "pr.sock")
    stub = PodResourcesStub(sock, [("default", "p1", "c1", "nvidia.com/gpu", ["nvidia1"])], service=service)
    try:
        assert metrics.get_devices_for_all_containers(sock) == {("default", "p1", "c1"): ["nvidia1"]}
    finally:
        stub.server.stop(0)


def test_container_device_map_filters_resource_and_virtual_ids(tmp_path):
    sock = str(tmp_path / "pr.sock")
    stub = PodResourcesStub(sock, [("default", "p1", "c1", "nvidia.com/gpu", ["nvidia0", "nvidia1"]), ("default", "p2", "c1", "nvidia.com/gpu", ["nvidia0/vgpu1"]),
                                   ("kube-system", "p3", "c9", "example.com/fpga", ["f0"])])
    try:
        got = metrics.get_devices_for_all_containers(sock)
        assert got == {("default", "p1", "c1"): ["nvidia0", "nvidia1"], ("default", "p2", "c1"): []}
    finally:
        stub.server.stop(0)


def sample(reg, name, labels):
    return reg.get_sample_value(name, labels)


def test_update_metrics_and_minute_reset(tmp_path):
    dev = testing.make_fake_dev(str(tmp_path), 2)
    m = nvml.MockNvml(dev, uuids=["GPU-aaa", "GPU-bbb"], mem_total=180 << 30)
    m.utilisation = {"GPU-aaa": 78, "GPU-bbb": 150}        # 150 > 100 => skipped this tick
    clock = [1000.0]
    reg = CollectorRegistry()
    ms = metrics.MetricServer(m, registry=reg, coll_stats_glob=str(tmp_path / "none*"), now=lambda: clock[0])
    ms.discover_gpu_devices()
    ms.update_metrics({("ns", "pod", "ctr"): ["nvidia0", "nvidia1"]})
    lab = {"namespace": "ns", "pod": "pod", "container": "ctr", "make": "nvidia", "accelerator_id": "GPU-aaa", "model": "NVIDIA B200"}
    assert sample(reg, "duty_cycle", lab) == 78
    assert sample(reg, "memory_total", lab) == float(180 << 30)
    assert sample(reg, "request", {"namespace": "ns", "pod": "pod", "container": "ctr", "resource_name": "nvidia.com/gpu"}) == 2
    assert sample(reg, "duty_cycle", {**lab, "accelerator_id": "GPU-bbb"}) is None
    assert sample(reg, "duty_cycle_gpu_node", {"make": "nvidia", "accelerator_id": "GPU-aaa", "model": "NVIDIA B200"}) == 78
    clock[0] += 61
    ms.update_metrics({})                                   # dead container's series must disappear
    assert sample(reg, "duty_cycle", lab) is None and sample(reg, "duty_cycle_gpu_node", {"make": "nvidia", "accelerator_id": "GPU-aaa", "model": "NVIDIA B200"}) == 78


def test_coll_stats_page_is_exported(tmp_path):
    import struct
    page = bytearray(4096)
    page[0:8] = b"B200COLL"
    struct.pack_into("<6I", page, 8, 1, 4242, 3, 8, 3, 1)
    struct.pack_into("<17Q", page, 64, 10, 0, 0, 2, 1 << 30, 0, 0, 4096, 0, 7, 0, 1, 2, 0, 5, 12, 0)
    (tmp_path / "b200coll.4242.3").write_bytes(page)
    pages = metrics.read_coll_stats_pages(str(tmp_path / "b200coll.*"))
    assert pages[0]["pid"] == 4242 and pages[0]["calls"][0] == 10 and pages[0]["algo_calls"][1] == 7 and pages[0]["kernel_launches"] == 12
    dev = testing.make_fake_dev(str(tmp_path), 1)
    reg = CollectorRegistry()
    ms = metrics.MetricServer(nvml.MockNvml(dev), registry=reg, coll_stats_glob=str(tmp_path / "b200coll.*"))
    ms.update_metrics({})
    assert sample(reg, "b200coll_calls", {"pid": "4242", "rank": "3", "op": "all_reduce"}) == 10
    assert sample(reg, "b200coll_algo_calls", {"pid": "4242", "rank": "3", "algo": "ll"}) == 7
    assert sample(reg, "b200coll_calls", {"pid": "4242", "rank": "3", "op": "broadcast"}) == 0      # v1 page: no rooted-op counters


def test_coll_stats_page_v2_has_broadcast_and_reduce(tmp_path):
    import struct
    page = bytearray(4096)
    page[0:8] = b"B200COLL"
    struct.pack_into("<6I", page, 8, 2, 77, 0, 8, 0, 1)
    #                                 calls (6 ops)        bytes (6 ops)                     algo_calls (7)        launches staged
    struct.pack_into("<21Q", page, 64, 1, 2, 3, 4, 5, 6, 10, 20, 30, 40, 50, 60, 0, 1, 0, 2, 9, 0, 0, 21, 3)
    struct.pack_into("<3Q", page, 64 + 21 * 8, 7, 8, 9000)                     # p2p sends, recvs, bytes (appended to the v2 payload)
    struct.pack_into("<6Q", page, 64 + 24 * 8, 11, 1 << 33, 4, 5, 13, 17)      # host calls / bytes / zero-copy / pipelined, bulk launches, generic launches
    (tmp_path / "b200coll.77.0").write_bytes(page)
    pg = metrics.read_coll_stats_pages(str(tmp_path / "b200coll.*"))[0]
    assert (pg["p2p_sends"], pg["p2p_recvs"], pg["p2p_bytes"]) == (7, 8, 9000)
    assert pg["version"] == 2 and pg["calls"] == (1, 2, 3, 4, 5, 6) and pg["bytes"][4:] == (50, 60)
    assert pg["algo_calls"] == (0, 1, 0, 2, 9, 0, 0) and pg["kernel_launches"] == 21 and pg["staged_calls"] == 3
    reg = CollectorRegistry()
    ms = metrics.MetricServer(nvml.MockNvml(testing.make_fake_dev(str(tmp_path), 1)), registry=reg, coll_stats_glob=str(tmp_path / "b200coll.*"))
    ms.update_metrics({})
    assert sample(reg, "b200coll_calls", {"pid": "77", "rank": "0", "op": "reduce"}) == 6
    assert sample(reg, "b200coll_bytes", {"pid": "77", "rank": "0", "op": "broadcast"}) == 50
    assert sample(reg, "b200coll_p2p_calls", {"pid": "77", "rank": "0", "dir": "recv"}) == 8 and sample(reg, "b200coll_p2p_bytes", {"pid": "77", "rank": "0"}) == 9000
    assert (pg["host_calls"], pg["host_bytes"], pg["host_zero_copy"], pg["host_pipelined"], pg["bulk_launches"], pg["generic_launches"]) == (11, 1 << 33, 4, 5, 13, 17)
    assert sample(reg, "b200coll_host_calls", {"pid": "77", "rank": "0", "path": "pipelined"}) == 5 and sample(reg, "b200coll_host_bytes", {"pid": "77", "rank": "0"}) == 1 << 33
    assert sample(reg, "b200coll_kernel_family_launches", {"pid": "77", "rank": "0", "family": "generic"}) == 17
    # header timestamp: a fresh page is exported, one that has not been touched for more than an hour is a leftover of a dead process
    import time as _time
    struct.pack_into("<Q", page, 32, int(_time.time()) - 30); (tmp_path / "b200coll.77.0").write_bytes(page)
    assert len(metrics.read_coll_stats_pages(str(tmp_path / "b200coll.*"))) == 1
    struct.pack_into("<Q", page, 32, int(_time.time()) - 7200); (tmp_path / "b200coll.77.0").write_bytes(page)
    assert metrics.read_coll_stats_pages(str(tmp_path / "b200coll.*")) == []


# ------------------------------------------------------------------------------------------------- native binding
@pytest.fixture
def native(native_build, monkeypatch, tmp_path):
    monkeypatch.setenv("B200AGENT_NVML_LIB", os.path.join(native_build, "libfake_nvml.so"))
    monkeypatch.setenv("FAKE_NVML_GPUS", "3")
    return native_build


def run_py(code, env):
    import subprocess, sys
    return subprocess.run([sys.executable, "-c", code], env={**os.environ, **env}, capture_output=True, text=True, timeout=60)


def test_native_nvml_enumeration_sampler_and_events(native, tmp_path):
    # one subprocess per scenario: the native library resolves NVML once per process
    events = tmp_path / "events.txt"
    events.write_text("1 48\n-1 79\n0 31 2 0\n")
    code = """
import json
from container_engine_accelerators_b200.agent import nvml
n = nvml.NativeNvml(); n.init()
out = {"count": n.device_count(), "dev1": n.device(1).__dict__, "driver": n.driver_version(), "util": n.average_usage("GPU-fake-0", 0)}
h = n.events_open()
out["reg"] = [n.events_register(h, i) for i in range(3)]
evs = []
for _ in range(4):
    e = n.events_wait(h, 10)
    evs.append(None if e is None else [e.uuid, e.xid, e.gpu_instance_id, e.compute_instance_id, e.event_type])
out["events"] = evs
n.events_close(h)
print(json.dumps(out))
"""
    r = run_py(code, {"FAKE_NVML_EVENTS": str(events), "FAKE_NVML_UTIL": "40,60,80"})
    assert r.returncode == 0, r.stderr
    out = json.loads(r.stdout)
    assert out["count"] == 3 and out["dev1"]["minor"] == 1 and out["dev1"]["uuid"] == "GPU-fake-1" and out["dev1"]["bus_id"] == "00000000:1C:00.0"
    assert out["driver"] == "580.159.03" and out["util"] == 60 and out["reg"] == [True, True, True]
    assert out["events"] == [["GPU-fake-1", 48, 0xFFFFFFFF, 0xFFFFFFFF, 8], ["", 79, 0xFFFFFFFF, 0xFFFFFFFF, 8], ["GPU-fake-0", 31, 2, 0, 8], None]


def test_native_sampler_guards_zero_samples_and_unsupported_events(native):
    code = """
from container_engine_accelerators_b200.agent import nvml
n = nvml.NativeNvml(); n.init()
try:
    n.average_usage("GPU-fake-0", 0); print("no-error")
except nvml.NvmlError as e:
    print("code", e.code)
h = n.events_open(); print("reg", n.events_register(h, 0))
"""
    r = run_py(code, {"FAKE_NVML_UTIL": "", "FAKE_NVML_NO_EVENTS": "1"})
    assert r.returncode == 0, r.stderr
    assert "code -5" in r.stdout and "reg False" in r.stdout          # reference divides by sampleCount == 0 here (util.go:82)


def test_native_sampler_falls_back_when_the_driver_refuses_samples(native):
    """Some drivers size the utilisation sample buffer, then refuse to fill it (NOT_SUPPORTED). The duty cycle is then the driver's
    utilisation rate over its last sample period; a cut-off in the future still has no sample."""
    code = """
import time
from container_engine_accelerators_b200.agent import nvml
n = nvml.NativeNvml(); n.init()
print("util", n.average_usage("GPU-fake-0", int((time.time() - 10) * 1e6)))
try:
    n.average_usage("GPU-fake-0", int((time.time() + 3600) * 1e6)); print("no-error")
except nvml.NvmlError as e:
    print("future", e.code)
"""
    r = run_py(code, {"FAKE_NVML_UTIL": "40,60,95", "FAKE_NVML_SAMPLES_UNSUPPORTED": "1"})
    assert r.returncode == 0, r.stderr
    assert "util 95" in r.stdout and "future -5" in r.stdout, r.stdout


def test_native_without_nvml_library_reports_cleanly(native_build):
    code = """
from container_engine_accelerators_b200.agent import nvml
try:
    nvml.NativeNvml().init(); print("unexpected")
except nvml.NvmlError as e:
    print("code", e.code)
"""
    r = run_py(code, {"B200AGENT_NVML_LIB": "/nonexistent/libnvidia-ml.so.1"})
    assert r.returncode == 0 and ("code -1" in r.stdout or "unexpected" in r.stdout)


def test_health_checker_end_to_end_through_native_binding(native, tmp_path):
    """fake NVML -> native binding -> health checker -> manager queue -> ListAndWatch view."""
    events = tmp_path / "events.txt"
    events.write_text("2 48\n")
    code = f"""
import json
from container_engine_accelerators_b200.agent import nvml, health, manager, testing
from container_engine_accelerators_b200.agent.config import GPUConfig
dev = testing.make_fake_dev({str(tmp_path)!r}, 3)
n = nvml.NativeNvml(); n.init()
ngm = manager.GPUManager(dev, {str(tmp_path / 'proc')!r}, [], GPUConfig(), nvml=n, pci_root={str(tmp_path)!r})
ngm.start()
hc = health.GPUHealthChecker(ngm.list_physical_devices(), ngm.report_unhealthy, [], None, n, "node", wait_ms=10)
hc.start(background=False)
assert hc.poll_once()
d = ngm.health.get_nowait()
ngm.set_device_health(d.id, d.health, d.numa_node)
print(json.dumps({{k: v.health for k, v in ngm.list_devices().items()}}))
"""
    r = run_py(code, {"FAKE_NVML_EVENTS": str(events)})
    assert r.returncode == 0, r.stderr
    assert json.loads(r.stdout.strip().splitlines()[-1]) == {"nvidia0": "Healthy", "nvidia1": "Healthy", "nvidia2": "Unhealthy"}


def test_background_checker_lifecycle_and_api_failures(api, tmp_path, monkeypatch):
    """start() in the background (reset + heartbeat + listener threads), an event arriving while it runs, API-server failures on
    every path (logged, never fatal: the device still goes Unhealthy), and stop() joining the listener before the event set is freed."""
    monkeypatch.setattr(health, "HEARTBEAT_S", 0.05)
    stale = {"type": "XidCriticalError", "status": "True", "reason": '{"48":true}', "message": "boot-OLD", "lastHeartbeatTime": "2020-01-01T00:00:00Z"}
    api.add_node("node-1", boot_id="boot-A", conditions=[{"type": "Ready", "status": "True"}, dict(stale)])
    hc, m, reported = make_checker(api, tmp_path, PLAIN)
    closed = []
    orig_close = m.events_close
    m.events_close = lambda h: (closed.append(h), orig_close(h))[1]
    hc.start()                                                             # background=True
    deadline = time.time() + 5
    while time.time() < deadline and any(c["type"] == "XidCriticalError" for c in api.nodes["node-1"]["status"]["conditions"]):
        time.sleep(0.02)
    assert not any(c["type"] == "XidCriticalError" for c in api.nodes["node-1"]["status"]["conditions"])     # rebooted since: cleared at start-up
    m.events.append(nvml.XidEvent("GPU-aaa", 48))
    while time.time() < deadline and not reported:
        time.sleep(0.02)
    assert [(d.id, d.health) for d in reported] == [("nvidia0", "Unhealthy")]
    cond = lambda: next(c for c in api.nodes["node-1"]["status"]["conditions"] if c["type"] == "XidCriticalError")
    first = cond()["lastHeartbeatTime"]
    time.sleep(1.2)
    assert cond()["lastHeartbeatTime"] > first                              # heartbeat thread refreshes it
    # the API server goes away: events keep marking devices, nothing raises
    api.fail_next_gets = 10 ** 6
    m.events.append(nvml.XidEvent("GPU-bbb", 79))                           # monitored only; needs the API for everything it does
    m.events.append(nvml.XidEvent("GPU-bbb", 48))
    while time.time() < deadline + 5 and len(reported) < 2:
        time.sleep(0.02)
    assert [(d.id, d.health) for d in reported][1] == ("nvidia1", "Unhealthy")
    assert hc.update_last_heartbeat() is False
    hc.stop()
    assert closed and hc._event_set is None and not any(t.is_alive() for t in hc._threads)
    api.fail_next_gets = 0


def test_status_updates_survive_write_conflicts(api, tmp_path):
    """A kubelet status write between our GET and PUT makes the API server answer 409: re-read and retry, do not lose the condition."""
    api.add_node("node-1", boot_id="boot-A")
    hc, m, reported = make_checker(api, tmp_path, PLAIN)
    hc.start(background=False)
    api.stale_next_puts = 2
    m.events.append(nvml.XidEvent("GPU-aaa", 79))
    hc.poll_once()
    cond = [c for c in api.nodes["node-1"]["status"]["conditions"] if c["type"] == "XidCriticalError"]
    assert cond and cond[0]["reason"] == '{"79":true}' and api.conflicts == 2
    api.stale_next_puts = 1
    assert hc.update_last_heartbeat() is True and api.conflicts == 3
    api.stale_next_puts = 10                                     # persistent conflicts: give up after a few attempts, logged, not raised
    m.events.append(nvml.XidEvent("GPU-aaa", 63))
    hc.poll_once()
    assert json.loads([c for c in api.nodes["node-1"]["status"]["conditions"] if c["type"] == "XidCriticalError"][0]["reason"]) == {"79": True}
    api.stale_next_puts = 0
