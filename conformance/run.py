#!/usr/bin/env python3
"""Device-plugin conformance runner: drives ANY implementation of the plugin as a real process over real Unix sockets.

    python conformance/run.py --impl native            # build/agent/b200-device-plugin
    python conformance/run.py --impl python            # python -m container_engine_accelerators_b200.agent.main
    python conformance/run.py --command '/path/to/plugin -plugin-directory {plugin_dir} -gpu-config {gpu_config} \
        --dev-directory {dev_dir} --proc-directory {proc_dir} --pci-root {pci_root} --plugin-endpoint {endpoint}'

What it does (SURVEY §7.0: a language-neutral acceptance harness for BASELINE config 1; the scenarios are the reference's
pkg/gpu/nvidia/beta_plugin_test.go:36-614 plus the behaviours in SURVEY Appendix A.1-A.4): for every scenario it builds a throw-away
node — fake /dev (nvidiaN, nvidiactl, nvidia-uvm, ...), fake /proc MIG capability tree, fake /sys PCI tree, a gpu_config.json, a stub
kubelet listening on <plugin_dir>/kubelet.sock — starts the plugin with the scripted NVML (libfake_nvml.so, selected through
B200AGENT_NVML_LIB), plays the kubelet's side of the v1beta1 API with grpcio, and checks what comes back. Exit status 0 = all passed.
A plugin written in another language passes if it honours the same flags (or --command maps them) and loads NVML through an
overridable library path.
"""
from __future__ import annotations

import argparse
import json
import os
import shlex
import signal
import subprocess
import sys
import tempfile
import time
import traceback

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import grpc  # noqa: E402

from container_engine_accelerators_b200.agent import testing  # noqa: E402
from container_engine_accelerators_b200.agent.plugin import DevicePluginClient  # noqa: E402

FLAGS = ("-plugin-directory {plugin_dir} -gpu-config {gpu_config} --dev-directory {dev_dir} --proc-directory {proc_dir} --pci-root {pci_root} "
         "--plugin-endpoint {endpoint} --gpu-check-interval 0.6 --socket-check-interval 0.1")
PRESETS = {
    "native": os.path.join(ROOT, "build", "agent", "b200-device-plugin") + " " + FLAGS,
    "python": f"{shlex.quote(sys.executable)} -m container_engine_accelerators_b200.agent.main " + FLAGS.replace(" -plugin-directory", " --plugin-directory").replace("-gpu-config", "--gpu-config"),
}


class Node:
    """One throw-away node with a plugin process on it."""

    def __init__(self, command: str, gpus: int = 2, mig_parts: int = 0, config=None, numa=None, extra: str = "", env=None, kubelet: bool = True, real: bool = False):
        """real=True: no fakes on the device side — the host's /dev, /proc, /sys and the installed libnvidia-ml (tests/test_agent_gpu.py,
        run on a GPU box); the kubelet is still the stub."""
        self.tmp = tempfile.TemporaryDirectory(prefix="b200-conformance-", dir=testing.socket_tmp_root())
        root = self.tmp.name
        self.real = real
        self.plugin_dir = os.path.join(root, "device-plugins"); os.makedirs(self.plugin_dir)
        if real:
            self.dev, self.proc, self.pci_root = "/dev", "/proc", "/sys/bus/pci/devices"
        else:
            self.dev = testing.make_fake_dev(root, gpus)
            self.proc = testing.make_fake_mig(root, self.dev, gpus, mig_parts) if mig_parts else os.path.join(root, "proc")
            self.pci_root = os.path.join(root, "nopci")
            for i, node in enumerate(numa or []):                              # the scripted NVML reports 00000000:<1B+i>:00.0
                self.pci_root = testing.make_fake_pci(root, f"0000:{0x1b + i:02x}:00.0", node)
        self.gpu_config = os.path.join(root, "gpu_config.json")
        if config is not None:
            with open(self.gpu_config, "w") as f:
                f.write(config if isinstance(config, str) else json.dumps(config))
        self.endpoint = "nvidiaGPU-conformance.sock"
        self.kubelet = testing.KubeletStub(self.plugin_dir).start() if kubelet else None
        self.log_path = os.path.join(root, "plugin.log")
        self.log = open(self.log_path, "w")
        argv = shlex.split(command.format(plugin_dir=self.plugin_dir, gpu_config=self.gpu_config, dev_dir=self.dev, proc_dir=self.proc, pci_root=self.pci_root,
                                          endpoint=self.endpoint)) + shlex.split(extra)
        native_dir = os.path.join(ROOT, "build", "agent")
        penv = {**os.environ, "PYTHONPATH": ROOT + os.pathsep + os.environ.get("PYTHONPATH", ""), "B200AGENT_NVML_LIB": os.path.join(native_dir, "libfake_nvml.so"),
                "B200AGENT_NATIVE_LIB": os.path.join(native_dir, "libb200agent_nvml.so"), "FAKE_NVML_DEV_DIR": self.dev, "KUBERNETES_SERVICE_HOST": "", **(env or {})}
        if real:
            for k in ("B200AGENT_NVML_LIB", "FAKE_NVML_DEV_DIR"):
                penv.pop(k, None)
        self.process = subprocess.Popen(argv, env=penv, stdout=self.log, stderr=self.log)
        self.client = None

    def connect(self, timeout: float = 20.0) -> DevicePluginClient:
        path = os.path.join(self.plugin_dir, self.endpoint)
        deadline = time.time() + timeout
        while not os.path.exists(path):
            if time.time() > deadline or self.process.poll() is not None:
                raise AssertionError("plugin never created its socket:\n" + self.logs()[-3000:])
            time.sleep(0.05)
        if self.client:
            self.client.close()
        self.client = DevicePluginClient(path)
        self.client.wait_ready()
        return self.client

    def logs(self) -> str:
        self.log.flush()
        with open(self.log_path) as f:
            return f.read()

    def close(self) -> None:
        if self.client:
            self.client.close()
        if self.process.poll() is None:
            self.process.send_signal(signal.SIGTERM)
            try:
                self.process.wait(5)
            except subprocess.TimeoutExpired:
                self.process.kill()
        if self.kubelet:
            self.kubelet.stop()
        self.log.close()
        self.tmp.cleanup()


def first_list(client):
    stream = client.list_and_watch()
    return stream, {d.ID: d for d in next(stream).devices}


def expect_error(fn, needle: str) -> None:
    try:
        fn()
    except grpc.RpcError as e:
        assert needle in (e.details() or ""), f"wrong error: {e.details()!r}, wanted {needle!r}"
        return
    raise AssertionError(f"call succeeded, wanted an error containing {needle!r}")


# ------------------------------------------------------------------------------------------------- scenarios
def register_list_allocate(cmd):
    """Register{v1beta1, endpoint, nvidia.com/gpu} without options; full device list; 5 device specs + 2 read-only mounts per GPU."""
    n = Node(cmd)
    try:
        reg = n.kubelet.wait_registration(20)
        assert (reg.version, reg.endpoint, reg.resource_name) == ("v1beta1", n.endpoint, "nvidia.com/gpu") and not reg.HasField("options")
        c = n.connect()
        stream, devs = first_list(c)
        assert set(devs) == {"nvidia0", "nvidia1"} and all(d.health == "Healthy" for d in devs.values())
        cr = c.allocate(["nvidia0"]).container_responses[0]
        assert len(cr.devices) == 5 and len(cr.mounts) == 2 and dict(cr.envs) == {}
        assert cr.devices[0].host_path.endswith("/nvidia0") and all(d.permissions == "mrw" and d.host_path == d.container_path for d in cr.devices)
        assert all(m.read_only for m in cr.mounts) and cr.mounts[0].container_path == "/usr/local/nvidia"
        assert [len(r.devices) for r in c.allocate(["nvidia0", "nvidia1"], ["nvidia1"]).container_responses] == [6, 5]
        expect_error(lambda: c.allocate(["nvidia9"]), "invalid allocation request with non-existing device nvidia9")
        stream.cancel()
    finally:
        n.close()


def numa_topology(cmd):
    """TopologyInfo carries the NUMA node read from <pci-root>/<bus id>/numa_node."""
    n = Node(cmd, gpus=2, numa=[0, 1])
    try:
        _, devs = first_list(n.connect())
        assert [[x.ID for x in devs[d].topology.nodes] for d in ("nvidia0", "nvidia1")] == [[0], [1]]
    finally:
        n.close()


def time_sharing(cmd):
    """<id>/vgpu<k> fan-out; one virtual device per request under time-sharing."""
    n = Node(cmd, config={"GPUSharingConfig": {"GPUSharingStrategy": "time-sharing", "MaxSharedClientsPerGPU": 3}})
    try:
        c = n.connect()
        _, devs = first_list(c)
        assert set(devs) == {f"nvidia{g}/vgpu{k}" for g in range(2) for k in range(3)}
        assert c.allocate(["nvidia1/vgpu2"]).container_responses[0].devices[0].host_path.endswith("/nvidia1")
        expect_error(lambda: c.allocate(["nvidia0/vgpu0", "nvidia0/vgpu1"]), "time-sharing")
    finally:
        n.close()


def mig_seven_slices(cmd):
    """B200 1g.23gb: seven nvidia0/gi<N> resources, 7 device specs per slice (GPU + 2 caps + 4 defaults)."""
    n = Node(cmd, gpus=1, mig_parts=7, config={"GPUPartitionSize": "1g.23gb"})
    try:
        c = n.connect()
        _, devs = first_list(c)
        assert set(devs) == {f"nvidia0/gi{i}" for i in range(1, 8)}
        assert len(c.allocate(["nvidia0/gi3"]).container_responses[0].devices) == 7
        expect_error(lambda: c.allocate(["nvidia0/gi9"]), "non-existing GPU partition: nvidia0/gi9")
    finally:
        n.close()


def mig_with_time_sharing(cmd):
    """The fourth mode of the reference's matrix: MIG slices fanned out into time-shared replicas (nvidia0/gi<N>/vgpu<k>)."""
    n = Node(cmd, gpus=1, mig_parts=7, config={"GPUPartitionSize": "1g.23gb", "GPUSharingConfig": {"GPUSharingStrategy": "time-sharing", "MaxSharedClientsPerGPU": 2}})
    try:
        c = n.connect()
        _, devs = first_list(c)
        assert set(devs) == {f"nvidia0/gi{i}/vgpu{k}" for i in range(1, 8) for k in range(2)}
        cr = c.allocate(["nvidia0/gi5/vgpu1"]).container_responses[0]
        assert len(cr.devices) == 7 and cr.devices[0].host_path.endswith("/nvidia0")
        expect_error(lambda: c.allocate(["nvidia0/gi5/vgpu0", "nvidia0/gi5/vgpu1"]), "time-sharing")
        expect_error(lambda: c.allocate(["nvidia0/gi9/vgpu0"]), "non-existing GPU partition")
    finally:
        n.close()


def bad_config_falls_back(cmd):
    """An unparsable gpu_config.json is logged and ignored: whole GPUs are served."""
    n = Node(cmd, config="{broken json")
    try:
        _, devs = first_list(n.connect())
        assert set(devs) == {"nvidia0", "nvidia1"}
    finally:
        n.close()


def hot_add_and_socket_removal(cmd):
    """A new /dev/nvidiaN or a deleted plugin socket makes the plugin re-serve and re-register."""
    n = Node(cmd)
    try:
        n.kubelet.wait_registration(20)
        c = n.connect()
        testing.add_fake_gpu(n.dev, 2)
        assert n.kubelet.wait_registration(20).endpoint == n.endpoint
        _, devs = first_list(n.connect())
        assert set(devs) == {"nvidia0", "nvidia1", "nvidia2"}
        os.unlink(os.path.join(n.plugin_dir, n.endpoint))
        assert n.kubelet.wait_registration(20).endpoint == n.endpoint
        assert len(n.connect().allocate(["nvidia2"]).container_responses[0].devices) == 5
        del c
    finally:
        n.close()


def kubelet_appears_later(cmd):
    """No kubelet.sock at start: serve anyway, register when it shows up."""
    n = Node(cmd, kubelet=False)
    try:
        c = n.connect()
        assert len(c.allocate(["nvidia0"]).container_responses[0].devices) == 5
        n.kubelet = testing.KubeletStub(n.plugin_dir).start()
        assert n.kubelet.wait_registration(20).endpoint == n.endpoint
    finally:
        n.close()


def kubelet_restart(cmd):
    """The kubelet restarts (kubelet.sock is re-created): the plugin notices and registers again with the new instance."""
    n = Node(cmd)
    try:
        n.kubelet.wait_registration(20)
        n.connect()
        n.kubelet.stop()
        time.sleep(0.3)
        n.kubelet = testing.KubeletStub(n.plugin_dir).start()
        try:
            reg = n.kubelet.wait_registration(20)
        except TimeoutError as e:
            raise AssertionError(f"{e}; plugin log:\n{n.logs()[-2000:]}") from None
        assert reg.endpoint == n.endpoint and reg.resource_name == "nvidia.com/gpu"
        assert len(n.connect().allocate(["nvidia1"]).container_responses[0].devices) == 5
    finally:
        n.close()


def sigterm_clean_exit(cmd):
    """SIGTERM (pod deletion, rolling update): the plugin stops serving, removes its socket and exits 0 — also with a watch stream open."""
    n = Node(cmd)
    try:
        n.kubelet.wait_registration(20)
        c = n.connect()
        stream, devs = first_list(c)
        assert len(devs) == 2
        sock = os.path.join(n.plugin_dir, n.endpoint)
        assert os.path.exists(sock)
        n.process.send_signal(signal.SIGTERM)
        try:
            rc = n.process.wait(10)
        except subprocess.TimeoutExpired:
            raise AssertionError("plugin still running 10 s after SIGTERM; log:\n" + n.logs()[-2000:]) from None
        assert rc == 0, f"exit code {rc}; log:\n{n.logs()[-2000:]}"
        assert not os.path.exists(sock), "plugin socket left behind"
        stream.cancel()
    finally:
        n.close()


def xid_marks_unhealthy(cmd):
    """A health-critical Xid (XID_CONFIG) turns the device Unhealthy in the ListAndWatch stream and blocks its allocation; others are ignored."""
    events = tempfile.NamedTemporaryFile("w", suffix=".events", delete=False)
    events.close()
    n = Node(cmd, extra="-enable-health-monitoring", env={"FAKE_NVML_EVENTS": events.name, "XID_CONFIG": "31"})
    try:
        c = n.connect()
        stream, devs = first_list(c)
        assert all(d.health == "Healthy" for d in devs.values())
        time.sleep(1.0)
        with open(events.name, "a") as f:
            f.write("0 13\n1 31\n")
        assert {d.ID: d.health for d in next(stream).devices} == {"nvidia0": "Healthy", "nvidia1": "Unhealthy"}
        expect_error(lambda: c.allocate(["nvidia1"]), "unhealthy device nvidia1")
        stream.cancel()
    finally:
        n.close()
        os.unlink(events.name)


def xid_on_a_mig_slice(cmd):
    """An Xid that NVML attributes to GPU instance 3 takes down that slice only; one without a device id takes down everything."""
    events = tempfile.NamedTemporaryFile("w", suffix=".events", delete=False)
    events.close()
    n = Node(cmd, gpus=1, mig_parts=7, config={"GPUPartitionSize": "1g.23gb"}, extra="-enable-health-monitoring", env={"FAKE_NVML_EVENTS": events.name, "FAKE_NVML_MIG": "1"})
    try:
        c = n.connect()
        stream, devs = first_list(c)
        assert len(devs) == 7
        time.sleep(1.0)
        with open(events.name, "a") as f:
            f.write("0 48 3 0\n")
        health = {d.ID: d.health for d in next(stream).devices}
        assert health["nvidia0/gi3"] == "Unhealthy" and sum(1 for h in health.values() if h == "Unhealthy") == 1, health
        with open(events.name, "a") as f:
            f.write("-1 48\n")                                       # no device attached to the event: every device goes Unhealthy
        deadline = time.time() + 10
        while time.time() < deadline:
            health = {d.ID: d.health for d in next(stream).devices}
            if all(h == "Unhealthy" for h in health.values()):
                break
        assert all(h == "Unhealthy" for h in health.values()), health
        stream.cancel()
    finally:
        n.close()
        os.unlink(events.name)


def metrics_endpoint(cmd):
    """Prometheus text on the metrics port: per-container duty cycle / memory through the kubelet's PodResources API (virtual ids are not
    attributed), per-node gauges for every GPU, and the counters of a libb200coll page found in the stats directory."""
    import socket
    import struct
    import urllib.request
    from concurrent import futures
    from container_engine_accelerators_b200.agent import protos
    with tempfile.TemporaryDirectory(dir=testing.socket_tmp_root()) as d:
        pr = protos.podresources
        resp = pr.ListPodResourcesResponse()
        for ns, pod, ctr, ids in (("default", "trainer-0", "main", ["nvidia0"]), ("default", "shared-1", "main", ["nvidia1/vgpu0"])):
            resp.pod_resources.add(name=pod, namespace=ns).containers.add(name=ctr).devices.add(resource_name="nvidia.com/gpu", device_ids=ids)
        server = grpc.server(futures.ThreadPoolExecutor(max_workers=2))
        server.add_generic_rpc_handlers((grpc.method_handlers_generic_handler(protos.POD_RESOURCES_SERVICE, {"List": grpc.unary_unary_rpc_method_handler(
            lambda req, ctx: resp, pr.ListPodResourcesRequest.FromString, pr.ListPodResourcesResponse.SerializeToString)}),))
        sock = os.path.join(d, "pod-resources.sock")
        server.add_insecure_port(f"unix:{sock}")
        server.start()
        page = bytearray(4096); page[0:8] = b"B200COLL"
        struct.pack_into("<6I", page, 8, 2, 4242, 3, 8, 3, 1); struct.pack_into("<Q", page, 32, int(time.time()))
        struct.pack_into("<21Q", page, 64, 10, 0, 0, 2, 7, 1, 1 << 30, 0, 0, 4096, 512, 64, 0, 5, 0, 2, 13, 0, 0, 21, 0)
        with open(os.path.join(d, "b200coll.4242.3"), "wb") as f:
            f.write(page)
        s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
        n = Node(cmd, extra=f"-enable-container-gpu-metrics -gpu-metrics-port {port} -gpu-metrics-collection-interval 200 --pod-resources-socket {sock} --coll-stats-dir {d}",
                 env={"FAKE_NVML_UTIL": "40,60,80"})
        try:
            n.connect()
            body, deadline = "", time.time() + 20
            while time.time() < deadline and 'duty_cycle{' not in body:
                try:
                    body = urllib.request.urlopen(f"http://127.0.0.1:{port}/metrics", timeout=2).read().decode()
                except OSError:
                    pass
                time.sleep(0.2)
            lines = [l for l in body.splitlines() if not l.startswith("#")]
            find = lambda name, *labels: [l for l in lines if l.startswith(name + "{") and all(x in l for x in labels)]
            assert find("duty_cycle", 'pod="trainer-0"', 'container="main"', 'make="nvidia"', 'accelerator_id="GPU-fake-0"') and find("duty_cycle", 'pod="trainer-0"')[0].rsplit(" ", 1)[1] in ("60", "60.0"), body[-1500:]
            assert find("request", 'pod="trainer-0"', 'resource_name="nvidia.com/gpu"')[0].rsplit(" ", 1)[1] in ("1", "1.0")
            assert find("request", 'pod="shared-1"')[0].rsplit(" ", 1)[1] in ("0", "0.0") and not find("duty_cycle", 'pod="shared-1"')
            assert len(find("memory_total_gpu_node")) == 2 and len(find("duty_cycle_gpu_node")) == 2
            assert find("b200coll_calls", 'pid="4242"', 'rank="3"', 'op="all_reduce"')[0].rsplit(" ", 1)[1] in ("10", "10.0")
        finally:
            n.close()
            server.stop(0)


def mps_sharing(cmd):
    """MPS: the plugin only starts when nvidia-cuda-mps-control answers; one replica per container on multi-GPU nodes, several on a
    one-GPU node; allocations carry the thread-percentage / pinned-memory limits and the read-write /tmp/nvidia-mps mount."""
    cfg = {"GPUSharingConfig": {"GPUSharingStrategy": "mps", "MaxSharedClientsPerGPU": 4}}
    with tempfile.TemporaryDirectory() as d:
        ctl = os.path.join(d, "nvidia-cuda-mps-control")
        with open(ctl, "w") as f:
            f.write("#!/bin/sh\ncat > /dev/null\necho 100.0\n")
        os.chmod(ctl, 0o755)
        n = Node(cmd, config=cfg, extra=f"--mps-control-bin {ctl}")
        try:
            c = n.connect()
            _, devs = first_list(c)
            assert len(devs) == 8 and "nvidia1/vgpu3" in devs
            assert dict(c.allocate(["nvidia1/vgpu2"]).container_responses[0].envs)["CUDA_MPS_ACTIVE_THREAD_PERCENTAGE"] == "25"
            expect_error(lambda: c.allocate(["nvidia0/vgpu0", "nvidia0/vgpu1"]), "at most 1 nvidia.com/gpu can be requested on multi-GPU nodes")
        finally:
            n.close()
        n = Node(cmd, gpus=1, config=cfg, extra=f"--mps-control-bin {ctl}")          # a one-GPU node may hand several replicas to one container
        try:
            c = n.connect()
            cr = c.allocate(["nvidia0/vgpu0", "nvidia0/vgpu1"]).container_responses[0]
            env = dict(cr.envs)
            total_mib = (183359 << 20) // (1 << 20)                                  # what the scripted NVML reports per GPU
            assert env["CUDA_MPS_ACTIVE_THREAD_PERCENTAGE"] == "50" and env["CUDA_MPS_PINNED_DEVICE_MEM_LIMIT"] == f"0={2 * total_mib // 4}M", env
            assert ("/tmp/nvidia-mps", False) in [(m.container_path, m.read_only) for m in cr.mounts] and len(cr.mounts) == 3
        finally:
            n.close()
        with open(ctl, "w") as f:
            f.write("#!/bin/sh\nexit 1\n")
        n = Node(cmd, config=cfg, extra=f"--mps-control-bin {ctl}")
        try:
            time.sleep(1.5)
            assert not os.path.exists(os.path.join(n.plugin_dir, n.endpoint)) and n.process.poll() is None, "must not serve (and must keep retrying) while MPS is down"
            assert "MPS" in n.logs()
        finally:
            n.close()


def transport_profile(cmd):
    """GPUConfig.Transport = b200coll: Allocate exports the collective library's environment."""
    n = Node(cmd, config={"Transport": {"Name": "b200coll", "Env": {"B200COLL_ALGO": "nvls"}}})
    try:
        env = dict(n.connect().allocate(["nvidia0"]).container_responses[0].envs)
        assert env.get("B200COLL_LIB") == "/usr/local/nvidia/lib64/libb200coll.so" and env.get("B200COLL_ALGO") == "nvls"
    finally:
        n.close()


def real_hardware(cmd):
    """(--real only) No fakes on the device side: the host's /dev/nvidia*, /proc, /sys and the installed NVML; the stub kubelet must see every GPU node Healthy and get its device nodes on Allocate."""
    import re
    minors = sorted(int(m.group(1)) for m in (re.fullmatch(r"nvidia(\d+)", f) for f in os.listdir("/dev")) if m)
    assert minors, "no /dev/nvidia<N> on this host"
    n = Node(cmd, real=True)
    try:
        reg = n.kubelet.wait_registration(30)
        assert (reg.version, reg.resource_name) == ("v1beta1", "nvidia.com/gpu")
        c = n.connect()
        stream, devs = first_list(c)
        assert set(devs) == {f"nvidia{i}" for i in minors} and all(d.health == "Healthy" for d in devs.values()), devs
        first = f"nvidia{minors[0]}"
        paths = [d.host_path for d in c.allocate([first]).container_responses[0].devices]
        assert paths[0] == f"/dev/{first}" and "/dev/nvidiactl" in paths and all(os.path.exists(p) for p in paths), paths
        stream.cancel()
    finally:
        n.close()


SCENARIOS = [register_list_allocate, numa_topology, time_sharing, mig_seven_slices, mig_with_time_sharing, bad_config_falls_back, hot_add_and_socket_removal, kubelet_appears_later, kubelet_restart, sigterm_clean_exit,
             xid_marks_unhealthy, xid_on_a_mig_slice, metrics_endpoint, mps_sharing, transport_profile]


def main(argv=None) -> int:
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--impl", choices=sorted(PRESETS), help="one of this repository's two implementations")
    ap.add_argument("--command", help="command line template with {plugin_dir} {gpu_config} {dev_dir} {proc_dir} {pci_root} {endpoint}")
    ap.add_argument("--only", nargs="*", help="scenario names to run (default: all)")
    ap.add_argument("--list", action="store_true")
    ap.add_argument("--real", action="store_true", help="on a GPU node: run the one scenario that uses the host's real /dev, /proc, /sys and NVML instead of the fifteen fake-node scenarios")
    args = ap.parse_args(argv)
    if args.list:
        for s in SCENARIOS:
            print(f"{s.__name__:32s} {s.__doc__.strip()}")
        return 0
    cmd = args.command or PRESETS.get(args.impl or "")
    if not cmd:
        ap.error("give --impl or --command")
    if not os.path.exists(os.path.join(ROOT, "build", "agent", "libfake_nvml.so")):
        subprocess.run(["make", "-C", os.path.join(ROOT, "agent", "native"), "-j4"], check=True, capture_output=True)
    failed = 0
    for s in ([real_hardware] if args.real else SCENARIOS):
        if args.only and s.__name__ not in args.only:
            continue
        t0 = time.time()
        try:
            s(cmd)
            print(f"PASS  {s.__name__:32s} {time.time() - t0:5.1f}s")
        except Exception:
            failed += 1
            print(f"FAIL  {s.__name__:32s} {time.time() - t0:5.1f}s\n" + "\n".join("      " + l for l in traceback.format_exc().splitlines()[-12:]))
    print(f"{'FAILED' if failed else 'OK'}: {failed} scenario(s) failed" if failed else "OK: all scenarios passed")
    return 1 if failed else 0


if __name__ == "__main__":
    sys.exit(main())
