"""NRI device injector: annotation parsing (reference nri_device_injector_test.go:95-190 YAML cases), lstat-derived
device identity (:25-93, which needs root for mknod — here a fake lstat covers b/c/p and a real FIFO covers the syscall),
and the full wire path against a fake containerd NRI runtime (mux + ttrpc), which the reference does not test."""
import os
import stat
import threading
import types

import pytest

from container_engine_accelerators_b200.agent import nri, protos, testing

KEY = "devices.gke.io/container."


def test_get_devices_cases():
    assert nri.get_devices("c", {}) == []
    assert nri.get_devices("c", {KEY + "other": "- path: /dev/x"}) == []
    devs = nri.get_devices("c", {KEY + "c": "- path: /dev/nvidia0\n- path: /dev/nvidiactl\n  file_mode: 438\n- path: /dev/nvidia0\n  uid: 7\n"})
    assert [d["path"] for d in devs] == ["/dev/nvidia0", "/dev/nvidiactl"]       # duplicate path: first wins
    assert devs[1]["file_mode"] == 438 and "uid" not in devs[0]
    with pytest.raises(nri.DeviceError, match="invalid device annotation"):
        nri.get_devices("c", {KEY + "c": "- path: [unclosed"})
    with pytest.raises(nri.DeviceError, match="invalid device annotation"):
        nri.get_devices("c", {KEY + "c": "just a string"})


def fake_lstat(mode, major=195, minor=3):
    return lambda path: types.SimpleNamespace(st_mode=mode, st_rdev=os.makedev(major, minor))


@pytest.mark.parametrize("mode,want", [(stat.S_IFCHR | 0o666, "c"), (stat.S_IFBLK | 0o660, "b"), (stat.S_IFIFO | 0o600, "p")])
def test_to_nri_device_types(mode, want):
    d = nri.to_nri_device({"path": "/dev/nvidia3", "type": "ignored", "major": 1, "minor": 2}, fake_lstat(mode))
    assert (d.type, d.major, d.minor, d.path) == (want, 195, 3, "/dev/nvidia3")    # type/major/minor re-derived, annotation values ignored
    assert not d.HasField("file_mode") and not d.HasField("uid") and not d.HasField("gid")


def test_to_nri_device_optional_fields_and_errors(tmp_path):
    d = nri.to_nri_device({"path": "/dev/x", "file_mode": 0o666, "uid": 1000, "gid": 44}, fake_lstat(stat.S_IFCHR))
    assert (d.file_mode.value, d.uid.value, d.gid.value) == (0o666, 1000, 44)
    with pytest.raises(nri.DeviceError, match="invalid device type"):
        nri.to_nri_device({"path": "/tmp"}, fake_lstat(stat.S_IFDIR))
    with pytest.raises(nri.DeviceError, match="failed to get info from device path"):
        nri.to_nri_device({"path": str(tmp_path / "missing")})
    fifo = tmp_path / "fifo"
    os.mkfifo(fifo)
    assert nri.to_nri_device({"path": str(fifo)}).type == "p"


def test_create_container_nil_pod_is_noop():
    from container_engine_accelerators_b200.agent.protos import nri as pb
    adj = nri.create_container(None, pb.Container(name="c"))
    assert len(adj.linux.devices) == 0


def test_wire_register_configure_create_container(tmp_path):
    sock = str(tmp_path / "nri.sock")
    rt = testing.FakeNriRuntime(sock)
    fifo = tmp_path / "dev-fifo"
    os.mkfifo(fifo)
    plugin = nri.DeviceInjectorPlugin(sock)
    t = threading.Thread(target=plugin.run, daemon=True)
    t.start()
    try:
        reg = rt.wait_registered()
        assert (reg.plugin_name, reg.plugin_idx) == ("device_injector_nri", "10")
        cfg = rt.configure()
        assert cfg.events & (1 << 3)                      # subscribed to CREATE_CONTAINER
        rt.synchronize()
        resp = rt.create_container("pod", "rxdm", {KEY + "rxdm": f"- path: {fifo}\n  gid: 5\n- path: {fifo}\n", KEY + "other": "- path: /nonexistent"})
        devs = resp.adjust.linux.devices
        assert len(devs) == 1 and devs[0].path == str(fifo) and devs[0].type == "p" and devs[0].gid.value == 5
        assert len(rt.create_container("pod", "plain", {}).adjust.linux.devices) == 0
        with pytest.raises(RuntimeError, match="failed to get info from device path /nonexistent"):
            rt.create_container("pod", "other", {KEY + "other": "- path: /nonexistent"})      # error => container creation fails
    finally:
        rt.close()
        t.join(5)
    assert not t.is_alive()                                # plugin returns when the runtime goes away


def test_native_injector_wire_path(tmp_path, native_build):
    """The C++ plugin (build/agent/b200-nri-device-injector) against the same fake containerd NRI runtime."""
    import subprocess
    sock = str(tmp_path / "nri.sock")
    rt = testing.FakeNriRuntime(sock)
    fifo = tmp_path / "dev-fifo"
    os.mkfifo(fifo)
    proc = subprocess.Popen([os.path.join(native_build, "b200-nri-device-injector"), "--socket", sock], stderr=subprocess.PIPE)
    try:
        reg = rt.wait_registered()
        assert (reg.plugin_name, reg.plugin_idx) == ("device_injector_nri", "10")
        assert rt.configure().events & (1 << 3)
        rt.synchronize()
        resp = rt.create_container("pod", "rxdm", {KEY + "rxdm": f"- path: {fifo}\n  gid: 5\n  type: ignored\n- path: {fifo}\n", KEY + "other": "- path: /nonexistent"})
        devs = resp.adjust.linux.devices
        assert len(devs) == 1 and devs[0].path == str(fifo) and devs[0].type == "p" and devs[0].gid.value == 5 and not devs[0].HasField("uid")
        flow = rt.create_container("pod", "flow", {KEY + "flow": f"[{{path: {fifo}, file_mode: 438}}]"})
        assert flow.adjust.linux.devices[0].file_mode.value == 438
        assert len(rt.create_container("pod", "plain", {}).adjust.linux.devices) == 0
        with pytest.raises(RuntimeError, match="failed to get info from device path /nonexistent"):
            rt.create_container("pod", "other", {KEY + "other": "- path: /nonexistent"})
        with pytest.raises(RuntimeError, match="invalid device annotation"):
            rt.create_container("pod", "bad", {KEY + "bad": "- path: [unclosed"})
        with pytest.raises(RuntimeError, match="invalid device annotation"):
            rt.create_container("pod", "bad2", {KEY + "bad2": "just a string"})
    finally:
        rt.close()
        try:
            proc.wait(5)
        except subprocess.TimeoutExpired:
            proc.kill()
    assert proc.returncode == 0           # exits cleanly when the runtime goes away


def _mknod_or_skip(path, mode, major, minor):
    try:
        os.mknod(path, mode, os.makedev(major, minor))
    except PermissionError:
        pytest.skip("needs CAP_MKNOD (the reference runs this test under sudo: Makefile:97-102)")


def test_real_device_nodes_python_and_native_agree(tmp_path, native_build):
    """lstat on real char/block nodes (reference nri_device_injector_test.go:25-93): type, major and minor come from the node,
    never from the annotation — checked for the Python plugin's helper and for the C++ binary over the wire."""
    import subprocess
    ch, blk = tmp_path / "nvidia7", tmp_path / "loop9"
    _mknod_or_skip(ch, stat.S_IFCHR | 0o666, 195, 7)
    _mknod_or_skip(blk, stat.S_IFBLK | 0o660, 7, 9)
    d = nri.to_nri_device({"path": str(ch), "type": "b", "major": 1, "minor": 2})          # annotation lies: ignored
    assert (d.type, d.major, d.minor) == ("c", 195, 7)
    sock = str(tmp_path / "nri.sock")
    rt = testing.FakeNriRuntime(sock)
    proc = subprocess.Popen([os.path.join(native_build, "b200-nri-device-injector"), "--socket", sock], stderr=subprocess.PIPE)
    try:
        rt.wait_registered(); rt.configure(); rt.synchronize()
        devs = rt.create_container("pod", "c", {KEY + "c": f"- path: {ch}\n  type: b\n  major: 1\n- path: {blk}\n  uid: 7\n"}).adjust.linux.devices
        assert [(x.path, x.type, x.major, x.minor) for x in devs] == [(str(ch), "c", 195, 7), (str(blk), "b", 7, 9)]
        assert devs[1].uid.value == 7 and not devs[0].HasField("uid")
    finally:
        rt.close()
        try:
            proc.wait(5)
        except subprocess.TimeoutExpired:
            proc.kill()


def test_native_annotation_parser_agrees_with_pyyaml_on_generated_annotations(native_build):
    """The C++ plugin has its own parser for the subset of YAML that annotations use (block lists of flat mappings, flow form,
    JSON form, comments, quotes, octal modes). Property test: for generated documents in that subset it extracts exactly what
    the Python plugin (PyYAML) extracts."""
    import subprocess
    from hypothesis import HealthCheck, given, settings, strategies as st
    exe = os.path.join(native_build, "b200-nri-device-injector")
    seg = st.text(alphabet="abcdefghijklmnopqrstuvwxyz0123456789_-.", min_size=1, max_size=8)
    path = st.builds(lambda parts, colon: "/dev/" + "/".join(parts) + (":" + parts[0] if colon else ""), st.lists(seg, min_size=1, max_size=3), st.booleans())
    dev = st.fixed_dictionaries({"path": path}, optional={"file_mode": st.sampled_from([0o666, 0o660, 0o600, 438]), "uid": st.integers(0, 70000), "gid": st.integers(0, 70000),
                                                       "type": st.sampled_from(["c", "b"]), "major": st.integers(0, 511)})
    style = st.sampled_from(["block", "flow", "json", "block_comments", "block_quoted"])

    def render(devs, how):
        if how == "json":
            import json as _json
            return _json.dumps(devs)
        if how == "flow":
            return "[" + ", ".join("{" + ", ".join(f"{k}: {v}" for k, v in d.items()) + "}" for d in devs) + "]"
        lines = []
        for d in devs:
            first = True
            for k, v in d.items():
                val = f'"{v}"' if how == "block_quoted" and k == "path" else (f"0o{v:o}" if k == "file_mode" and v != 438 and how == "block_comments" else str(v))
                lines.append(("- " if first else "  ") + f"{k}: {val}" + ("   # note" if how == "block_comments" else ""))
                first = False
            if how == "block_comments":
                lines.append("# between items")
        return "\n".join(lines) + "\n"

    @settings(max_examples=150, deadline=None, suppress_health_check=[HealthCheck.too_slow])
    @given(st.lists(dev, min_size=1, max_size=4), style)
    def check(devs, how):
        text = render(devs, how)
        if how == "block_comments":                    # 0o666 is YAML 1.2; PyYAML (1.1) would read it as a string: compare against the source data instead
            want = [d for i, d in enumerate(devs) if d["path"] not in [x["path"] for x in devs[:i]]]
        else:
            want = nri.get_devices("c", {KEY + "c": text})
        r = subprocess.run([exe, "--parse-annotation"], input=text.encode(), capture_output=True, timeout=20)
        assert r.returncode == 0, (text, r.stdout)
        got = [l.split(" ") for l in r.stdout.decode().splitlines()]
        assert got == [[d["path"], str(int(d.get("file_mode") or 0)), str(int(d.get("uid") or 0)), str(int(d.get("gid") or 0))] for d in want], text
    check()
    for bad in ("just a string", "- path: [unclosed", "[{path: /dev/x}", "key: value"):
        r = subprocess.run([exe, "--parse-annotation"], input=bad.encode(), capture_output=True, timeout=20)
        assert r.returncode == 1 and r.stdout.startswith(b"ERR"), bad


def test_python_injector_as_a_process(tmp_path):
    """`python -m container_engine_accelerators_b200.agent.nri --socket ...`: the entry point the Python image runs."""
    import subprocess, sys
    sock = str(tmp_path / "nri.sock")
    rt = testing.FakeNriRuntime(sock)
    fifo = tmp_path / "f"; os.mkfifo(fifo)
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    proc = subprocess.Popen([sys.executable, "-m", "container_engine_accelerators_b200.agent.nri", "--socket", sock, "--idx", "10"], cwd=root, stderr=subprocess.PIPE, text=True)
    try:
        reg = rt.wait_registered(timeout=30)
        assert (reg.plugin_name, reg.plugin_idx) == ("device_injector_nri", "10")
        rt.configure(); rt.synchronize()
        devs = rt.create_container("pod", "c", {KEY + "c": f'[{{"path": "{fifo}", "uid": 3}}]'}).adjust.linux.devices          # JSON-style annotation
        assert len(devs) == 1 and devs[0].type == "p" and devs[0].uid.value == 3
    finally:
        rt.close()
        try:
            proc.wait(10)
        except subprocess.TimeoutExpired:
            proc.kill()
    assert proc.returncode == 0, proc.stderr.read()
    missing = subprocess.run([sys.executable, "-m", "container_engine_accelerators_b200.agent.nri", "--socket", str(tmp_path / "absent.sock")], cwd=root, capture_output=True, text=True, timeout=60)
    assert missing.returncode == 1 and "plugin exited with error" in missing.stderr


def test_wire_constants_match_the_vendored_containerd_sources():
    """Our two NRI stacks are tested against our own fake runtime; pin the framing constants to containerd's sources so that
    agreement is not just self-consistency: ttrpc header 10 bytes / request 1 / response 2, mux header 8 bytes, conn ids 1 and 2,
    CREATE_CONTAINER = 4 (event mask bit 3). The vendored sources' values are recorded in tests/golden/reference_facts.json
    (oracle/reference_facts.py)."""
    import json
    with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_facts.json")) as f:
        wire = json.load(f)["containerd_wire"]
    assert (wire["ttrpc_header_bytes"], wire["ttrpc_request_type"], wire["ttrpc_response_type"]) == (10, 1, 2)
    assert (wire["mux_header_bytes"], wire["mux_max_payload_bytes"]) == (8, 1 << 24) and wire["mux_conn_id_big_endian_at_0"] is True
    assert (wire["plugin_service_conn"], wire["runtime_service_conn"]) == (1, 2)
    assert wire["create_container_event"] == 4
    assert (nri.PLUGIN_SERVICE_CONN, nri.RUNTIME_SERVICE_CONN) == (1, 2) and protos.NRI_EVENT_CREATE_CONTAINER == 1 << wire["create_container_event"] - 1
    native = open(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "agent", "native", "dp", "nri_injector.cc")).read()
    assert "kPluginConn = 1, kRuntimeConn = 2" in native and "kRequest = 1, kResponse = 2" in native and "pb::put_int(&resp, 2, 1 << 3)" in native
