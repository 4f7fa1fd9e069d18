"""b200-partition-gpu and b200-persistenced against stub nvidia-smi / nvidia-persistenced scripts.
The reference tests only the pure parsers with canned `nvidia-smi mig -lgi` tables (partition_gpu/partition_gpu_test.go:68-171)
and swaps readFile (nvidia_persistenced_installer_test.go:25-98); here the real binaries run end to end against a scripted
nvidia-smi that records every invocation (SURVEY §4 take-away 3)."""
import json
import os
import stat
import subprocess

import pytest

LGI_HEADER = """+-------------------------------------------------------+
| GPU instances:                                        |
| GPU   Name             Profile  Instance   Placement  |
|                          ID       ID       Start:Size |
|=======================================================|
"""


def lgi_table(rows):
    body = "".join(f"|   {g}  MIG {name:<14}  {pid:>3}      {iid:>3}       {place:<9} |\n+-------------------------------------------------------+\n" for g, name, pid, iid, place in rows)
    return LGI_HEADER + body


def make_smi(tmp_path, mig_mode="Enabled", gpu_name="NVIDIA B200", lgi="No GPU instances found.\n", lgi_rc=0, fail=()):
    """A fake nvidia-smi: logs argv to calls.log, answers from files so tests can change state between calls."""
    d = tmp_path / "smi"
    d.mkdir(exist_ok=True)
    (d / "mig_mode").write_text(mig_mode + "\n")
    (d / "gpu_name").write_text(gpu_name + "\n")
    (d / "lgi").write_text(lgi)
    script = d / "nvidia-smi"
    script.write_text(f"""#!/bin/bash
D={d}
echo "$*" >> $D/calls.log
case "$*" in
  "--query-gpu=mig.mode.current --format=csv,noheader") cat $D/mig_mode ;;
  "--query-gpu=gpu_name --format=csv,noheader") cat $D/gpu_name ;;
  "-mig 1") echo Enabled > $D/mig_mode ;;
  "mig -lgi") cat $D/lgi; exit {lgi_rc} ;;
  "mig -dci") {"echo 'No compute instances found'; exit 6" if "dci-empty" in fail else "echo destroyed"} ;;
  "mig -dgi") {"echo boom; exit 1" if "dgi" in fail else "echo destroyed"} ;;
  "mig -cgi "*) {"echo nope; exit 1" if "cgi" in fail else "echo created"} ;;
  "mig -cci") echo created ;;
  "conf-compute -srs 1") {"echo 'No devices were found'; exit 1" if "nodev" in fail else "echo ok"} ;;
  "") echo status ;;
esac
""")
    script.chmod(script.stat().st_mode | stat.S_IEXEC)
    return d


def calls(d):
    p = d / "calls.log"
    return p.read_text().splitlines() if p.exists() else []


def run_partitioner(native_build, smi_dir, cfg_path, env=None):
    return subprocess.run([os.path.join(native_build, "b200-partition-gpu"), f"-nvidia-smi-path={smi_dir}/nvidia-smi", "-gpu-config", str(cfg_path)],
                          capture_output=True, text=True, timeout=30, env={**os.environ, **(env or {})})


def test_no_config_or_empty_size_is_a_noop(native_build, tmp_path):
    d = make_smi(tmp_path)
    assert run_partitioner(native_build, d, tmp_path / "absent.json").returncode == 0
    cfg = tmp_path / "gpu_config.json"
    cfg.write_text("{}")
    assert run_partitioner(native_build, d, cfg).returncode == 0
    cfg.write_text("not json at all")
    assert run_partitioner(native_build, d, cfg).returncode == 0
    assert calls(d) == []


def test_b200_seven_slices_from_scratch(native_build, tmp_path):
    """BASELINE config #5: 1g.23gb -> `mig -cgi 19 x7`."""
    d = make_smi(tmp_path, fail=("dci-empty",))
    cfg = tmp_path / "gpu_config.json"
    cfg.write_text(json.dumps({"GPUPartitionSize": "1g.23gb"}))
    r = run_partitioner(native_build, d, cfg)
    assert r.returncode == 0, r.stderr
    assert calls(d) == ["--query-gpu=mig.mode.current --format=csv,noheader", "mig -lgi", "mig -dci", "mig -dgi", "mig -cgi 19,19,19,19,19,19,19", "mig -cci", ""]


def test_already_in_desired_state_changes_nothing(native_build, tmp_path):
    rows = [(g, "1g.23gb", 19, 7 + i, f"{i}:1") for g in (0, 1) for i in range(7)]
    d = make_smi(tmp_path, lgi=lgi_table(rows))
    cfg = tmp_path / "gpu_config.json"
    cfg.write_text(json.dumps({"GPUPartitionSize": "1g.23gb"}))
    r = run_partitioner(native_build, d, cfg)
    assert r.returncode == 0, r.stderr
    assert calls(d) == ["--query-gpu=mig.mode.current --format=csv,noheader", "mig -lgi", ""]


@pytest.mark.parametrize("rows,why", [
    ([(0, "1g.23gb", 19, 7 + i, f"{i}:1") for i in range(6)], "too few instances"),
    ([(0, "1g.23gb", 19, 7, "0:1"), (0, "2g.45gb", 14, 5, "2:2")], "non-uniform profiles"),
    ([(0, "2g.45gb", 14, 3 + i, f"{2 * i}:2") for i in range(3)], "uniform but wrong profile"),
])
def test_mismatch_triggers_rebuild(native_build, tmp_path, rows, why):
    d = make_smi(tmp_path, lgi=lgi_table(rows))
    cfg = tmp_path / "gpu_config.json"
    cfg.write_text(json.dumps({"GPUPartitionSize": "3g.90gb"}))
    r = run_partitioner(native_build, d, cfg)
    assert r.returncode == 0, r.stderr
    assert "mig -cgi 9,9" in calls(d) and "mig -dgi" in calls(d), why


def test_blackwell_enables_mig_without_reboot_and_a100_reboots(native_build, tmp_path):
    cfg = tmp_path / "gpu_config.json"
    cfg.write_text(json.dumps({"GPUPartitionSize": "7g.180gb"}))
    d = make_smi(tmp_path, mig_mode="Disabled", gpu_name="NVIDIA B200")
    hook = tmp_path / "rebooted"
    r = run_partitioner(native_build, d, cfg, env={"B200_PARTITION_REBOOT_HOOK": str(hook)})
    assert r.returncode == 0 and not hook.exists()
    assert calls(d)[:3] == ["--query-gpu=mig.mode.current --format=csv,noheader", "--query-gpu=gpu_name --format=csv,noheader", "-mig 1"]
    assert "mig -cgi 0" in calls(d)
    (d / "calls.log").unlink()
    cfg.write_text(json.dumps({"GPUPartitionSize": "1g.5gb"}))
    d = make_smi(tmp_path, mig_mode="Disabled", gpu_name="NVIDIA A100-SXM4-40GB")
    r = run_partitioner(native_build, d, cfg, env={"B200_PARTITION_REBOOT_HOOK": str(hook)})
    assert r.returncode == 1 and hook.exists()
    assert calls(d)[-1] == "-mig 1"                      # nothing after the reboot request


def test_failures_exit_one(native_build, tmp_path):
    cfg = tmp_path / "gpu_config.json"
    cfg.write_text(json.dumps({"GPUPartitionSize": "9g.1tb"}))
    assert run_partitioner(native_build, make_smi(tmp_path), cfg).returncode == 1          # unknown size
    cfg.write_text(json.dumps({"GPUPartitionSize": "1g.23gb"}))
    assert run_partitioner(native_build, make_smi(tmp_path, fail=("dgi",)), cfg).returncode == 1
    assert run_partitioner(native_build, make_smi(tmp_path, fail=("cgi",)), cfg).returncode == 1
    assert run_partitioner(native_build, make_smi(tmp_path, mig_mode="garbage"), cfg).returncode == 1
    assert run_partitioner(native_build, tmp_path / "no-smi-here", cfg).returncode == 1


def test_partitioner_table_matches_plugin_table(native_build):
    from container_engine_accelerators_b200.agent import mig
    out = subprocess.run([os.path.join(native_build, "b200-partition-gpu"), "--print-table"], capture_output=True, text=True).stdout.split("\n")
    rows = {l.split()[0]: (int(l.split()[1]), int(l.split()[2])) for l in out if l.strip()}
    assert rows == {k: (v.profile_id, v.max_count) for k, v in mig.PROFILES.items()}


# ------------------------------------------------------------------------------------------------- persistenced
def make_prefix(tmp_path, smi_dir, persistenced_rc=0):
    prefix = tmp_path / "nvidia"
    (prefix / "bin").mkdir(parents=True, exist_ok=True)
    os.symlink(smi_dir / "nvidia-smi", prefix / "bin" / "nvidia-smi")
    p = prefix / "bin" / "nvidia-persistenced"
    p.write_text(f"#!/bin/bash\necho \"$*\" >> {tmp_path}/persistenced.log\nexit {persistenced_rc}\n")
    p.chmod(0o755)
    ldc = tmp_path / "ldconfig"
    ldc.write_text("#!/bin/bash\nexit 0\n"); ldc.chmod(0o755)
    return prefix


def run_persistenced(native_build, tmp_path, prefix, node_type=None, driver="570.124.06", machine=None, extra_env=None):
    cg = tmp_path / "confidential_node_type.txt"
    if node_type is not None:
        cg.write_bytes(node_type)
    ver = tmp_path / "version"
    ver.write_text(f"NVRM version: NVIDIA UNIX Open Kernel Module for x86_64  {driver}  Release Build\n")
    mt = tmp_path / "machine_type.txt"
    if machine is not None:
        mt.write_text(machine)
    env = {**os.environ, "B200_PERSISTENCED_PROC_VERSION": str(ver), "B200_PERSISTENCED_LDCONF": str(tmp_path / "nvidia.conf"), "B200_PERSISTENCED_LDCONFIG": str(tmp_path / "ldconfig"),
           "B200_PERSISTENCED_REBOOT_HOOK": str(tmp_path / "rebooted"), "B200_PERSISTENCED_POLL_MS": "10", **(extra_env or {})}
    return subprocess.run([os.path.join(native_build, "b200-persistenced"), "--oneshot", "-container-path", str(prefix), "-cgpu-config", str(cg), "-machine-type-file", str(mt),
                           "-ready-delay-ms=1"], capture_output=True, text=True, timeout=30, env=env)


@pytest.mark.parametrize("content,enabled", [(b"TDX\n\x00", True), (b" sev \r\n", True), (b"none", False), (None, False)])
def test_persistenced_enablement(native_build, tmp_path, content, enabled):
    d = make_smi(tmp_path)
    prefix = make_prefix(tmp_path, d)
    r = run_persistenced(native_build, tmp_path, prefix, content)
    assert r.returncode == 0, r.stderr
    log = tmp_path / "persistenced.log"
    assert log.exists() == enabled
    if enabled:
        assert log.read_text().strip() == f"--uvm-persistence-mode --nvidia-cfg-path={prefix}/lib64"
        assert calls(d) == ["conf-compute -srs 1"]
        assert (tmp_path / "nvidia.conf").read_text() == f"{prefix}/lib64"


def test_persistenced_old_driver_has_no_uvm_flag(native_build, tmp_path):
    d = make_smi(tmp_path)
    prefix = make_prefix(tmp_path, d)
    assert run_persistenced(native_build, tmp_path, prefix, b"tdx", driver="535.230.02").returncode == 0
    assert (tmp_path / "persistenced.log").read_text().strip() == f"--nvidia-cfg-path={prefix}/lib64"


def test_persistenced_reboots_when_no_devices(native_build, tmp_path):
    d = make_smi(tmp_path, fail=("nodev",))
    prefix = make_prefix(tmp_path, d)
    r = run_persistenced(native_build, tmp_path, prefix, b"tdx")
    assert r.returncode == 1 and (tmp_path / "rebooted").exists()


def test_gridd_only_on_g4(native_build, tmp_path):
    d = make_smi(tmp_path)
    prefix = make_prefix(tmp_path, d)
    root = tmp_path / "root"
    (root / "lib64").mkdir(parents=True)
    linker = root / "lib64" / "ld-linux-x86-64.so.2"
    linker.write_text(f"#!/bin/bash\necho \"$*\" >> {tmp_path}/gridd.log\n"); linker.chmod(0o755)
    (prefix / "bin" / "nvidia-gridd").write_text("")
    r = run_persistenced(native_build, tmp_path, prefix, None, machine="a4-highgpu-8g\n", extra_env={"ROOT_MOUNT_DIR": str(root)})
    assert r.returncode == 0 and not (tmp_path / "gridd.log").exists()
    r = run_persistenced(native_build, tmp_path, prefix, None, machine="g4-standard-12\n", extra_env={"ROOT_MOUNT_DIR": str(root)})
    assert r.returncode == 0
    assert (tmp_path / "gridd.log").read_text().strip() == f"--library-path {prefix}/gridd-libs:{root}/lib64:{root}/usr/lib64 {prefix}/bin/nvidia-gridd"


# ------------------------------------------------------------------------------------------------- native building blocks
def test_native_selftest_json_kube_hpack_protobuf(native_build):
    """agent/native/dp/selftest.cc: JSON reader/writer (escapes, int64 fidelity, depth bound), HTTP response parsing,
    HPACK against the RFC 7541 Appendix C vectors plus hostile input, protobuf varints and truncated messages."""
    r = subprocess.run([os.path.join(native_build, "b200-native-selftest")], capture_output=True, text=True, timeout=60)
    assert r.returncode == 0, r.stdout + r.stderr
    assert ", 0 failed" in r.stdout


def test_nvml_abi_header_matches_the_toolkit_header(tmp_path):
    """agent/native/nvml_abi.h restates enumerator values and struct layouts; pin them against NVIDIA's nvml.h when a CUDA
    toolkit is present (the native build itself never needs it)."""
    real = "/usr/local/cuda/include/nvml.h"
    if not os.path.exists(real):
        pytest.skip("no CUDA toolkit header to compare against")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    mine = open(os.path.join(root, "agent", "native", "nvml_abi.h")).read()
    import re
    enums = dict(re.findall(r"\b(NVML_[A-Z_]+) = (\d+)", mine))
    assert len(enums) >= 15
    checks = " && ".join(f"{k} == {v}" for k, v in enums.items())
    src = tmp_path / "abi.cc"
    src.write_text(f"""#include <nvml.h>
#include <cstddef>
static_assert({checks}, "enumerators");
static_assert(sizeof(nvmlPciInfo_t) == 68 && offsetof(nvmlPciInfo_t, domain) == 16 && offsetof(nvmlPciInfo_t, busId) == 36, "pci");
static_assert(sizeof(nvmlEventData_t) == 32 && offsetof(nvmlEventData_t, eventData) == 16 && offsetof(nvmlEventData_t, computeInstanceId) == 28, "event");
static_assert(sizeof(nvmlSample_t) == 16 && offsetof(nvmlSample_t, sampleValue) == 8 && sizeof(nvmlMemory_t) == 24 && offsetof(nvmlMemory_t, used) == 16, "sample/memory");
static_assert(nvmlEventTypeXidCriticalError == 8, "event type");
int main() {{ return 0; }}
""")
    r = subprocess.run(["g++", "-std=c++17", "-fsyntax-only", "-I/usr/local/cuda/include", str(src)], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr


def test_native_json_agrees_with_python_on_generated_documents(native_build):
    """Property test: any JSON document Python can produce survives the C++ reader/writer with the same meaning (the Node objects
    the health checker rewrites go through exactly this path)."""
    from hypothesis import given, settings, strategies as st, HealthCheck
    exe = os.path.join(native_build, "b200-native-selftest")
    leaves = st.one_of(st.none(), st.booleans(), st.integers(min_value=-(2 ** 63), max_value=2 ** 63 - 1), st.floats(allow_nan=False, allow_infinity=False),
                       st.text(max_size=40))
    docs = st.recursive(leaves, lambda kids: st.one_of(st.lists(kids, max_size=6), st.dictionaries(st.text(max_size=12), kids, max_size=6)), max_leaves=40)

    @settings(max_examples=120, deadline=None, suppress_health_check=[HealthCheck.too_slow])
    @given(docs, st.booleans())
    def check(doc, ascii_only):
        text = json.dumps(doc, ensure_ascii=ascii_only)                 # ascii_only exercises \\uXXXX escapes and surrogate pairs
        r = subprocess.run([exe, "--json-roundtrip"], input=text.encode("utf-8", "surrogatepass"), capture_output=True, timeout=20)
        assert r.returncode == 0, r.stderr
        out = r.stdout.decode("utf-8", "surrogatepass")
        if out.startswith("ERR") and not text.startswith('"ERR'):
            raise AssertionError(f"rejected valid JSON: {text!r}: {out}")
        assert json.loads(out) == json.loads(text)
    check()
    for bad in ("{", "[1,]", '{"a" 1}', "tru", '"\\x"', "[1] 2", ""):
        r = subprocess.run([exe, "--json-roundtrip"], input=bad.encode(), capture_output=True, timeout=20)
        assert r.stdout.startswith(b"ERR"), (bad, r.stdout)


def test_mig_table_covers_every_size_the_reference_knows():
    """mig_profiles.inc is the single table behind the plugin and the partitioner; every (size -> profile id, max count) the reference
    lists in its two tables (partition_gpu.go:37-139, pkg/gpu/nvidia/mig/mig.go:35-82) must be there with the same numbers. The
    reference's tables are recorded in tests/golden/reference_facts.json (oracle/reference_facts.py)."""
    import re
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    with open(os.path.join(root, "tests", "golden", "reference_facts.json")) as f:
        tables = json.load(f)["mig_tables"]
    ids, counts, plugin_counts = tables["partition_profile_ids"], tables["partition_max_counts"], tables["plugin_max_counts"]
    ours = {m.group(1): (m.group(2), m.group(3)) for m in re.finditer(r'MIG_PROFILE\("([\w.]+)",\s*(\d+),\s*(\d+),', open(os.path.join(root, "agent", "native", "mig_profiles.inc")).read())}
    assert len(ids) >= 20 and set(ids) <= set(ours), sorted(set(ids) - set(ours))
    for size, pid in ids.items():
        assert ours[size] == (pid, counts[size]), (size, ours[size], pid, counts[size])
    for size, n in plugin_counts.items():
        assert ours[size][1] == n, (size, ours[size], n)
    assert ours["1g.23gb"] == ("19", "7") and ours["7g.180gb"] == ("0", "1")          # the B200 rows the north-star names
