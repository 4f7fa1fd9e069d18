#!/usr/bin/env python
"""Regenerate tests/golden/reference_facts.json from a checkout of the upstream container-engine-accelerators project.

    python oracle/reference_facts.py <path to the upstream checkout>

The tests compare the agent's wire schemas, MIG tables and contract constants with the values recorded in that file, so that the
comparison runs on any machine, with or without the upstream sources. Only the extracted values are stored, never the sources.
Run this again when the project is moved to a newer upstream revision, and review the diff of the JSON file.
"""
from __future__ import annotations

import json
import os
import re
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
OUT = os.path.join(ROOT, "tests", "golden", "reference_facts.json")

PROTOS = {
    "deviceplugin": "vendor/k8s.io/kubelet/pkg/apis/deviceplugin/v1beta1/api.proto",
    "podresources": "vendor/k8s.io/kubelet/pkg/apis/podresources/v1alpha1/api.proto",
    "nri": "vendor/github.com/containerd/nri/pkg/api/api.proto",
}


def parse_proto(path: str) -> dict:
    """Minimal .proto reader: {message: {field name: [number, type, repeated]}, "__enums__": [enum names]} — enough to compare names,
    numbers, types and cardinality."""
    text = re.sub(r"//[^\n]*", "", open(path).read())
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    text = re.sub(r"\[[^\]]*\]", "", text)                       # field options such as (gogoproto.customname)
    out, enums, stack = {}, set(), []
    for tok in re.finditer(r"message\s+(\w+)\s*\{|enum\s+(\w+)\s*\{|oneof\s+\w+\s*\{|\}|(repeated\s+|optional\s+)?(map\s*<\s*\w+\s*,\s*[\w.]+\s*>|[\w.]+)\s+(\w+)\s*=\s*(\d+)\s*;", text):
        if tok.group(1):
            stack.append(tok.group(1)); out.setdefault(tok.group(1), {})
        elif tok.group(2):
            stack.append("enum:" + tok.group(2)); enums.add(tok.group(2))
        elif tok.group(0).startswith("oneof"):
            stack.append("oneof")
        elif tok.group(0) == "}":
            if stack:
                stack.pop()
        else:
            owner = next((s for s in reversed(stack) if not s.startswith("enum:") and s != "oneof"), None)
            if owner is None or (stack and stack[-1].startswith("enum:")):
                continue
            typ = re.sub(r"\s+", "", tok.group(4))
            out[owner][tok.group(5)] = [int(tok.group(6)), typ.split(".")[-1] if not typ.startswith("map<") else typ, bool(tok.group(3) and tok.group(3).strip() == "repeated")]
    out["__enums__"] = sorted(enums)
    return out


def _one(pattern: str, text: str, what: str, flags=0) -> str:
    m = re.search(pattern, text, flags)
    if not m:
        raise SystemExit(f"reference_facts: {what} not found (pattern {pattern!r})")
    return m.group(1)


def contract_constants(ref: str) -> dict:
    """Names other systems key on: monitored Xids, condition / event strings, gauge names, annotation keys, resource name, topology
    labels, NRI annotation prefix."""
    read = lambda rel: open(os.path.join(ref, rel)).read()
    hc = read("pkg/gpu/nvidia/health_check/health_checker.go")
    vv = read("pkg/gpu/nvidia/version_visibility/version_visibility.go")
    sched = read("gke-topology-scheduler/schedule-daemon.py")
    inj = read("nri_device_injector/nri_device_injector.go")
    labels = dict(re.findall(r"^(\w+_LABEL) = '([^']+)'", sched, re.M))
    device_key = _one(r'\bdeviceKeyPrefix\s*=\s*"([^"]+)"', inj, "deviceKeyPrefix")
    ctr_key = _one(r'ctrDeviceKeyPrefix\s*=\s*deviceKeyPrefix\s*\+\s*"([^"]+)"', inj, "ctrDeviceKeyPrefix")
    return {
        "monitor_xids": [int(x) for x in _one(r"monitorCriticalXid := \[\]int\{([^}]*)\}", hc, "monitorCriticalXid").split(",")],
        "xid_condition_type": _one(r'XIDConditionType\s*=\s*"([^"]+)"', hc, "XIDConditionType"),
        "event_source": _one(r'eventSource\s*=\s*"([^"]+)"', hc, "eventSource"),
        "gauges": re.findall(r'Name: "(\w+)"', read("pkg/gpu/nvidia/metrics/metrics.go")),
        "driver_version_prefix": _one(r'DriverVersionPrefix\s*=\s*"([^"]+)"', vv, "DriverVersionPrefix"),
        "field_manager": _one(r'FieldManager:\s*"([^"]+)"', vv, "FieldManager"),
        "resource_name": _one(r'resourceName\s*=\s*"([^"]+)"', read("pkg/gpu/nvidia/manager.go"), "resourceName"),
        "topology_labels": {"prerelease": [labels["PRERELEASE_CLUSTER_LABEL"], labels["PRERELEASE_RACK_LABEL"], labels["PRERELEASE_HOST_LABEL"]],
                            "ga": [labels["CLUSTER_LABEL"], labels["RACK_LABEL"], labels["HOST_LABEL"]]},
        "nri_container_device_key_prefix": device_key + ctr_key,
    }


def mig_tables(ref: str) -> dict:
    """The two MIG tables: the partitioner's size -> profile id and size -> max count, and the plugin's size -> max count."""
    go = open(os.path.join(ref, "partition_gpu/partition_gpu.go")).read()
    ids = dict(re.findall(r'"(\d+g\.\d+gb)":\s*"(\d+)"', go[go.index("partitionSizeToProfileID"):go.index("partitionSizeMaxCount")]))
    counts = dict(re.findall(r'"(\d+g\.\d+gb)":\s*(\d+),', go[go.index("partitionSizeMaxCount"):]))
    plugin = dict(re.findall(r'"(\d+g\.\d+gb)":\s*(\d+),', open(os.path.join(ref, "pkg/gpu/nvidia/mig/mig.go")).read()))
    return {"partition_profile_ids": ids, "partition_max_counts": counts, "plugin_max_counts": plugin}


def containerd_wire(ref: str) -> dict:
    """NRI framing constants from the vendored containerd sources (ttrpc channel, NRI connection multiplexer, NRI event ids)."""
    base = os.path.join(ref, "vendor/github.com/containerd")
    chan = open(os.path.join(base, "ttrpc/channel.go")).read()
    mux = open(os.path.join(base, "nri/pkg/net/multiplex/mux.go")).read()
    ids = open(os.path.join(base, "nri/pkg/net/multiplex/ttrpc.go")).read()
    api = open(os.path.join(base, "nri/pkg/api/api.proto")).read()
    payload = re.search(r"maxPayloadSize\s*=\s*(\d+)\s*<<\s*(\d+)", mux)
    conn_ids = re.search(r"PluginServiceConn ConnID = iota \+ (\d+)\s*\n\s*//[^\n]*\n\s*RuntimeServiceConn\b", ids)
    if not payload or not conn_ids:
        raise SystemExit("reference_facts: multiplexer constants not found")
    return {
        "ttrpc_header_bytes": int(_one(r"messageHeaderLength\s*=\s*(\d+)", chan, "messageHeaderLength")),
        "ttrpc_request_type": int(_one(r"messageTypeRequest\s+messageType\s*=\s*(0x[0-9a-fA-F]+|\d+)", chan, "messageTypeRequest"), 0),
        "ttrpc_response_type": int(_one(r"messageTypeResponse\s+messageType\s*=\s*(0x[0-9a-fA-F]+|\d+)", chan, "messageTypeResponse"), 0),
        "mux_header_bytes": int(_one(r"headerLen\s*=\s*(\d+)", mux, "headerLen")),
        "mux_max_payload_bytes": int(payload.group(1)) << int(payload.group(2)),
        "mux_conn_id_big_endian_at_0": "binary.BigEndian.PutUint32(hdr[0:4], uint32(id))" in mux,
        "plugin_service_conn": int(conn_ids.group(1)),
        "runtime_service_conn": int(conn_ids.group(1)) + 1,
        "create_container_event": int(_one(r"CREATE_CONTAINER\s*=\s*(\d+)\s*;", api, "CREATE_CONTAINER")),
    }


def main(argv: list[str]) -> int:
    if len(argv) != 2 or not os.path.isdir(argv[1]):
        print(__doc__, file=sys.stderr)
        return 2
    ref = argv[1]
    facts = {"proto_schemas": {name: parse_proto(os.path.join(ref, rel)) for name, rel in PROTOS.items()},
             "proto_sources": PROTOS,
             "contract_constants": contract_constants(ref),
             "mig_tables": mig_tables(ref),
             "containerd_wire": containerd_wire(ref)}
    os.makedirs(os.path.dirname(OUT), exist_ok=True)
    with open(OUT, "w") as f:
        json.dump(facts, f, indent=1, sort_keys=True)
        f.write("\n")
    print(f"wrote {os.path.relpath(OUT, ROOT)}")
    return 0


if __name__ == "__main__":
    sys.exit(main(sys.argv))
