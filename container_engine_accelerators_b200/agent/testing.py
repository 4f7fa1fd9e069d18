"""Conformance fixtures: a stub kubelet (Registration gRPC server on <dir>/kubelet.sock) and builders for fake
/dev, /proc and /sys trees — the reference's test techniques (pkg/gpu/nvidia/beta_plugin_test.go:36-70 KubeletStub;
pkg/gpu/nvidia/mig/mig_test.go:55-83 fake capability files; manager_test.go:223-310 fake numa_node files) as a reusable,
language-neutral harness: anything that speaks v1beta1 over a Unix socket can be driven by it (SURVEY §7.0).
"""
from __future__ import annotations

import os
import tempfile
import threading
from concurrent import futures
from pathlib import Path

import grpc

from . import protos
from .protos import deviceplugin as pb

# A Unix socket's address holds at most 107 bytes, and the fakes and plugins bind theirs inside temporary directories (the longest
# name used is "device-plugins/nvidiaGPU-conformance.sock"). A directory path no longer than SOCKET_DIR_MAX leaves room for it.
SOCKET_DIR_MAX = 64


def socket_tmp_root() -> str:
    """Where to create temporary directories that will hold Unix sockets: the usual temporary directory when its path takes at most half
    of SOCKET_DIR_MAX (the rest is for the directory made inside it), otherwise /tmp."""
    base = tempfile.gettempdir()
    return base if len(base) <= SOCKET_DIR_MAX // 2 else "/tmp"


class KubeletStub:
    """Records every RegisterRequest; `wait_registration()` blocks until one arrives."""

    def __init__(self, plugin_dir: str, socket_name: str = "kubelet.sock"):
        self.socket_path = os.path.join(plugin_dir, socket_name)
        self.requests: list = []
        self._event = threading.Event()
        self._server = None

    def _register(self, request, context):
        self.requests.append(request)
        self._event.set()
        return pb.Empty()

    def start(self) -> "KubeletStub":
        try:
            os.unlink(self.socket_path)         # grpc may remove it itself while shutting down
        except FileNotFoundError:
            pass
        self._server = grpc.server(futures.ThreadPoolExecutor(max_workers=2))
        handler = grpc.method_handlers_generic_handler(protos.REGISTRATION_SERVICE, {
            "Register": grpc.unary_unary_rpc_method_handler(self._register, pb.RegisterRequest.FromString, pb.Empty.SerializeToString)})
        self._server.add_generic_rpc_handlers((handler,))
        self._server.add_insecure_port(f"unix:{self.socket_path}")
        self._server.start()
        return self

    def wait_registration(self, timeout: float = 10.0):
        if not self._event.wait(timeout):
            raise TimeoutError("plugin did not register with the stub kubelet")
        self._event.clear()
        return self.requests[-1]

    def stop(self) -> None:
        if self._server:
            self._server.stop(grace=0.5).wait()      # let a Register call that is being answered finish: the caller treats a failed registration as fatal
            self._server = None
        try:
            os.unlink(self.socket_path)         # grpc may remove it itself while shutting down
        except FileNotFoundError:
            pass


def make_fake_dev(root: str, gpus: int = 2, with_optional: bool = True) -> str:
    """<root>/dev with nvidiactl, nvidia-uvm, [nvidia-uvm-tools, nvidia-modeset] and nvidia0..N-1 as empty files."""
    dev = Path(root) / "dev"
    dev.mkdir(parents=True, exist_ok=True)
    names = ["nvidiactl", "nvidia-uvm"] + (["nvidia-uvm-tools", "nvidia-modeset"] if with_optional else [])
    for n in names + [f"nvidia{i}" for i in range(gpus)]:
        (dev / n).touch()
    return str(dev)


def add_fake_gpu(dev_dir: str, index: int) -> None:
    (Path(dev_dir) / f"nvidia{index}").touch()


def make_fake_mig(root: str, dev_dir: str, gpus: int, partitions_per_gpu: int) -> str:
    """<root>/proc/driver/nvidia/capabilities/gpu<N>/mig/gi<M>/{access,ci0/access} + /dev/nvidia-caps/nvidia-cap<minor>."""
    proc = Path(root) / "proc"
    caps = Path(dev_dir) / "nvidia-caps"
    caps.mkdir(parents=True, exist_ok=True)
    minor = 10
    for g in range(gpus):
        base = proc / "driver/nvidia/capabilities" / f"gpu{g}" / "mig"
        for p in range(partitions_per_gpu):
            gi = base / f"gi{p + 1}"
            (gi / "ci0").mkdir(parents=True, exist_ok=True)
            (gi / "access").write_text(f"DeviceFileMinor: {minor}\nDeviceFileMode: 292\n")
            (caps / f"nvidia-cap{minor}").touch(); minor += 1
            (gi / "ci0" / "access").write_text(f"DeviceFileMinor: {minor}\nDeviceFileMode: 292\n")
            (caps / f"nvidia-cap{minor}").touch(); minor += 1
    (proc / "driver/nvidia/capabilities" / "mig").mkdir(parents=True, exist_ok=True)   # non-gpu entry must be skipped
    return str(proc)


def make_fake_pci(root: str, bus_id: str, numa_node: int) -> str:
    pci = Path(root) / "sys/bus/pci/devices"
    d = pci / bus_id
    d.mkdir(parents=True, exist_ok=True)
    (d / "numa_node").write_text(f"{numa_node}\n")
    return str(pci)


# ------------------------------------------------------------------------------------------------- fake kube-apiserver
import json as _json
import re as _re
from http.server import BaseHTTPRequestHandler, ThreadingHTTPServer
from urllib.parse import parse_qs, urlparse


class FakeKubeApi:
    """In-process kube-apiserver double (the role of client-go's fake clientset in the reference's tests,
    health_checker_test.go:235,315-338): nodes, pods, events; `fail_next_gets` injects transient GET failures."""

    def __init__(self):
        self.nodes: dict = {}
        self.pods: dict = {}        # (ns, name) -> pod
        self.events: list = []
        self.requests: list = []    # (method, path, content-type)
        self.bearer_tokens: list = []
        self.fail_next_gets = 0
        self.conflicts = 0          # PUTs refused because their resourceVersion was stale (optimistic concurrency, like the real API server)
        self.stale_next_puts = 0    # make the next N node PUTs look stale: what a kubelet status write between our GET and PUT does
        self._srv = None
        self.url = ""

    def add_node(self, name: str, boot_id: str = "boot-1", labels=None, annotations=None, conditions=None, allocatable=None, taints=None) -> dict:
        node = {"apiVersion": "v1", "kind": "Node", "metadata": {"name": name, "uid": f"uid-{name}", "resourceVersion": "1", "labels": dict(labels or {}), "annotations": dict(annotations or {})},
                "spec": {"taints": list(taints or [])},
                "status": {"nodeInfo": {"bootID": boot_id}, "conditions": list(conditions or [{"type": "Ready", "status": "True"}]), "allocatable": dict(allocatable or {})}}
        self.nodes[name] = node
        return node

    def add_pod(self, pod: dict) -> None:
        self.pods[(pod["metadata"].get("namespace", "default"), pod["metadata"]["name"])] = pod

    def start(self, tls_cert: str = "", tls_key: str = "") -> "FakeKubeApi":
        """Plain HTTP by default; with a certificate/key pair the same server speaks HTTPS (TLS path of the native client)."""
        api = self

        class H(BaseHTTPRequestHandler):
            def log_message(self, *a):
                pass

            def _send(self, code, obj):
                body = _json.dumps(obj).encode()
                self.send_response(code); self.send_header("Content-Type", "application/json"); self.send_header("Content-Length", str(len(body))); self.end_headers()
                self.wfile.write(body)

            def _body(self):
                n = int(self.headers.get("Content-Length") or 0)
                return _json.loads(self.rfile.read(n) or b"{}")

            def _route(self, method):
                u = urlparse(self.path)
                q = parse_qs(u.query)
                api.requests.append((method, u.path, self.headers.get("Content-Type", "")))
                api.bearer_tokens.append(self.headers.get("Authorization", ""))
                m = _re.fullmatch(r"/api/v1/nodes/([^/]+)(/status)?", u.path)
                if m:
                    name, status = m.group(1), bool(m.group(2))
                    if method == "GET":
                        if api.fail_next_gets > 0:
                            api.fail_next_gets -= 1
                            return self._send(500, {"message": "injected failure"})
                        return self._send(200, api.nodes[name]) if name in api.nodes else self._send(404, {"message": "not found"})
                    if name not in api.nodes:
                        return self._send(404, {"message": "not found"})
                    body = self._body()
                    def bump():
                        meta = api.nodes[name].setdefault("metadata", {})
                        meta["resourceVersion"] = str(int(meta.get("resourceVersion", "0")) + 1)
                    if method == "PUT":
                        sent = (body.get("metadata") or {}).get("resourceVersion")
                        current = api.nodes[name].get("metadata", {}).get("resourceVersion")
                        if api.stale_next_puts > 0 or (sent is not None and current is not None and sent != current):
                            if api.stale_next_puts > 0:
                                api.stale_next_puts -= 1
                                bump()
                            api.conflicts += 1
                            return self._send(409, {"kind": "Status", "reason": "Conflict", "message": f"Operation cannot be fulfilled on nodes \"{name}\": the object has been modified"})
                        if status:
                            api.nodes[name]["status"] = body.get("status", {})
                        else:
                            body.setdefault("metadata", {})["resourceVersion"] = current
                            api.nodes[name] = body
                        bump()
                        return self._send(200, api.nodes[name])
                    if method == "PATCH":
                        ctype = self.headers.get("Content-Type", "")
                        meta = body.get("metadata", {})
                        if "apply-patch" in ctype and not q.get("fieldManager"):
                            return self._send(422, {"message": "fieldManager is required for apply"})
                        for key in ("labels", "annotations"):
                            for k, v in (meta.get(key) or {}).items():
                                if v is None:
                                    api.nodes[name]["metadata"].setdefault(key, {}).pop(k, None)
                                else:
                                    api.nodes[name]["metadata"].setdefault(key, {})[k] = v
                        bump()
                        return self._send(200, api.nodes[name])
                if u.path == "/api/v1/nodes" and method == "GET":
                    return self._send(200, {"items": list(api.nodes.values())})
                m = _re.fullmatch(r"/api/v1/namespaces/([^/]+)/events", u.path)
                if m and method == "POST":
                    ev = self._body(); api.events.append(ev)
                    return self._send(201, ev)
                m = _re.fullmatch(r"/api/v1(?:/namespaces/([^/]+))?/pods", u.path)
                if m and method == "GET":
                    items = [p for (ns, _), p in api.pods.items() if not m.group(1) or ns == m.group(1)]
                    for sel in (q.get("fieldSelector") or [""])[0].split(","):
                        if sel.startswith("status.phase="):
                            items = [p for p in items if p.get("status", {}).get("phase") == sel.split("=", 1)[1]]
                        if sel.startswith("spec.nodeName="):
                            items = [p for p in items if p.get("spec", {}).get("nodeName") == sel.split("=", 1)[1]]
                    return self._send(200, {"items": items})
                m = _re.fullmatch(r"/api/v1/namespaces/([^/]+)/pods/([^/]+)", u.path)
                if m:
                    key = (m.group(1), m.group(2))
                    if key not in api.pods:
                        return self._send(404, {"message": "not found"})
                    if method == "GET":
                        return self._send(200, api.pods[key])
                    if method == "PUT":
                        api.pods[key] = self._body()
                        return self._send(200, api.pods[key])
                return self._send(404, {"message": f"no route {method} {u.path}"})

            def do_GET(self): self._route("GET")
            def do_PUT(self): self._route("PUT")
            def do_POST(self): self._route("POST")
            def do_PATCH(self): self._route("PATCH")

        self._srv = ThreadingHTTPServer(("127.0.0.1", 0), H)
        scheme = "http"
        if tls_cert:
            import ssl
            ctx = ssl.SSLContext(ssl.PROTOCOL_TLS_SERVER)
            ctx.load_cert_chain(tls_cert, tls_key)
            self._srv.socket = ctx.wrap_socket(self._srv.socket, server_side=True)
            scheme = "https"
        self.url = f"{scheme}://127.0.0.1:{self._srv.server_address[1]}"
        threading.Thread(target=self._srv.serve_forever, daemon=True).start()
        return self

    def stop(self) -> None:
        if self._srv:
            self._srv.shutdown(); self._srv.server_close(); self._srv = None


def rbac_violations(cluster_role: dict, requests: list) -> list:
    """Which of the (method, path, content-type) requests a fake API server saw would a real one have refused under this ClusterRole?
    Keeps the generated RBAC manifests honest: every call an agent makes in the tests must be covered by the role it is deployed with."""
    verb_of = {"GET": "get", "PUT": "update", "PATCH": "patch", "POST": "create", "DELETE": "delete"}
    bad = []
    for method, path, _ in requests:
        parts = [p for p in path.split("/") if p]                      # api v1 [namespaces <ns>] <resource> [<name> [<subresource>]]
        rest = parts[2:]
        if rest[:1] == ["namespaces"] and len(rest) >= 3:
            rest = rest[2:]
        resource = rest[0] + ("/" + rest[2] if len(rest) >= 3 else "")
        verb = verb_of[method]
        if method == "GET" and len(rest) == 1:
            verb = "list"
        if not any(resource in r.get("resources", []) and (verb in r.get("verbs", []) or "*" in r.get("verbs", [])) and "" in r.get("apiGroups", [""]) for r in cluster_role.get("rules", [])):
            bad.append((verb, resource, path))
    return bad


def make_self_signed_cert(directory: str, ip: str = "127.0.0.1", dns: str = "localhost"):
    """(cert.pem, key.pem) for a throwaway CA-less server certificate with IP and DNS subject-alt-names."""
    import datetime
    import ipaddress
    from cryptography import x509
    from cryptography.hazmat.primitives import hashes, serialization
    from cryptography.hazmat.primitives.asymmetric import ec
    from cryptography.x509.oid import NameOID
    key = ec.generate_private_key(ec.SECP256R1())
    name = x509.Name([x509.NameAttribute(NameOID.COMMON_NAME, "fake-kube-apiserver")])
    now = datetime.datetime.now(datetime.timezone.utc)
    cert = (x509.CertificateBuilder().subject_name(name).issuer_name(name).public_key(key.public_key()).serial_number(x509.random_serial_number())
            .not_valid_before(now - datetime.timedelta(minutes=5)).not_valid_after(now + datetime.timedelta(days=1))
            .add_extension(x509.SubjectAlternativeName([x509.IPAddress(ipaddress.ip_address(ip)), x509.DNSName(dns)]), critical=False)
            .add_extension(x509.BasicConstraints(ca=True, path_length=None), critical=True)
            .sign(key, hashes.SHA256()))
    cert_path, key_path = os.path.join(directory, "cert.pem"), os.path.join(directory, "key.pem")
    with open(cert_path, "wb") as f:
        f.write(cert.public_bytes(serialization.Encoding.PEM))
    with open(key_path, "wb") as f:
        f.write(key.private_bytes(serialization.Encoding.PEM, serialization.PrivateFormat.TraditionalOpenSSL, serialization.NoEncryption()))
    return cert_path, key_path


# ------------------------------------------------------------------------------------------------- fake NRI runtime
class FakeNriRuntime:
    """containerd's side of NRI for tests: accepts one plugin on a Unix socket, serves Runtime.RegisterPlugin on mux
    conn 2 and drives Plugin.Configure / Synchronize / CreateContainer on mux conn 1."""

    def __init__(self, socket_path: str):
        import socket as _socket
        self.socket_path = socket_path
        self.registered = threading.Event()
        self.registration = None
        self._listener = _socket.socket(_socket.AF_UNIX, _socket.SOCK_STREAM)
        if os.path.exists(socket_path):
            os.unlink(socket_path)
        self._listener.bind(socket_path)
        self._listener.listen(1)
        self.client = None
        self.mux = None
        threading.Thread(target=self._accept, daemon=True).start()

    def _accept(self) -> None:
        from . import nri
        conn, _ = self._listener.accept()
        self.mux = nri.Mux(conn)

        def register(req):
            self.registration = req
            self.registered.set()
            return protos.nri.Empty()
        self.client = nri.TtrpcClient(nri.MuxStream(self.mux, nri.PLUGIN_SERVICE_CONN))
        server = nri.TtrpcServer(nri.MuxStream(self.mux, nri.RUNTIME_SERVICE_CONN), protos.NRI_RUNTIME_SERVICE, {"RegisterPlugin": (protos.nri.RegisterPluginRequest, register)})
        threading.Thread(target=server.serve, daemon=True).start()

    def wait_registered(self, timeout: float = 10.0):
        if not self.registered.wait(timeout):
            raise TimeoutError("plugin did not register")
        return self.registration

    def configure(self):
        return self.client.call(protos.NRI_PLUGIN_SERVICE, "Configure", protos.nri.ConfigureRequest(runtime_name="containerd", runtime_version="2.0"), protos.nri.ConfigureResponse)

    def synchronize(self):
        return self.client.call(protos.NRI_PLUGIN_SERVICE, "Synchronize", protos.nri.SynchronizeRequest(), protos.nri.SynchronizeResponse)

    def create_container(self, pod_name: str, ctr_name: str, annotations: dict, namespace: str = "default"):
        req = protos.nri.CreateContainerRequest()
        req.pod.name, req.pod.namespace = pod_name, namespace
        for k, v in annotations.items():
            req.pod.annotations[k] = v
        req.container.name = ctr_name
        return self.client.call(protos.NRI_PLUGIN_SERVICE, "CreateContainer", req, protos.nri.CreateContainerResponse)

    def close(self) -> None:
        if self.mux:
            self.mux.close()
        self._listener.close()
        try:
            os.unlink(self.socket_path)         # grpc may remove it itself while shutting down
        except FileNotFoundError:
            pass
