"""Generate tests/golden/lifecycle_reference.json: what the reference's lifecycle hooks do to this service, and the pod-spec
literals its controller uses.

  prestop / poststart: presets/ragengine/lifecycle/manager.py (prestop_handler / poststart_handler), executed unmodified
      against this service over the oracle engine double.  Recorded: every HTTP request it sends (method, URL as sent,
      status, JSON body), the snapshot directory name, metadata.json and the LATEST link.  Between the two runs this
      service's own hooks restore the reference's snapshot and write one of their own, which the reference then restores.
  pod_contract: the literals of pkg/ragengine/manifests/manifests.go and pkg/ragengine/controllers/preset_rag.go that
      deploy/ has to satisfy (hook commands, environment, container command, port, probe path).

Absolute paths are stored as placeholders: {snapshot} for the snapshot directory, {timestamp} for the time parts.
Run: python oracle/gen_golden_lifecycle.py <checkout of the kaito repository>"""
import importlib.util
import json
import os
import re
import shutil
import socket
import sys
import tempfile
import threading
import time
import types
from datetime import datetime

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
OUT = os.path.join(ROOT, "tests", "golden", "lifecycle_reference.json")
HOOKS = os.path.join(ROOT, "deploy", "app", "ragengine", "lifecycle", "hooks.py")
POD_UID = "feedfacecafe"
SNAP_TS = "%Y-%m-%dT%H-%M-%S"


def pod_contract(ref_root):
    man = open(os.path.join(ref_root, "pkg", "ragengine", "manifests", "manifests.go")).read()
    pre = open(os.path.join(ref_root, "pkg", "ragengine", "controllers", "preset_rag.go")).read()

    def command(hook):
        block = re.search(hook + r":\s*&corev1\.LifecycleHandler\{.*?Command:\s*\[\]string\{(.*?)\}", man, re.S).group(1)
        return re.findall(r'"((?:[^"\\]|\\.)*)"', block)
    env = [e for e in ("POD_NAME", "POD_UID", "DEFAULT_VECTOR_DB_PERSIST_DIR") if re.search(r'Name:\s+"' + e + '"', man)]
    return {"poststart_command": command("PostStart"), "prestop_command": command("PreStop"), "env": env,
            "container_command": re.search(r'utils\.ShellCmd\("([^"]+)"\)', pre).group(1),
            "port": int(re.search(r"PortInferenceServer\s*=\s*(\d+)", pre).group(1)),
            "probe_path": re.search(r'ProbePath\s*=\s*"([^"]+)"', pre).group(1)}


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def hooks_traffic(ref_root):
    import requests
    import uvicorn
    from starlette.testclient import TestClient
    from kaito_b200.embedding import HashingEmbedding
    from kaito_b200.service import create_app
    from kaito_b200.vector_store import VectorStore
    from oracle import oracle as o
    from tests.oracle_engine import OracleEngine

    o.build()
    base = tempfile.mkdtemp(prefix="krag-lifecycle-")
    port = _free_port()
    url = f"http://127.0.0.1:{port}"
    app = create_app(VectorStore(HashingEmbedding(64), OracleEngine(o)), {"persist_dir": base, "llm_inference_url": None})
    server = uvicorn.Server(uvicorn.Config(app, host="127.0.0.1", port=port, log_level="error"))
    th = threading.Thread(target=server.run, daemon=True)
    th.start()
    while not server.started:
        time.sleep(0.02)

    spec = importlib.util.spec_from_file_location("ref_lifecycle_manager", os.path.join(ref_root, "presets", "ragengine", "lifecycle", "manager.py"))
    ref = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(ref)
    ref.wait_for_service.__defaults__ = (url + "/indexes", 60)
    for fn in (ref.get_indexes, ref.load_index, ref.persist_index):
        fn.__defaults__ = (url,)
    ref.time = types.SimpleNamespace(sleep=lambda s: None, time=time.time)       # its 0.5 s rate limiting
    log = []

    def recorded(method):
        def call(u, **kw):
            r = getattr(requests, method)(u, **kw)
            log.append({"method": r.request.method, "url": r.request.url[len(url):], "status": r.status_code, "body": r.json()})
            return r
        return call
    ref.requests = types.SimpleNamespace(get=recorded("get"), post=recorded("post"))

    def placeholders(obj, snap_dir):
        if isinstance(obj, str):
            return obj.replace(snap_dir, "{snapshot}")
        if isinstance(obj, list):
            return [placeholders(x, snap_dir) for x in obj]
        if isinstance(obj, dict):
            return {k: placeholders(v, snap_dir) for k, v in obj.items()}
        return obj

    os.environ["POD_UID"] = POD_UID
    os.environ.pop("POD_NAME", None)
    os.environ.update(RAG_SERVICE_URL=url, DEFAULT_VECTOR_DB_PERSIST_DIR=base)
    hspec = importlib.util.spec_from_file_location("hooks", HOOKS)
    hooks = importlib.util.module_from_spec(hspec)
    hspec.loader.exec_module(hooks)
    try:
        c = TestClient(app)
        docs = [{"text": "First document about retrieval engines"}, {"text": "Second document about Kubernetes operators"}]
        assert c.post("/index", json={"index_name": "idx_a", "documents": docs}).status_code == 200
        before = c.post("/retrieve", json={"index_name": "idx_a", "query": "retrieval engines", "max_node_count": 2}).json()

        # the reference's PreStop writes a snapshot of this service ...
        assert ref.prestop_handler(base) == 0
        (name,) = os.listdir(os.path.join(base, "systemsnapshots"))
        snap_dir = os.path.join(os.path.realpath(base), "systemsnapshots", name)
        ts = name.split("_pod-")[0]
        datetime.strptime(ts, SNAP_TS)
        meta = json.load(open(os.path.join(snap_dir, "metadata.json")))
        datetime.fromisoformat(meta["timestamp"])
        prestop = {"snapshot_name": name.replace(ts, "{timestamp}"), "snapshot_timestamp_format": SNAP_TS,
                   "requests": placeholders(log, snap_dir), "metadata": dict(meta, timestamp="{timestamp}"),
                   "latest": os.readlink(os.path.join(base, "LATEST")).replace(name, "{snapshot_name}")}
        # ... which this service's PostStart restores
        assert c.delete("/indexes/idx_a").status_code == 200
        assert hooks.poststart() == 0
        assert c.post("/retrieve", json={"index_name": "idx_a", "query": "retrieval engines", "max_node_count": 2}).json() == before

        # this service's PreStop writes a snapshot, the reference's PostStart restores it
        time.sleep(1.1)                                   # snapshot names have one-second resolution
        assert hooks.prestop() == 0
        assert c.delete("/indexes/idx_a").status_code == 200
        del log[:]
        assert ref.poststart_handler(base) == 0
        assert c.get("/indexes").json() == ["idx_a"]
        assert c.post("/retrieve", json={"index_name": "idx_a", "query": "retrieval engines", "max_node_count": 2}).json() == before
        poststart = {"requests": placeholders(log, os.path.realpath(os.path.join(base, "LATEST")))}
    finally:
        server.should_exit = True
        th.join(timeout=5)
        app.state.batcher.close()
        shutil.rmtree(base, ignore_errors=True)
    return {"pod_uid": POD_UID, "documents": docs, "prestop": prestop, "poststart": poststart}


def main():
    doc = {"meta": {"source": "presets/ragengine/lifecycle/manager.py executed unmodified against this service; literals of "
                              "pkg/ragengine/manifests/manifests.go and pkg/ragengine/controllers/preset_rag.go",
                    "generator": "oracle/gen_golden_lifecycle.py"},
           "pod_contract": pod_contract(sys.argv[1]), **hooks_traffic(sys.argv[1])}
    json.dump(doc, open(OUT, "w"), indent=1, sort_keys=True)
    print(json.dumps(doc, indent=1))


if __name__ == "__main__":
    main()
