"""PostStart / PreStop shims (deploy/app/ragengine/lifecycle/hooks.py) against a live service: the snapshot protocol the
controller's hooks rely on (pkg/ragengine/manifests/manifests.go:116-134; presets/ragengine/lifecycle/manager.py:126-326):
  <persist_dir>/systemsnapshots/<ts>_pod-<uid8>/<index>/..., metadata.json {index_names, version}, LATEST -> newest snapshot,
restore of every index of LATEST at start.  CPU: uvicorn in a thread over the oracle engine double."""
import importlib.util
import json
import os
import re
import socket
import threading
import time
import urllib.request
from datetime import datetime

from kaito_b200.embedding import HashingEmbedding
from kaito_b200.service import create_app, resolve_model_dir
from kaito_b200.vector_store import VectorStore

HOOKS = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "deploy", "app", "ragengine", "lifecycle", "hooks.py")


def _free_port():
    s = socket.socket(); s.bind(("127.0.0.1", 0)); p = s.getsockname()[1]; s.close()
    return p


def _serve(app, port):
    import uvicorn
    server = uvicorn.Server(uvicorn.Config(app, host="127.0.0.1", port=port, log_level="error"))
    th = threading.Thread(target=server.run, daemon=True)
    th.start()
    for _ in range(100):
        try:
            socket.create_connection(("127.0.0.1", port), timeout=0.2).close()
            return server, th
        except OSError:
            time.sleep(0.05)
    raise RuntimeError("server did not start")


def _load_hooks(monkeypatch, port, persist_dir, uid):
    monkeypatch.setenv("RAG_SERVICE_URL", f"http://127.0.0.1:{port}")
    monkeypatch.setenv("DEFAULT_VECTOR_DB_PERSIST_DIR", str(persist_dir))
    monkeypatch.setenv("POD_UID", uid)
    spec = importlib.util.spec_from_file_location(f"hooks_{uid}", HOOKS)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)          # BASE / ROOT are read from the environment at import, as in the pod
    return mod


def test_prestop_snapshot_and_poststart_restore(oracle, tmp_path, monkeypatch):
    from starlette.testclient import TestClient
    from tests.oracle_engine import OracleEngine
    port = _free_port()
    store = VectorStore(HashingEmbedding(64), OracleEngine(oracle))
    app = create_app(store, {"persist_dir": str(tmp_path), "llm_inference_url": None})
    server, th = _serve(app, port)
    try:
        c = TestClient(app)
        docs = [{"text": "First document about retrieval engines"}, {"text": "Second document about Kubernetes operators", "metadata": {"k": "v"}}]
        assert c.post("/index", json={"index_name": "idx_a", "documents": docs}).status_code == 200
        assert c.post("/index", json={"index_name": "idx b", "documents": docs[:1]}).status_code == 200     # name needing URL quoting
        before = c.post("/retrieve", json={"index_name": "idx_a", "query": "Kubernetes operators", "max_node_count": 2}).json()

        hooks = _load_hooks(monkeypatch, port, tmp_path, "0123456789abcdef")
        monkeypatch.setenv("POD_NAME", "ragengine-0")
        assert hooks.prestop() == 0
        root = tmp_path / "systemsnapshots"
        snaps = os.listdir(root)
        assert len(snaps) == 1 and re.fullmatch(r"\d{4}-\d\d-\d\dT\d\d-\d\d-\d\d_pod-01234567", snaps[0])      # manager.py:229-232
        meta = json.load(open(root / snaps[0] / "metadata.json"))
        assert set(meta) == {"timestamp", "pod_name", "pod_uid", "index_names", "version"}                         # manager.py:268-274
        assert meta["index_names"] == ["idx_a", "idx b"] and meta["version"] == 1 and meta["pod_uid"] == "01234567" and meta["pod_name"] == "ragengine-0"
        assert os.readlink(tmp_path / "LATEST") == os.path.join("systemsnapshots", snaps[0])                       # relative, at the base dir
        assert os.path.isfile(root / snaps[0] / "idx_a" / "docstore.json")

        # a fresh pod: empty service, PostStart restores every index named in LATEST/metadata.json
        for name in ("idx_a", "idx b"):
            assert c.delete(f"/indexes/{name}").status_code == 200
        assert c.get("/indexes").json() == []
        assert hooks.poststart() == 0
        assert sorted(c.get("/indexes").json()) == ["idx b", "idx_a"]
        after = c.post("/retrieve", json={"index_name": "idx_a", "query": "Kubernetes operators", "max_node_count": 2}).json()
        assert after == before
        assert c.get("/indexes/idx_a/documents").json()["total_items"] == 2

        # LATEST lost: PostStart falls back to the newest snapshot directory and recreates the link (manager.py:153-178)
        os.remove(tmp_path / "LATEST")
        assert c.delete("/indexes/idx_a").status_code == 200
        assert hooks.poststart() == 0 and "idx_a" in c.get("/indexes").json()
        assert os.readlink(tmp_path / "LATEST") == os.path.join("systemsnapshots", snaps[0])

        # retention: only the newest 5 snapshots are kept
        for i in range(6):
            os.makedirs(root / f"2000-01-0{i + 1}T00-00-00_pod-old{i}")
        time.sleep(1.1)                                    # snapshot names have one-second resolution
        assert hooks.prestop() == 0
        kept = sorted(os.listdir(root))
        assert len(kept) == 5 and os.path.realpath(tmp_path / "LATEST") == os.path.realpath(root / kept[-1])
    finally:
        server.should_exit = True
        th.join(timeout=5)


GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "lifecycle_reference.json")


def _replay(url, requests, snapshot):
    """send recorded requests (URLs as the reference's hooks sent them) and check each answer against the recording"""
    for r in requests:
        req = urllib.request.Request(url + r["url"].replace("{snapshot}", snapshot), method=r["method"],
                                     data=b"" if r["method"] == "POST" else None)
        with urllib.request.urlopen(req, timeout=30) as resp:
            assert (resp.status, json.loads(resp.read())) == (r["status"], json.loads(json.dumps(r["body"]).replace("{snapshot}", snapshot)))


def test_reference_lifecycle_manager_drives_this_service(oracle, tmp_path, monkeypatch):
    """Drop-in check against the reference's own PreStop/PostStart handlers (lifecycle/manager.py), replayed from
    tests/golden/lifecycle_reference.json (oracle/gen_golden_lifecycle.py ran them against this service): a snapshot laid
    out by the reference's PreStop restores under our PostStart, and the reference's PostStart requests restore a snapshot
    written by our PreStop."""
    from starlette.testclient import TestClient
    from tests.oracle_engine import OracleEngine
    gold = json.load(open(GOLD))
    pre = gold["prestop"]
    port = _free_port()
    url = f"http://127.0.0.1:{port}"
    app = create_app(VectorStore(HashingEmbedding(64), OracleEngine(oracle)), {"persist_dir": str(tmp_path), "llm_inference_url": None})
    server, th = _serve(app, port)
    try:
        monkeypatch.setenv("POD_UID", gold["pod_uid"])
        c = TestClient(app)
        assert c.post("/index", json={"index_name": "idx_a", "documents": gold["documents"]}).status_code == 200
        before = c.post("/retrieve", json={"index_name": "idx_a", "query": "retrieval engines", "max_node_count": 2}).json()
        # reference PreStop -> our PostStart
        name = pre["snapshot_name"].replace("{timestamp}", datetime.now().strftime(pre["snapshot_timestamp_format"]))
        snap = tmp_path / "systemsnapshots" / name
        snap.mkdir(parents=True)
        _replay(url, pre["requests"], str(snap))
        meta = dict(pre["metadata"], timestamp=datetime.now().isoformat())
        (snap / "metadata.json").write_text(json.dumps(meta, indent=2))
        os.symlink(pre["latest"].replace("{snapshot_name}", name), tmp_path / "LATEST")
        assert c.delete("/indexes/idx_a").status_code == 200
        hooks = _load_hooks(monkeypatch, port, tmp_path, gold["pod_uid"])
        assert hooks.poststart() == 0
        assert c.post("/retrieve", json={"index_name": "idx_a", "query": "retrieval engines", "max_node_count": 2}).json() == before
        # our PreStop -> reference PostStart: the layout its handler reads, then the requests it sends
        time.sleep(1.1)
        assert hooks.prestop() == 0
        latest = os.readlink(tmp_path / "LATEST")
        assert re.fullmatch(re.escape(pre["latest"]).replace(re.escape("{snapshot_name}"), r"\d{4}-\d\d-\d\dT\d\d-\d\d-\d\d_pod-")
                            + re.escape(pre["metadata"]["pod_uid"]), latest)
        ours = json.load(open(tmp_path / latest / "metadata.json"))
        assert set(ours) == set(pre["metadata"]) and ours["index_names"] == pre["metadata"]["index_names"]
        assert c.delete("/indexes/idx_a").status_code == 200
        _replay(url, gold["poststart"]["requests"], os.path.realpath(tmp_path / "LATEST"))
        assert c.get("/indexes").json() == ["idx_a"]
        assert c.post("/retrieve", json={"index_name": "idx_a", "query": "retrieval engines", "max_node_count": 2}).json() == before
        assert len(os.listdir(tmp_path / "systemsnapshots")) == 2
    finally:
        server.should_exit = True
        th.join(timeout=5)


def test_poststart_without_snapshot_is_a_noop(oracle, tmp_path, monkeypatch, capsys):
    from tests.oracle_engine import OracleEngine
    port = _free_port()
    app = create_app(VectorStore(HashingEmbedding(64), OracleEngine(oracle)), {"persist_dir": str(tmp_path), "llm_inference_url": None})
    server, th = _serve(app, port)
    try:
        hooks = _load_hooks(monkeypatch, port, tmp_path, "ffff")
        assert hooks.poststart() == 0
        assert "No previous snapshots found" in capsys.readouterr().out
        assert hooks.prestop() == 0                       # no indexes: the empty snapshot directory is removed again
        assert not os.path.lexists(tmp_path / "LATEST") and os.listdir(tmp_path / "systemsnapshots") == []
    finally:
        server.should_exit = True
        th.join(timeout=5)


def test_resolve_model_dir(tmp_path, monkeypatch):
    """service.resolve_model_dir: explicit KRAG_MODEL_DIR, MODEL_ID as a path, hub cache layout; None when nothing is local"""
    def snap(p):
        os.makedirs(p)
        for f in ("config.json", "vocab.txt"):
            open(os.path.join(p, f), "w").write("{}")
        return str(p)
    monkeypatch.delenv("KRAG_MODEL_DIR", raising=False)
    monkeypatch.setenv("HF_HOME", str(tmp_path / "hf"))
    assert resolve_model_dir("BAAI/bge-small-en-v1.5") is None
    hub = snap(tmp_path / "hf" / "hub" / "models--BAAI--bge-small-en-v1.5" / "snapshots" / "abc123")
    assert resolve_model_dir("BAAI/bge-small-en-v1.5") == hub
    local = snap(tmp_path / "mymodel")
    assert resolve_model_dir(local) == local
    monkeypatch.setenv("KRAG_MODEL_DIR", snap(tmp_path / "explicit"))
    assert resolve_model_dir("BAAI/bge-small-en-v1.5") == str(tmp_path / "explicit")


def test_deploy_tree_satisfies_the_controllers_pod_contract():
    """The literals the unmodified controller puts into the pod spec (pkg/ragengine/manifests/manifests.go:116-134, 146-279;
    pkg/ragengine/controllers/preset_rag.go:33-64, 186), stored in tests/golden/lifecycle_reference.json, resolve inside
    deploy/: hook script path and verbs, `python3 main.py` in the image WORKDIR, port and probe path, and the environment
    variables the hooks read."""
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    pod = json.load(open(GOLD))["pod_contract"]
    assert pod["poststart_command"] == ["python3", "/app/ragengine/lifecycle/hooks.py", "poststart"]
    hook_path = pod["poststart_command"][1]
    assert os.path.isfile(os.path.join(root, "deploy", hook_path.lstrip("/")))
    assert f"python3 {hook_path} prestop" in pod["prestop_command"][-1]
    hooks_src = open(os.path.join(root, "deploy", hook_path.lstrip("/"))).read()
    for verb in ("poststart", "prestop"):
        assert f'"{verb}"' in hooks_src
    assert pod["env"] == ["POD_NAME", "POD_UID", "DEFAULT_VECTOR_DB_PERSIST_DIR"]
    for env in pod["env"]:
        assert env in hooks_src
    assert pod["container_command"] == "python3 main.py" and os.path.isfile(os.path.join(root, "deploy", "app", "ragengine", "main.py"))
    dockerfile = open(os.path.join(root, "deploy", "Dockerfile")).read()
    assert "WORKDIR /app/ragengine" in dockerfile and "python3 main.py" in dockerfile and "EXPOSE 5000" in dockerfile
    port, probe = pod["port"], pod["probe_path"]
    svc = open(os.path.join(root, "kaito_b200", "service.py")).read()
    assert f"port={port}" in svc and f'@app.get("{probe}"' in svc
