"""KRAG_HTTP_WORKERS: a front-end worker process (kaito_b200/frontend.py) in front of the engine process -- /retrieve over the
RPC (kaito_b200/rpc.py), everything else reverse-proxied to the engine's FastAPI app.  Answers, error bodies and metrics must be
those of the single-process service (presets/ragengine/main.py:742-771)."""
import json
import os
import shutil
import socket
import tempfile
import threading
import time
import urllib.error
import urllib.request

import pytest

from kaito_b200 import frontend, vector_store as vs
from kaito_b200.embedding import HashingEmbedding
from kaito_b200.rpc import RetrieveRpcServer
from kaito_b200.service import RAG_MAX_TOP_K, create_app
from kaito_b200.vector_store import VectorStore


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


@pytest.fixture
def rpc_path():
    """unix-socket path in a fresh directory under /tmp: a socket path is limited to 107 bytes, which pytest's tmp_path
    exceeds when TMPDIR is deep"""
    d = tempfile.mkdtemp(prefix="krag-", dir="/tmp")
    yield os.path.join(d, "rpc.sock")
    shutil.rmtree(d, ignore_errors=True)


def _http(method, url, body=None):
    req = urllib.request.Request(url, None if body is None else json.dumps(body).encode(), {"Content-Type": "application/json"}, method=method)
    try:
        with urllib.request.urlopen(req, timeout=10) as r:
            return r.status, json.loads(r.read() or b"null") if "json" in r.headers.get("content-type", "") else r.read().decode()
    except urllib.error.HTTPError as e:
        return e.code, json.loads(e.read() or b"null")


def test_parse_retrieve_matches_the_request_model():
    ok = frontend.parse_retrieve
    assert ok(b'{"index_name":"a","query":"q"}', 300) == ("a", "q", 5, None)
    assert ok(b'{"index_name":"a","query":"q","max_node_count":7,"metadata_filter":{"k":1},"extra":true}', 300) == ("a", "q", 7, {"k": 1})
    for bad in (b'{', b'[]', b'{"query":"q"}', b'{"index_name":1,"query":"q"}', b'{"index_name":"a","query":"q","max_node_count":0}',
                b'{"index_name":"a","query":"q","max_node_count":301}', b'{"index_name":"a","query":"q","max_node_count":true}',
                b'{"index_name":"a","query":"q","max_node_count":"3"}', b'{"index_name":"a","query":"q","metadata_filter":[1]}'):
        assert ok(bad, 300) is None, bad


def test_worker_process_serves_retrieve_and_proxies_the_rest(oracle, tmp_path, rpc_path):
    import uvicorn
    from fastapi import HTTPException as FHE
    from tests.oracle_engine import OracleEngine
    store = VectorStore(HashingEmbedding(64), OracleEngine(oracle))
    app = create_app(store, {"persist_dir": str(tmp_path), "llm_inference_url": None})
    engine_port, public_port = _free_port(), _free_port()
    srv = uvicorn.Server(uvicorn.Config(app, host="127.0.0.1", port=engine_port, log_level="warning", access_log=False))
    th = threading.Thread(target=srv.run, daemon=True)
    th.start()
    while not srv.started:
        time.sleep(0.02)
    rpc = RetrieveRpcServer(app.state.batcher, app.state.observe_retrieve, (vs.HTTPException, FHE), path=rpc_path)
    procs = frontend.spawn(1, "127.0.0.1", public_port, f"127.0.0.1:{engine_port}", rpc.path, None, RAG_MAX_TOP_K)
    base = f"http://127.0.0.1:{public_port}"
    try:
        for _ in range(300):
            try:
                if _http("GET", base + "/health")[0] == 200:
                    break
            except Exception:
                time.sleep(0.05)
        else:
            pytest.fail("front-end worker did not come up")
        # proxied: /health, /index, /indexes, validation errors, /metrics
        assert _http("GET", base + "/health") == (200, {"status": "Healthy", "detail": None})
        docs = [{"text": f"document number {i} about topic {i % 7}", "metadata": {"bucket": i % 3}} for i in range(40)]
        st, out = _http("POST", base + "/index", {"index_name": "w", "documents": docs})
        assert st == 200 and len(out) == 40
        assert _http("GET", base + "/indexes") == (200, ["w"])
        assert _http("GET", base + "/indexes/w/documents?limit=2")[1]["count"] == 2
        assert _http("POST", base + "/retrieve", {"index_name": "w", "query": "q", "max_node_count": 0})[0] == 422
        assert _http("POST", base + "/retrieve", {"query": "q"})[0] == 422
        # RPC path: same answer as the store; per-request errors with the reference's bodies
        before = rpc.requests
        for q, k, flt in (("topic 3 document", 4, None), ("topic 5", 3, {"bucket": 1})):
            st, got = _http("POST", base + "/retrieve", {"index_name": "w", "query": q, "max_node_count": k, "metadata_filter": flt})
            want = store.retrieve("w", q, k, flt)
            for r in want["results"]:
                r.setdefault("dense_score", None); r.setdefault("sparse_score", None); r.setdefault("source", None)
            assert st == 200 and got == want
        assert _http("POST", base + "/retrieve", {"index_name": "nope", "query": "q"}) == (404, {"detail": "No such index: 'nope' exists."})
        assert _http("POST", base + "/retrieve", {"index_name": "w", "query": "  "}) == (400, {"detail": "Query string cannot be empty."})
        assert rpc.requests - before == 4
        # concurrent requests through the worker are coalesced by the engine
        b0, r0 = app.state.batcher.batches, app.state.batcher.requests
        res = [None] * 24
        def go(i):
            res[i] = _http("POST", base + "/retrieve", {"index_name": "w", "query": f"topic {i % 7}", "max_node_count": 3})
        ts = [threading.Thread(target=go, args=(i,)) for i in range(24)]
        for t in ts: t.start()
        for t in ts: t.join()
        assert all(r[0] == 200 and r[1]["count"] == 3 for r in res)
        assert app.state.batcher.requests - r0 == 24 and app.state.batcher.batches - b0 < 24
        st, metrics = _http("GET", base + "/metrics")
        assert st == 200 and 'rag_indexes_retrieve_requests_total{status="success"}' in metrics and 'rag_indexes_retrieve_requests_total{status="failure"}' in metrics
    finally:
        for p in procs:
            p.terminate()
        for p in procs:
            p.wait(timeout=10)
        rpc.close()
        srv.should_exit = True
        th.join(timeout=5)
        app.state.batcher.close()


def test_rpc_client_survives_an_engine_restart(oracle, rpc_path):
    """the worker's connection to the engine is re-established on the next request after it broke; requests in flight at the
    time fail with ConnectionError (the worker answers 503)"""
    import asyncio
    from fastapi import HTTPException as FHE
    from tests.oracle_engine import OracleEngine
    from kaito_b200.batcher import RetrieveBatcher
    from kaito_b200.rpc import RetrieveRpcClient
    store = VectorStore(HashingEmbedding(64), OracleEngine(oracle))
    store.index_documents("r", [{"text": f"alpha beta {i}"} for i in range(12)])
    seen = []

    def start():
        b = RetrieveBatcher(store, max_batch=16, max_wait_s=0.002)
        return b, RetrieveRpcServer(b, lambda status, seconds, out: seen.append(status), (vs.HTTPException, FHE), path=rpc_path)

    async def scenario():
        b, srv = start()
        cli = RetrieveRpcClient(rpc_path)
        st, body = await cli.retrieve("r", "alpha 3", 2, None)
        assert st == 200 and json.loads(body)["count"] == 2
        st, body = await cli.retrieve("nope", "q", 2, None)
        assert st == 404 and json.loads(body) == {"detail": "No such index: 'nope' exists."}
        srv.close(); b.close()
        await asyncio.sleep(0.1)
        with pytest.raises((ConnectionError, OSError)):
            await cli.retrieve("r", "alpha 3", 2, None)
        b, srv = start()
        st, body = await cli.retrieve("r", "alpha 4", 3, None)
        assert st == 200 and json.loads(body)["count"] == 3
        srv.close(); b.close()
    asyncio.run(scenario())
    assert seen.count("success") == 2 and seen.count("failure") == 1
