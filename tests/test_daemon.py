"""Engine daemon + client shim: the reference's module API over a Unix socket (CPU, test doubles)."""

import shutil
import tempfile
import threading
from pathlib import Path

import pytest

from aurora_b200 import retriever as R
from aurora_b200.daemon import Client, serve
from tests.doubles import HashEmbedder, OracleIndex


@pytest.fixture()
def sock_dir():
    """A short directory for the daemon's sockets: a Unix socket path holds at most 107 bytes, and tmp_path under a
    deep TMPDIR or --basetemp can be longer than that."""
    base = tempfile.gettempdir()
    d = tempfile.mkdtemp(prefix="aur-", dir=base if len(base) <= 64 else "/tmp")
    yield Path(d)
    shutil.rmtree(d, ignore_errors=True)


@pytest.fixture()
def daemon(sock_dir):
    R.configure(encoder=HashEmbedder(64), capacity=1024, index_factory=lambda dim, cap: OracleIndex(dim, cap))
    path = str(sock_dir / "kb.sock")
    srv = serve(path, background=True)
    yield path
    srv.shutdown(); srv.close_all(final_save=False); srv.server_close()
    R.configure(factory=lambda: (_ for _ in ()).throw(RuntimeError("backend down")))


def _chunks(*texts):
    return [{"content": t, "heading_context": "", "chunk_index": i} for i, t in enumerate(texts)]


def test_client_roundtrip_and_concurrency(daemon):
    kb = Client(daemon)
    assert kb.health()["ready"]
    assert kb.insert_chunks("u", "d", "f.md", _chunks("redis failover steps", "postgres vacuum", "kafka lag")) == 3
    res = kb.search_knowledge_base("u", "redis failover", limit=2)
    assert res[0]["content"] == "redis failover steps" and set(res[0]) == {"content", "heading_context", "source_filename",
                                                                           "document_id", "chunk_index", "score"}
    assert kb.get_document_chunk_count("u", "d") == 3
    errs = []

    def worker(i):
        try:
            c = Client(daemon)
            for _ in range(20):
                assert c.search_knowledge_base("u", "kafka lag", limit=1)[0]["chunk_index"] == 2
        except Exception as e:      # pragma: no cover
            errs.append(e)

    ts = [threading.Thread(target=worker, args=(i,)) for i in range(8)]   # 2 gunicorn workers x 4 threads
    [t.start() for t in ts]; [t.join() for t in ts]
    assert not errs
    assert kb.delete_document_chunks("u", "d") == 3 and kb.search_knowledge_base("u", "redis") == []


def test_error_conventions_without_a_daemon(sock_dir):
    kb = Client(str(sock_dir / "nobody.sock"))
    assert kb.health()["ready"] is False
    assert kb.search_knowledge_base("u", "q") == []
    assert kb.delete_document_chunks("u", "d") == -1 and kb.delete_user_chunks("u") == -1
    assert kb.get_document_chunk_count("u", "d") == 0 and kb.delete_discovery_chunks("o") == 0
    assert kb.insert_chunks("u", "d", "f", []) == 0
    with pytest.raises(Exception):
        kb.insert_chunks("u", "d", "f", _chunks("x"))


def test_backend_failure_is_reported_not_swallowed_for_insert(daemon):
    R.configure(factory=lambda: (_ for _ in ()).throw(RuntimeError("backend down")))
    kb = Client(daemon)
    with pytest.raises(RuntimeError):
        kb.insert_chunks("u", "d", "f", _chunks("x"))          # Celery retries (weaviate_client.py:210-212)
    assert kb.search_knowledge_base("u", "q") == []


def test_bootstrap_requires_its_variables(monkeypatch):
    from aurora_b200 import bootstrap

    monkeypatch.delenv("AURORA_B200_ENCODER_WEIGHTS", raising=False)
    monkeypatch.delenv("AURORA_B200_VOCAB", raising=False)
    with pytest.raises(RuntimeError, match="AURORA_B200_ENCODER_WEIGHTS"):
        bootstrap.configure_from_env()
    with pytest.raises(ValueError):
        bootstrap._model_config("gpt-2")
    assert bootstrap._model_config("minilm-l6").hidden == 384


def test_socket_is_private_and_facade_and_learn_over_the_wire(sock_dir):
    import os
    import stat

    from aurora_b200 import incident_knowledge as K
    from aurora_b200.filters import Filter, HybridFusion

    R.configure(encoder=HashEmbedder(64), capacity=1024, index_factory=lambda dim, cap: OracleIndex(dim, cap))
    K.configure(encoder=HashEmbedder(64), capacity=256, index_factory=lambda dim, cap: OracleIndex(dim, cap), org_resolver=lambda u: "acme")
    path = str(sock_dir / "kb.sock")
    srv = serve(path, background=True, learn_module=K)
    try:
        assert stat.S_IMODE(os.stat(path).st_mode) == 0o600            # any process that can open it reads every tenant
        kb = Client(path)
        kb.insert_chunks("u", "discovery:20260101:ab", "gke-topology", _chunks("checkout depends on payments and redis"), org_id="o")
        kb.insert_chunks("u", "other", "notes.md", _chunks("checkout depends on payments and redis"), org_id="o")
        # chat/background/rca_prompt_builder.py:276-317, unchanged, against the daemon client
        _, collection = kb._get_weaviate_client()
        f = Filter.by_property("org_id").equal("o") & Filter.by_property("document_id").like("discovery:*")
        resp = collection.query.hybrid(query="checkout payments", limit=3, alpha=0.5, fusion_type=HybridFusion.RANKED,
                                       filters=f, return_metadata=["score"])
        assert [o.properties["source_filename"] for o in resp.objects] == ["gke-topology"] and resp.objects[0].metadata.score > 0
        assert kb.store_good_rca("alice", "inc-1", "fb-1", "Payments API latency high", "payments", "grafana", "critical",
                                 "pool exhausted", [{"content": "checked pool"}], [], org_id="acme") is True
        hits = kb.search_similar_good_rcas("bob", "Payments API latency high", "payments", "grafana", limit=2, min_score=0.2)
        assert hits and hits[0]["incident_id"] == "inc-1" and hits[0]["thoughts"] == [{"content": "checked pool"}]
        assert kb.delete_incident_knowledge("alice", "inc-1") is True and kb.delete_user_knowledge("alice") == 0
    finally:
        srv.shutdown(); srv.close_all(final_save=False); srv.server_close()
        R.configure(factory=lambda: (_ for _ in ()).throw(RuntimeError("backend down")))
        K.configure(factory=lambda: (_ for _ in ()).throw(RuntimeError("backend down")), org_resolver=lambda u: None)
    off = Client(str(sock_dir / "gone.sock"))
    assert off.store_good_rca("a", "i", "f", "t", "s", "g", "c", "s", [], []) is False and off.search_similar_good_rcas("a", "t", "s", "g") == []
    assert off.delete_incident_knowledge("a", "i") is False and off.delete_user_knowledge("a") == -1
    with pytest.raises(Exception):
        off._get_weaviate_client()


def test_concurrent_searches_are_coalesced_into_encoder_batches(sock_dir):
    """64 client threads, one query each at a time (the reference's call pattern): the daemon gathers them into a few
    encoder batches instead of 64 x N single-sequence forwards, and every caller still gets exactly its own answer."""
    emb = HashEmbedder(64)
    R.configure(encoder=emb, capacity=4096, index_factory=lambda dim, cap: OracleIndex(dim, cap))
    path = str(sock_dir / "kb.sock")
    srv = serve(path, background=True, coalesce_us=20000)
    try:
        kb = Client(path)
        for t in range(8):
            kb.insert_chunks(f"user{t}", f"doc{t}", "f.md", _chunks(*[f"topic{t} item{i} runbook entry" for i in range(6)]))
        calls_before = emb.calls
        errs, n_threads, per_thread = [], 64, 5

        def worker(i):
            try:
                c = Client(path)
                for j in range(per_thread):
                    t, it = i % 8, (i + j) % 6
                    res = c.search_knowledge_base(f"user{t}", f"topic{t} item{it} runbook entry", limit=1, alpha=1.0)
                    assert res[0]["document_id"] == f"doc{t}" and res[0]["chunk_index"] == it, (i, j, res)
            except Exception as e:      # pragma: no cover
                errs.append(e)

        ts = [threading.Thread(target=worker, args=(i,)) for i in range(n_threads)]
        [t.start() for t in ts]; [t.join() for t in ts]
        assert not errs, errs[0]
        encoder_calls = emb.calls - calls_before
        h = kb.health()
        assert h["coalesced_requests"] >= n_threads * per_thread
        assert encoder_calls * 4 <= n_threads * per_thread, (encoder_calls, h)        # far fewer encoder batches than requests
    finally:
        srv.shutdown(); srv.close_all(final_save=False); srv.server_close()
        R.configure(factory=lambda: (_ for _ in ()).throw(RuntimeError("backend down")))


def test_snapshot_policy_saves_and_restores(tmp_path, sock_dir):
    import os

    emb = HashEmbedder(64)
    R.configure(encoder=emb, capacity=1024, index_factory=lambda dim, cap: OracleIndex(dim, cap))
    snap = str(tmp_path / "snap")
    path = str(sock_dir / "kb.sock")
    srv = serve(path, background=True, snapshot_dir=snap, save_every=3, save_seconds=3600)
    try:
        kb = Client(path)
        kb.insert_chunks("u", "d", "f.md", _chunks("redis failover steps", "postgres vacuum", "kafka lag"))     # 3 mutations >= save_every
        deadline = __import__("time").time() + 10
        while not os.path.exists(os.path.join(snap, "meta.json")) and __import__("time").time() < deadline:
            __import__("time").sleep(0.1)
        assert os.path.exists(os.path.join(snap, "meta.json")) and kb.health()["unsaved_mutations"] == 0
        kb.insert_chunks("u", "d2", "g.md", _chunks("one more"))
        assert kb.health()["unsaved_mutations"] == 1
        assert kb.save()["saved"] is True and kb.health()["unsaved_mutations"] == 0          # on demand
        kb.delete_document_chunks("u", "d2")
    finally:
        srv.shutdown(); srv.close_all(final_save=True); srv.server_close()                       # the shutdown path saves too
    b = R.KnowledgeBase.load(snap, emb, capacity=1024, index_loader=lambda p, cap: OracleIndex.load(p, cap))
    assert b.count_where(lambda p: p["document_id"] == "d") == 3 and b.count_where(lambda p: p["document_id"] == "d2") == 0
    assert [n for n in os.listdir(snap) if n.startswith("shard.")] == [json_meta(snap)["shard"]]     # one generation on disk
    R.configure(factory=lambda: (_ for _ in ()).throw(RuntimeError("backend down")))


def json_meta(snap):
    import json
    import os

    return json.load(open(os.path.join(snap, "meta.json")))


def test_daemon_crash_between_snapshots_loses_nothing_acknowledged(tmp_path, sock_dir):
    """The deployment's durability story end to end (CPU doubles): a daemon with a snapshot directory and the mutation
    log takes a snapshot, acknowledges more inserts and a delete, and dies without saving; the next daemon restores
    the snapshot, replays the log and serves exactly what the first one had acknowledged."""
    import os

    emb = HashEmbedder(64)
    snap = str(tmp_path / "snap")
    os.makedirs(snap)

    def make():          # what bootstrap.configure_from_env installs, with test doubles
        if os.path.exists(os.path.join(snap, "meta.json")):
            kb = R.KnowledgeBase.load(snap, emb, capacity=1024, index_loader=lambda p, cap: OracleIndex.load(p, cap))
        else:
            kb = R.KnowledgeBase(emb, capacity=1024, index_factory=lambda dim, cap: OracleIndex(dim, cap))
        kb.attach_wal(os.path.join(snap, "mutations.log"))
        return kb

    R.configure(factory=make)
    path = str(sock_dir / "kb.sock")
    srv = serve(path, background=True, snapshot_dir=snap, save_every=10 ** 9, save_seconds=10 ** 9)
    try:
        kb = Client(path)
        assert kb.insert_chunks("u", "d1", "a.md", _chunks("redis failover steps", "postgres vacuum")) == 2
        assert kb.save()["saved"] is True
        assert kb.insert_chunks("u", "d2", "b.md", _chunks("kafka lag alert zx77", "nginx 502 runbook")) == 2
        assert kb.insert_chunks("u", "d1", "a.md", _chunks("redis failover steps, second edition")) == 1      # upsert
        assert kb.delete_document_chunks("u", "d2") == 2
        assert kb.insert_chunks("v", "d9", "z.md", _chunks("another tenant")) == 1
        want = kb.search_knowledge_base("u", "redis failover", limit=5)
        assert kb.health()["unsaved_mutations"] == 6
    finally:
        srv.shutdown(); srv.close_all(final_save=False); srv.server_close()          # "crash": no final snapshot
    R.configure(factory=make)                                                          # a new process would start like this
    path2 = str(sock_dir / "kb2.sock")
    srv2 = serve(path2, background=True, snapshot_dir=snap, save_every=10 ** 9, save_seconds=10 ** 9)
    try:
        kb2 = Client(path2)
        got = kb2.search_knowledge_base("u", "redis failover", limit=5)
        assert [(r["document_id"], r["chunk_index"], r["content"]) for r in got] == [(r["document_id"], r["chunk_index"], r["content"]) for r in want]
        assert got[0]["content"] == "redis failover steps, second edition"
        assert kb2.get_document_chunk_count("u", "d2") == 0 and kb2.get_document_chunk_count("v", "d9") == 1
        assert kb2.search_knowledge_base("u", "zx77", limit=3, alpha=0.0) == []       # the deleted document stays deleted
    finally:
        srv2.shutdown(); srv2.close_all(final_save=False); srv2.server_close()
    R.configure(factory=lambda: (_ for _ in ()).throw(RuntimeError("backend down")))
