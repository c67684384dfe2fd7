"""Characterisation of the reference chunker (server/routes/knowledge_base/document_processor.py:14-16, :183-337), which
stays as it is upstream of the encoder (SURVEY.md 8 a9).  tests/golden/chunker_ref.json was produced by running the REAL
class (oracle/gen_golden_chunks.py); here we pin the properties the ingest path relies on and check the fixture against
tests/golden/chunker_ref_run.json, the record of the real chunker re-run over the fixture as written."""

import json
import os

from oracle.gen_golden_chunks import input_digest

HERE = os.path.dirname(os.path.abspath(__file__))
GOLD = json.load(open(os.path.join(HERE, "golden", "chunker_ref.json"), encoding="utf-8"))
RUN = json.load(open(os.path.join(HERE, "golden", "chunker_ref_run.json"), encoding="utf-8"))


def test_constants_and_chunk_shape():
    assert GOLD["constants"] == {"TARGET_CHUNK_SIZE": 1500, "CHUNK_OVERLAP": 200, "MIN_CHUNK_SIZE": 100}     # :14-16
    for d in GOLD["documents"]:
        idx = [c["chunk_index"] for c in d["chunks"]]
        assert idx == list(range(len(idx)))                                     # insert_chunks keys on (user, doc, chunk_index)
        for c in d["chunks"]:
            assert set(c) == {"content", "heading_context", "chunk_index"} and c["content"] == c["content"].strip()


def test_known_behaviours_are_pinned():
    by = {d["name"]: d for d in GOLD["documents"]}
    assert by["empty.txt"]["chunks"] == [] and by["headings_only.md"]["chunks"] == []
    assert len(by["short.md"]["chunks"]) == 1 and by["short.md"]["chunks"][0]["heading_context"] == "Title"
    assert [len(c["content"]) for c in by["no_breaks.txt"]["chunks"]] == [1500, 1500, 1500, 1100]       # _force_split, 200 overlap
    over = [len(c["content"]) for c in by["oversized_chunk.txt"]["chunks"]]
    assert over[0] > 4000                  # one chunk far above the target (:266-267) -- kept, the encoder side copes
    md = by["runbook.md"]["chunks"]
    assert any(" > " in c["heading_context"] for c in md) and all(len(c["content"]) <= 1500 for c in md)
    assert by["latin1.txt"]["chunks"][0]["content"].startswith("Caf")             # decoded as latin-1 after utf-8 failed


def test_fixture_matches_the_real_reference_chunker():
    assert RUN["reference_file"] == GOLD["reference_file"]
    assert [r["name"] for r in RUN["documents"]] == [d["name"] for d in GOLD["documents"]]
    for d, r in zip(GOLD["documents"], RUN["documents"]):
        assert input_digest(d) == r["input_sha256"], d["name"]          # the chunker was given exactly this input
        assert r["chunks"] == d["chunks"], d["name"]
