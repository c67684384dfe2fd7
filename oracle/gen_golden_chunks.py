#!/usr/bin/env python
"""Generate tests/golden/chunker_ref.json and chunker_ref_run.json by running the REAL reference chunker.

Test infrastructure.  Run in the authoring container only (``/root/reference`` does not exist on the
GPU box):  ``python oracle/gen_golden_chunks.py``.  The output is committed; nothing at GPU-test time
reads ``/root/reference``.

Imported from the reference (by file path, read-only, no bytecode written, so ``routes/__init__`` -> Flask
is never touched):
  server/routes/knowledge_base/document_processor.py -> DocumentProcessor.process (:27-60) and through it
  _decode_text, _chunk_markdown (:124-177), _chunk_plaintext, _split_text (:183-285), _force_split (:305-337),
  _get_overlap; constants TARGET_CHUNK_SIZE / CHUNK_OVERLAP / MIN_CHUNK_SIZE (:14-16).

The chunker stays as it is in the reference (SURVEY.md 8 a9: CPU string work upstream of the encoder);
these fixtures characterise its output -- including the > 1500-character chunk it emits when one paragraph
exceeds the target before any chunk exists (SURVEY.md 4) -- and are what the GPU test feeds through
insert_chunks -> WordPiece -> encoder forward -> shard.
"""

from __future__ import annotations

import hashlib
import importlib.util
import json
import os
import sys

import numpy as np

REF_FILE = "/root/reference/server/routes/knowledge_base/document_processor.py"
HERE = os.path.dirname(os.path.abspath(__file__))
OUT = os.path.join(os.path.dirname(HERE), "tests", "golden", "chunker_ref.json")
RUN_OUT = os.path.join(os.path.dirname(HERE), "tests", "golden", "chunker_ref_run.json")

_WORDS = ("alert latency service restart payment database kafka consumer lag rollback deploy canary cpu memory "
          "disk pod node cluster ingress certificate expiry rotate credentials failover replica primary timeout "
          "retry circuit breaker queue backlog throughput error budget burn rate incident postmortem runbook "
          "mitigation escalation pager dashboard grafana prometheus trace span log index shard").split()


def load_reference_module():
    spec = importlib.util.spec_from_file_location("ref_document_processor", REF_FILE)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def _sentence(rng, n):
    return " ".join(rng.choice(_WORDS) for _ in range(n)).capitalize() + "."


def _paragraph(rng, chars):
    out = []
    while sum(len(s) + 1 for s in out) < chars:
        out.append(_sentence(rng, int(rng.integers(6, 16))))
    return " ".join(out)


def documents():
    """Seeded synthetic runbooks / postmortems covering the chunker's branches."""
    rng = np.random.default_rng(20260921)
    docs = []
    md = ["# Payments runbook", "", _paragraph(rng, 300), "", "## Latency alerts", "", _paragraph(rng, 900), "",
          _paragraph(rng, 800), "", "### Restart procedure", "", "- drain the node", "- restart the payment service",
          "- verify the canary", "", _paragraph(rng, 2600), "", "## Database failover", "", _paragraph(rng, 1200), "",
          "```", "kubectl rollout restart deploy/payments", "```", "", _paragraph(rng, 500)]
    docs.append({"name": "runbook.md", "file_type": "markdown", "text": "\n".join(md)})
    # one paragraph far above the target before any chunk exists (the 4 199-character case of SURVEY.md 4)
    docs.append({"name": "wall_of_text.txt", "file_type": "plaintext", "text": _paragraph(rng, 4150)})
    # a short lead-in (< MIN_CHUNK_SIZE) followed by one oversized paragraph: document_processor.py:266-267 glues
    # them into ONE chunk far above the target (kept as is -- the encoder side must cope with > 512 tokens)
    docs.append({"name": "oversized_chunk.txt", "file_type": "plaintext",
                 "text": "Overview of the outage.\n\n" + _paragraph(rng, 4150) + "\n\n" + _paragraph(rng, 600)})
    docs.append({"name": "short.md", "file_type": "markdown", "text": "# Title\n\nToo short to matter."})
    docs.append({"name": "no_breaks.txt", "file_type": "plaintext", "text": "x" * 5000})
    docs.append({"name": "postmortem.txt", "file_type": "plaintext",
                 "text": "\n\n".join(_paragraph(rng, int(rng.integers(200, 1400))) for _ in range(9))})
    docs.append({"name": "latin1.txt", "file_type": "plaintext", "encoding": "latin-1",
                 "text": "Café résumé naïve über. " + _paragraph(rng, 700)})
    docs.append({"name": "headings_only.md", "file_type": "markdown", "text": "# A\n\n## B\n\n### C\n"})
    docs.append({"name": "empty.txt", "file_type": "plaintext", "text": "   \n\n  "})
    return docs


def main():
    sys.dont_write_bytecode = True
    mod = load_reference_module()
    out = {"reference_file": "server/routes/knowledge_base/document_processor.py",
           "constants": {"TARGET_CHUNK_SIZE": mod.TARGET_CHUNK_SIZE, "CHUNK_OVERLAP": mod.CHUNK_OVERLAP,
                         "MIN_CHUNK_SIZE": mod.MIN_CHUNK_SIZE},
           "documents": []}
    for d in documents():
        raw = d["text"].encode(d.get("encoding", "utf-8"))
        proc = mod.DocumentProcessor("user-1", f"doc-{d['name']}", d["name"])
        chunks = proc.process(raw, d["file_type"])
        out["documents"].append({"name": d["name"], "file_type": d["file_type"], "encoding": d.get("encoding", "utf-8"),
                                 "text": d["text"], "chunks": chunks})
        lens = [len(c["content"]) for c in chunks]
        print(f"{d['name']:18s} {len(raw):6d} B -> {len(chunks):2d} chunks, lengths {lens}")
    with open(OUT, "w", encoding="utf-8") as f:
        json.dump(out, f, ensure_ascii=False, indent=1)
    print("wrote", OUT)
    record_run(mod)


def input_digest(d) -> str:
    """SHA-256 of what the chunker is given for one fixture document (text, encoding, file type)."""
    key = json.dumps([d["text"], d["encoding"], d["file_type"]], ensure_ascii=False).encode("utf-8")
    return hashlib.sha256(key).hexdigest()


def record_run(mod):
    """Re-run the chunker over the fixture as it was written and store what it returned, keyed by document with the
    digest of its input: tests/test_chunker_characterisation.py checks the fixture against this record, so the
    fixture stays pinned to the real chunker's output without the reference tree."""
    with open(OUT, encoding="utf-8") as f:
        gold = json.load(f)
    run = {"reference_file": gold["reference_file"], "documents": []}
    for d in gold["documents"]:
        chunks = mod.DocumentProcessor("user-1", f"doc-{d['name']}", d["name"]).process(d["text"].encode(d["encoding"]), d["file_type"])
        run["documents"].append({"name": d["name"], "input_sha256": input_digest(d), "chunks": chunks})
    with open(RUN_OUT, "w", encoding="utf-8") as f:
        json.dump(run, f, ensure_ascii=False, indent=1)
    print("wrote", RUN_OUT)


if __name__ == "__main__":
    main()
