"""CPU-side checks: the C-ABI library loads and exports every declared symbol, the host
featuriser / fingerprint mirror / synthetic generator agree with the reference-derived goldens,
and the product refuses to run without a GPU instead of falling back."""
import ctypes
import re
from pathlib import Path

import numpy as np
import pytest

from oracle import tfidf_oracle as O

REPO = Path(__file__).resolve().parent.parent


def test_library_exports_every_declared_symbol(built_lib):
    from kakveda_b200 import _capi

    header = (REPO / "include" / "kakveda_b200.h").read_text()
    declared = set(re.findall(r"\b(kv_[a-z0-9_]+)\s*\(", header))
    assert declared, "no prototypes parsed"
    lib = ctypes.CDLL(str(built_lib))
    for name in sorted(declared):
        assert hasattr(lib, name), f"{name} declared in include/kakveda_b200.h but not exported"
    assert declared == set(_capi.SIGNATURES), declared ^ set(_capi.SIGNATURES)
    assert b"sm_100a" in _capi.load().kv_version()


def test_no_cpu_fallback(built_lib):
    import os
    import subprocess
    import sys

    # a child process that sees no device (CUDA_VISIBLE_DEVICES=""), so the check also runs where a GPU is present
    child = ("import pytest\n"
             "from kakveda_b200 import _capi\n"
             "from kakveda_b200.similarity import SimilarityEngine\n"
             "assert _capi.load().kv_device_count() == 0\n"
             "with pytest.raises(RuntimeError, match='no CUDA device'):\n"
             "    SimilarityEngine().score('alpha beta', ['alpha beta gamma'])\n")
    out = subprocess.run([sys.executable, "-c", child], cwd=REPO, env=dict(os.environ, CUDA_VISIBLE_DEVICES=""),
                         stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    assert out.returncode == 0, out.stdout
    # the product package must not import the oracle or scikit-learn
    for py in (REPO / "kakveda_b200").glob("*.py"):
        src = py.read_text()
        assert "import oracle" not in src and "from oracle" not in src, py
        assert "import sklearn" not in src and "from sklearn" not in src, py


def test_featurizer_matches_sklearn_analyzer(built_lib, golden):
    from kakveda_b200.similarity import Vocabulary
    from kakveda_b200 import synth

    edge = golden("edge_cases.json")
    docs = synth.corpus(500) + edge["corpus"] + edge["queries"] + ["\x1fweird start", "UPPER lower Upper"]
    v = Vocabulary()
    fb = v.featurize(docs, grow=True)
    assert fb.n == len(docs)
    id2s, s2id = {}, {}
    for i, d in enumerate(docs):
        toks = O.tokens(d)
        inter = [x for i, t in enumerate(toks) for x in ([t] + ([t + " " + toks[i + 1]] if i + 1 < len(toks) else []))]
        order = list(dict.fromkeys(inter))  # 1-grams and 2-grams interleaved in token order
        counts = O.features(d)
        ids = fb.ids[fb.indptr[i]:fb.indptr[i + 1]]
        tf = fb.tf[fb.indptr[i]:fb.indptr[i + 1]]
        assert len(ids) == len(order), (d, len(ids), len(order))
        for f, a, b in zip(order, ids, tf):
            assert counts[f] == b
            assert id2s.setdefault(int(a), f) == f and s2id.setdefault(f, int(a)) == int(a)
    assert len(v) == len(s2id)
    # queries: no growth, out-of-vocabulary mass reported as sum of tf^2
    q = v.featurize(["alpha zzzunseen zzzunseen beta", ""], grow=False)
    assert len(v) == len(s2id)
    feats = O.features("alpha zzzunseen zzzunseen beta")
    oov = sum(c * c for f, c in feats.items() if f not in s2id)
    assert q.oov[0] == oov and q.oov[1] == 0.0
    assert q.indptr[1] - q.indptr[0] == sum(1 for f in feats if f in s2id)
    # ids do not depend on the number of worker threads
    a = Vocabulary().featurize(docs, grow=True, n_threads=1)
    b = Vocabulary().featurize(docs, grow=True, n_threads=7)
    assert np.array_equal(a.ids, b.ids) and np.array_equal(a.tf, b.tf) and np.array_equal(a.indptr, b.indptr)


def test_featurizer_rejects_non_ascii_raw(built_lib):
    from kakveda_b200 import _capi
    from kakveda_b200.similarity import Vocabulary

    v = Vocabulary()
    data = "plain ascii".encode() + "café".encode("utf-8")
    off = np.array([0, 11, len(data)], dtype=np.int64)
    with pytest.raises(ValueError, match="non-ASCII"):
        v.featurize_packed(data, off, _capi.KV_TEXT_RAW_ASCII, grow=True)


def test_fingerprint_mirror(golden):
    from kakveda_b200 import fingerprint as fp

    g = golden("signature_text.json")
    for c in g["cases"]:
        env = {k: 1 for k in c["env_keys"]}
        assert fp.signature_text(c["prompt"], c["tools"], env) == c["signature_text"]
        assert fp.fingerprint(c["prompt"], c["tools"], env) == c["fingerprint"]
        assert fp.normalize_prompt(c["prompt"]) == c["normalized"]
        assert fp.fingerprint_u64(c["signature_text"]) == O.fingerprint64(c["signature_text"])


def test_synthetic_rows_have_signature_text_shape(built_lib):
    from kakveda_b200 import fingerprint as fp, synth

    rows = synth.corpus(3000)
    checked = 0
    for row in rows:
        parts = row.split(" | ")
        assert [p.split(":", 1)[0] for p in parts] == ["intent_tags", "prompt_hint", "tools", "env_keys"]
        hint = parts[1][len("prompt_hint:"):]
        assert len(hint) <= 80
        if len(hint) < 80:
            tools = [t for t in parts[2][len("tools:"):].split(",") if t]
            env = {k: 1 for k in parts[3][len("env_keys:"):].split(",") if k}
            assert fp.signature_text(hint, tools, env) == row
            checked += 1
    assert checked > 1000
    dup = len(rows) - len(set(rows))
    assert 0.2 * len(rows) < dup < 0.45 * len(rows)  # ~30 % version rows
    qs = synth.queries(400, 3000)
    hits = sum(q in set(rows) for q in qs)
    assert 150 < hits < 250  # ~half the queries repeat a stored failure
    # any range of a stream is reproducible
    assert synth.signatures(synth.CORPUS_SEED, 1000, 50) == rows[1000:1050]
    feats = [len(O.features(r)) for r in rows[:300]]
    assert 15 <= min(feats) and max(feats) <= 70


def test_gfkb_match_semantics(golden):
    """Handler logic (services/gfkb/app.py:88-100) with the oracle standing in for the engine."""
    from kakveda_b200 import gfkb

    class OracleEngine:
        def score(self, query, corpus):
            return O.score_sklearn(query, corpus)

    g = golden("fixture54.json")
    for case in g["match"]:
        got = gfkb.match_records(OracleEngine(), case["signature_text"], g["records"], case["failure_type"])
        assert got == case["matches"]
    assert gfkb.match_records(OracleEngine(), "x", []) == []


def test_block_builder_roundtrip(tmp_path):
    """Host-side scan-layout construction (kakveda_b200/csrc/block_builder.cuh): decoding the column blocks gives back
    every row, the block invariants hold, the threaded build equals the sequential one, and the fixed-point row sums
    agree with float64 (tests/cpp/block_builder_check.cu; host code only, nvcc is just the compiler)."""
    import shutil
    import subprocess

    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    exe = tmp_path / "block_builder_check"
    src = REPO / "tests" / "cpp" / "block_builder_check.cu"
    subprocess.run([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-O2", "-std=c++17", "--expt-relaxed-constexpr",
                    "-Xcompiler", "-pthread", "-w", "-o", str(exe), str(src)],
                   check=True, stdout=subprocess.PIPE, stderr=subprocess.STDOUT)
    out = subprocess.run([str(exe)], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    assert out.returncode == 0, out.stdout
    assert "all block-builder cases passed" in out.stdout
