"""Host logic of the drop-in services, on CPU (no GPU, no library compute calls): text
preparation, CSV rules of the build tool, C-ABI export list, loud failure without a GPU."""
import ctypes
import hashlib
import importlib
import json
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _golden(name):
    with open(os.path.join(ROOT, "tests", "golden", name), encoding="utf-8") as fh:
        return json.load(fh)


def test_library_exports_every_declared_symbol(native):
    """include/icdrag.h <-> libicdrag.so: every declared function is exported (no compute calls)."""
    hdr = open(os.path.join(ROOT, "include", "icdrag.h")).read()
    declared = sorted(set(re.findall(r"\b(icd_[a-z0-9_]+)\s*\(", hdr)))
    assert declared == sorted(native.SYMBOLS)
    assert os.path.exists(native.LIB_PATH), "run __graft_entry__.build() first"
    lib = ctypes.CDLL(native.LIB_PATH)
    for name in declared:
        assert hasattr(lib, name), name
    assert native.lib().icd_version() >= 100


def test_no_gpu_fails_loudly(native):
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    idx = importlib.import_module("rag-project-icd10_b200.engine.index")
    with pytest.raises(native.NativeError):
        idx.VectorIndex(768)
    enc = importlib.import_module("rag-project-icd10_b200.engine.encoder")
    with pytest.raises(native.NativeError):
        enc.EncoderEngine("does-not-matter")
    store = importlib.import_module("rag-project-icd10_b200.engine.store")
    with pytest.raises(native.NativeError):
        store.IcdStoreClient(uri="/tmp/x.db")


def test_product_never_imports_the_oracle():
    pkg_dir = os.path.join(ROOT, "rag-project-icd10_b200")
    for dirpath, _, files in os.walk(pkg_dir):
        for fn in files:
            if not fn.endswith(".py"):
                continue
            src = open(os.path.join(dirpath, fn), encoding="utf-8").read()
            hits = [l for l in src.splitlines() if re.match(r"\s*(from|import)\s+oracle\b", l)]
            assert not hits, (fn, hits)


def test_build_tool_records_match_reference():
    B = importlib.import_module("rag-project-icd10_b200.tools.build_database")
    g = _golden("records_golden.json")
    b = B.DatabaseBuilder.__new__(B.DatabaseBuilder)
    recs = b.load_csv_data(os.path.join(ROOT, "data", "ICD_10v601.csv"))
    assert len(recs) == g["count"]
    canon = json.dumps(recs, ensure_ascii=False, sort_keys=True).encode("utf-8")
    assert hashlib.sha256(canon).hexdigest() == g["sha256"]
    for n, want in g["batch_sizes"].items():
        assert b._calculate_optimal_batch_size(int(n)) == want


def test_embedding_service_text_rules_and_errors(monkeypatch):
    E = importlib.import_module("rag-project-icd10_b200.services.embedding_service")
    g = _golden("embedding_service_golden.json")

    class Rec:
        max_seq_length = 128
        calls = []

        def __init__(self, name, device=None):
            self.name, self.device = name, device

        def get_sentence_embedding_dimension(self):
            return 8

        def encode(self, texts, **kw):
            import numpy as np
            Rec.calls.append({"texts": texts, "kwargs": {k: kw[k] for k in sorted(kw)}})
            n = 1 if isinstance(texts, str) else len(texts)
            out = np.ones((n, 8), np.float32)
            return out[0] if isinstance(texts, str) else out

    old = E.EmbeddingService.engine_factory
    E.EmbeddingService.engine_factory = Rec
    monkeypatch.setenv("EMBEDDING_MODEL_NAME", "shibing624/text2vec-base-chinese")
    monkeypatch.setenv("EMBEDDING_DEVICE", "cpu")       # restored afterwards: later GPU tests build services on cuda
    try:
        es = E.EmbeddingService()
        probe = ["急性胃肠炎", "query: 已带前缀", "passage: 已带前缀", "", " 前导空格", "Query: 大写不算"]
        for t in probe:
            es.encode_single(t)
            es.encode_query(t)
        assert es.encode_batch([]) == g["outs"]["encode_batch_empty"]
        eb = es.encode_batch(probe, show_progress=False)
        assert [type(eb).__name__, type(eb[0]).__name__, type(eb[0][0]).__name__] == g["outs"]["encode_batch_type"]
        es.encode_icd_record({"code": "A00", "preferred_zh": "霍乱"})
        es.encode_icd_record({"code": "A00", "preferred_zh": "  "})
        es.encode_icd_record({"preferred_zh": ""})
        assert es.get_model_info() == g["model_info"]
        te = es.test_embedding("测试")
        assert sorted(te.keys()) == g["test_embedding_keys"] and list(te["embedding_shape"]) == g["test_embedding_shape"]
        assert Rec.calls == g["calls"]           # every text and kwarg the reference sends its engine
        es.model = None
        with pytest.raises(RuntimeError, match="嵌入模型未加载"):
            es.encode_single("x")
        with pytest.raises(RuntimeError):
            es.encode_batch(["x"])
        assert es.get_model_info() == {"loaded": False}
    finally:
        E.EmbeddingService.engine_factory = old


def test_tokenizers_read_the_vocab_file(tmp_path):
    """transformers >= 5 ignores BertTokenizerFast(vocab_file=...) and falls back to a 5-token vocabulary, which turns
    every character into [UNK]: both the oracle's and the product's tokenizer must really use vocab.txt (ids of
    bert-base-chinese specials, no [UNK] for characters the vocabulary holds) and agree with each other."""
    import importlib
    from oracle import encoder as oenc
    texts = ["query: 霍乱 | 未特指的霍乱 | ICD-10: A00.901", "急性胃肠炎 发热"]
    vocab = oenc.make_vocab(texts, size=3000)
    p = tmp_path / "vocab.txt"
    p.write_text("\n".join(vocab) + "\n", encoding="utf-8")
    a = oenc.make_tokenizer(str(p))
    b = importlib.import_module("rag-project-icd10_b200.engine.encoder").load_tokenizer(str(tmp_path))
    for tok in (a, b):
        assert tok.vocab_size == 3000
        assert (tok.pad_token_id, tok.unk_token_id, tok.cls_token_id, tok.sep_token_id) == (0, 100, 101, 102)
        ids = tok(texts[1])["input_ids"]
        assert ids[0] == 101 and ids[-1] == 102 and 100 not in ids and len(set(ids)) >= 8
    assert a(texts)["input_ids"] == b(texts)["input_ids"]


def test_header_is_plain_c_and_matches_the_library(tmp_path):
    """include/icdrag.h is the drop-in boundary: it must compile as C (no C++/torch/CUDA types in the signatures) and a
    C program that references every declared function must link against libicdrag.so."""
    import re
    import shutil
    import subprocess
    if shutil.which("gcc") is None:
        pytest.skip("gcc not available")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    hdr = os.path.join(root, "include", "icdrag.h")
    src = open(hdr, encoding="utf-8").read()
    names = sorted(set(re.findall(r"\b(icd_[a-z0-9_]+)\s*\(", re.sub(r"/\*.*?\*/", "", src, flags=re.S))))
    native = importlib.import_module("rag-project-icd10_b200._native")
    assert names == sorted(native.SYMBOLS), (set(names) ^ set(native.SYMBOLS))
    c = tmp_path / "use_all.c"
    c.write_text('#include "icdrag.h"\n#include <stdio.h>\ntypedef void (*fn)(void);\nint main(void) {\n  fn p[] = {' +
                 ", ".join(f"(fn){n}" for n in names) + "};\n  printf(\"%d %d\\n\", (int)(sizeof p / sizeof p[0]), icd_version());\n  return 0;\n}\n")
    exe = tmp_path / "use_all"
    libdir = os.path.dirname(native.LIB_PATH)
    out = subprocess.run(["gcc", "-std=c99", "-Wall", "-Werror", "-pedantic", "-I", os.path.dirname(hdr), str(c), "-o", str(exe),
                          "-L", libdir, "-licdrag", f"-Wl,-rpath,{libdir}"], capture_output=True, text=True)
    assert out.returncode == 0, out.stderr
    run = subprocess.run([str(exe)], capture_output=True, text=True)
    assert run.returncode == 0 and run.stdout.split()[0] == str(len(names)), (run.stdout, run.stderr)


def test_lazy_batch_is_a_read_only_sequence_of_candidate_lists():
    """MilvusService.search_batch hands back a LazyBatch: element b behaves like the list search() returns for query b,
    built on access from the [B, k] result arrays (missing hits are -1 at the tail of a row)."""
    import numpy as np
    ms = importlib.import_module("rag-project-icd10_b200.services.milvus_service")

    class _Svc:                                     # stands where MilvusService stands: one dict per (row, distance)
        calls = 0

        def _candidate_of_row(self, row_id, distance):
            _Svc.calls += 1
            return {"code": f"R{row_id}", "original_score": distance}

    ids = np.array([[5, 3, 9], [7, -1, -1], [-1, -1, -1]], np.int64)
    raw = np.array([[0.9, 0.8, 0.7], [0.5, 0.0, 0.0], [0.0, 0.0, 0.0]], np.float32)
    batch = ms.LazyBatch(_Svc(), raw, ids)
    assert len(batch) == 3 and _Svc.calls == 0                       # nothing is materialised up front
    assert [len(c) for c in batch] == [3, 1, 0]
    assert [h["code"] for h in batch[0]] == ["R5", "R3", "R9"] and _Svc.calls == 3
    assert batch[0][1] == {"code": "R3", "original_score": float(np.float32(0.8))} and _Svc.calls == 3   # cached
    assert batch[-2] == [{"code": "R7", "original_score": 0.5}] and list(batch[2]) == []
    assert [len(c) for c in batch[1:]] == [1, 0] and batch[0] is batch[0]
    assert batch == [list(c) for c in batch] and batch.row_ids is ids and batch.raw_scores is raw
    assert list(batch[0].row_ids) == [5, 3, 9] and list(batch[1].raw_scores) == [0.5]
    with pytest.raises(IndexError):
        batch[3]
    # the per-query object alone (what search_batch returned before): trims the tail itself
    one = ms.LazyCandidates(_Svc(), raw[1], ids[1])
    assert len(one) == 1 and one == [{"code": "R7", "original_score": 0.5}] and one[-1]["code"] == "R7"


def test_every_documented_knob_is_accepted_and_unknown_ones_are_not(native):
    """icd_tune is host state only (no GPU needed): every key include/icdrag.h documents is accepted, anything else is an
    argument error with a message; the defaults are restored afterwards."""
    hdr = open(os.path.join(ROOT, "include", "icdrag.h")).read()
    doc = hdr[hdr.index("process-wide tuning knobs"):hdr.index("int icd_tune(")]
    keys = sorted(set(re.findall(r'"((?:scan|enc)_[a-z_]+)"', doc)))
    defaults = dict(scan_sample=-1, scan_drift=4, scan_tmax=16, scan_kbs=3, scan_kbs_pair=6, scan_pair=-1, scan_qsplit=-1,
                    scan_qtmem=0, scan_generic=0, scan_pre_slots=1, scan_small_pre=1, enc_pdl=1, enc_skinny=1)
    assert keys == sorted(defaults), (keys, sorted(defaults))
    try:
        for k in keys:
            native.tune(**{k: 0})
    finally:
        native.tune(**defaults)
    with pytest.raises(native.NativeError, match="unknown key"):
        native.tune(scan_no_such_knob=1)
