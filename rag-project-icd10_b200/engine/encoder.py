"""EncoderEngine -- the object EmbeddingService holds where the reference holds a
``SentenceTransformer`` (/root/reference/services/embedding_service.py:61): same members the
reference uses -- ``encode(str | list, batch_size=, show_progress_bar=, normalize_embeddings=)``,
``get_sentence_embedding_dimension()``, ``max_seq_length`` -- with the BERT forward, pooling and
normalisation running in libicdrag.so on the GPU.  Only tokenisation stays on the host.
"""
from __future__ import annotations

import ctypes as C
import os
import threading
import time
from concurrent.futures import ThreadPoolExecutor
from typing import List, Optional, Sequence, Union

import numpy as np

from .. import _native as N
from . import weights as W
from .tokenizer import NativeTokenizer

MAX_S = 512  # kernel limit (BERT's position table); text2vec-base-chinese's own max_seq_length is 128, e5-large's 512
FEED_CHUNK = 32768   # sentences tokenised / length-bucketed / copied back as one unit of the feeder pipeline
SMALL_BATCH = 256    # up to this many sentences take the direct path (one tokeniser call, synchronous launches)


class EncoderEngine:
    def __init__(self, model_name_or_path: Optional[str] = None, device: Union[str, int, None] = None, *,
                 cfg: Optional[N.BertCfg] = None, blob: Optional[np.ndarray] = None, tokenizer=None,
                 max_seq_length: int = 128, max_tokens: int = 4096 * 64, vocab_path: Optional[str] = None,
                 host_threads: Optional[int] = None, position_offset: int = 0, unk_id: Optional[int] = None):
        """position_offset / unk_id (programmatic use with cfg= / blob=; a model directory supplies its own): token t
        of a sequence reads position row position_offset + t (XLM-R: pad_token_id + 1), ids outside the vocabulary
        read row unk_id (None: [UNK] = 100 of BERT vocabularies)."""
        N.require_gpu()
        self.device_index = _device_index(device)
        if blob is None:
            path = W.resolve_model_dir(model_name_or_path)
            cfg, blob, meta = W.load_model_dir(path)
            max_seq_length = meta["max_seq_length"]
            position_offset, unk_id = meta["position_offset"], meta["unk_id"]
            if tokenizer is None:
                tokenizer = load_tokenizer(path)
        if tokenizer is None:
            raise ValueError("a tokenizer is required")
        self.cfg = cfg
        self.tokenizer = tokenizer
        self.position_offset = int(position_offset)
        self.unk_id = unk_id
        # position rows position_offset .. position_offset + S - 1 must exist (XLM-R: 514 rows, offset 2 -> 512 tokens)
        self.max_seq_length = min(int(max_seq_length), MAX_S, cfg.max_position - self.position_offset)
        self.max_tokens = int(max_tokens)
        self.vocab_path = vocab_path
        self.last_stats: dict = {}
        self._feed = None          # pinned staging buffers, created on first bulk encode
        # one in-flight call per native handle (include/icdrag.h): the reference serves requests from a thread pool
        # (FastAPI sync endpoints), and ctypes releases the GIL during a call
        self._lock = threading.RLock()
        # host feeder: multi-threaded WordPiece in libicdrag for plain BERT tokenizers, the tokenizer itself otherwise
        self._ntok = NativeTokenizer(tokenizer, threads=host_threads) if hasattr(tokenizer, "backend_tokenizer") else None
        self._h = C.c_void_p()
        blob = np.ascontiguousarray(blob, np.float32)
        N.check(N.lib().icd_encoder_create(N.buf_ptr(blob), blob.size, C.byref(cfg), self.device_index,
                                           C.byref(self._h)), "icd_encoder_create")
        N.check(N.lib().icd_encoder_set_embedding_ids(self._h, self.position_offset, -1 if unk_id is None else int(unk_id)),
                "icd_encoder_set_embedding_ids")

    # ---------------------------------------------------------------- SentenceTransformer surface
    def get_sentence_embedding_dimension(self) -> int:
        return int(self.cfg.hidden)

    def encode(self, sentences, batch_size: int = 32, show_progress_bar=None, normalize_embeddings: bool = False,
               convert_to_numpy: bool = True, convert_to_tensor: bool = False, **_ignored):
        """convert_to_tensor=True (SentenceTransformer's switch) returns a float32 CUDA tensor: the embeddings stay on
        the device they were computed on (the sharded build appends them to that GPU's table without a host round trip)."""
        single = isinstance(sentences, str)
        items: List[str] = [sentences] if single else list(sentences)
        if not items:
            if convert_to_tensor:
                import torch
                return torch.zeros((0, self.cfg.hidden), dtype=torch.float32, device=torch.device("cuda", self.device_index))
            return np.zeros((0, self.cfg.hidden), np.float32)
        out = self._encode_texts(items, normalize_embeddings, to_device=convert_to_tensor)
        return out[0] if single else out

    def close(self) -> None:
        if getattr(self, "_feed", None) is not None:
            self._feed["pool"].shutdown(wait=True)
            self._feed = None
        if getattr(self, "_h", None) is not None and self._h.value:
            N.lib().icd_encoder_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---------------------------------------------------------------- host side
    def tokenize(self, texts: Sequence[str]) -> List[List[int]]:
        ids, lens = self._token_table(list(texts))
        return [ids[i, :lens[i]].tolist() for i in range(len(lens))]

    def _token_table(self, texts: List[str]):
        """ids [n, max_seq_length] int32 (row i valid up to lens[i]) and lens [n] int32."""
        L = self.max_seq_length
        if self._ntok is not None:
            return self._ntok.encode(texts, L)
        enc = self.tokenizer(texts, padding=False, truncation=True, max_length=L, add_special_tokens=True,
                             return_attention_mask=False, return_token_type_ids=False)["input_ids"]
        ids = np.zeros((len(enc), L), np.int32)
        lens = np.zeros((len(enc),), np.int32)
        for i, row in enumerate(enc):
            lens[i] = len(row)
            ids[i, :len(row)] = row
        return ids, lens

    def _pack(self, ids, lens, rows, S, out_ids, out_lens) -> None:
        if self._ntok is not None:
            self._ntok.pack(ids, lens, rows, S, out_ids, out_lens)
        else:
            out_ids[:] = ids[rows, :S]
            out_lens[:] = np.minimum(lens[rows], S)
            out_ids[np.arange(S)[None, :] >= out_lens[:, None]] = 0

    def _batches(self, lens: np.ndarray):
        """Length-bucketed batches over one chunk: rows by descending token count, cut where B*S would exceed
        max_tokens.  Yields (rows, S)."""
        order = np.argsort(-lens.astype(np.int64), kind="stable")
        lo, n = 0, len(order)
        while lo < n:
            S = max(1, int(lens[order[lo]]))
            B = max(1, min(n - lo, self.max_tokens // S))
            yield order[lo:lo + B], S
            lo += B

    def _encode_texts(self, items: List[str], normalise: bool, to_device: bool = False):
        n, H = len(items), int(self.cfg.hidden)
        if n <= SMALL_BATCH and not to_device:
            # direct path (the reference's live pattern is batch 1): one tokeniser call, synchronous launches
            t0 = time.perf_counter()
            ids, lens = self._token_table(items)
            t1 = time.perf_counter()
            out = np.empty((n, H), np.float32)
            for rows, S in self._batches(lens):
                mat = np.empty((len(rows), S), np.int32)
                bl = np.empty((len(rows),), np.int32)
                self._pack(ids, lens, rows, S, mat, bl)
                out[rows] = self.forward_ids(mat, bl, normalise=normalise)
            self.last_stats = {"sentences": n, "tokens": int(lens.sum()), "tokenize_s": t1 - t0,
                               "encode_s": time.perf_counter() - t1, "h2d_bytes": int(lens.sum()) * 4,
                               "tokenizer": self._tokenizer_kind()}
            return out
        with self._lock:     # the pipeline owns the pinned slots and the stream for its whole duration
            return self._encode_pipelined(items, normalise, to_device)

    def _tokenizer_kind(self) -> str:
        if self._ntok is not None and self._ntok.native:
            return f"native WordPiece, {self._ntok.threads} host threads ({self._ntok.fallbacks} sentences via the wrapped tokenizer)"
        return "wrapped tokenizer (transformers)"

    def _feed_buffers(self):
        """Pinned staging, allocated once: two id / length slots (a batch is packed while the previous one is in
        flight) and two output slots (a chunk's embeddings are copied back while the next chunk runs)."""
        if self._feed is None:
            import torch
            dev = torch.device("cuda", self.device_index)
            f = {"dev": dev, "stream": torch.cuda.Stream(device=dev)}
            f["ids"] = [torch.empty((self.max_tokens,), dtype=torch.int32).pin_memory() for _ in range(2)]
            f["lens"] = [torch.empty((self.max_tokens,), dtype=torch.int32).pin_memory() for _ in range(2)]
            f["in_ev"] = [torch.cuda.Event() for _ in range(2)]
            f["out"] = [torch.empty((FEED_CHUNK, int(self.cfg.hidden)), dtype=torch.float32).pin_memory() for _ in range(2)]
            f["out_ev"] = [torch.cuda.Event() for _ in range(2)]
            f["d_sorted"] = torch.empty((FEED_CHUNK, int(self.cfg.hidden)), dtype=torch.float32, device=dev)
            f["inv"] = [torch.empty((FEED_CHUNK,), dtype=torch.int64).pin_memory() for _ in range(2)]
            f["d_inv"] = torch.empty((FEED_CHUNK,), dtype=torch.int64, device=dev)
            f["pool"] = ThreadPoolExecutor(max_workers=1)
            self._feed = f
        return self._feed

    def _encode_pipelined(self, items: List[str], normalise: bool, to_device: bool = False):
        """The feeder (SURVEY section 7 "hard part"): while the GPU encodes chunk c, a worker thread tokenises chunk
        c+1 (the C call releases the GIL) and the main thread packs length-bucketed batches into pinned slots; every
        launch is asynchronous on one stream, embeddings land in sorted order on the device, are un-sorted there and
        leave through pinned buffers while the next chunk runs."""
        import torch
        f = self._feed_buffers()
        n, H = len(items), int(self.cfg.hidden)
        out = None if to_device else np.empty((n, H), np.float32)
        out_dev = torch.empty((n, H), dtype=torch.float32, device=f["dev"]) if to_device else None
        stream = f["stream"]
        chunks = [(lo, min(n, lo + FEED_CHUNK)) for lo in range(0, n, FEED_CHUNK)]
        stats = {"sentences": n, "tokens": 0, "h2d_bytes": 0, "tokenize_wait_s": 0.0, "pack_s": 0.0, "slot_wait_s": 0.0,
                 "launch_s": 0.0, "unsort_s": 0.0, "copy_out_s": 0.0, "batches": 0}
        t_all = time.perf_counter()
        fut = f["pool"].submit(self._token_table, items[chunks[0][0]:chunks[0][1]])
        pending = None       # (chunk index, lo, hi) whose output copy is in flight
        slot = 0

        def finish(p):
            ci, lo, hi = p
            t0 = time.perf_counter()
            f["out_ev"][ci & 1].synchronize()
            np.copyto(out[lo:hi], f["out"][ci & 1].numpy()[:hi - lo])
            stats["copy_out_s"] += time.perf_counter() - t0

        with torch.cuda.stream(stream):
            for ci, (lo, hi) in enumerate(chunks):
                t0 = time.perf_counter()
                ids, lens = fut.result()
                stats["tokenize_wait_s"] += time.perf_counter() - t0
                if ci + 1 < len(chunks):
                    fut = f["pool"].submit(self._token_table, items[chunks[ci + 1][0]:chunks[ci + 1][1]])
                m = hi - lo
                stats["tokens"] += int(lens.sum())
                d_sorted = f["d_sorted"]
                perm = np.empty((m,), np.int64)
                row0 = 0
                for rows, S in self._batches(lens):
                    B = len(rows)
                    t0 = time.perf_counter()
                    f["in_ev"][slot].synchronize()          # the batch that used this slot two launches ago is done
                    t1 = time.perf_counter()
                    h_ids = f["ids"][slot].numpy()[:B * S].reshape(B, S)
                    h_lens = f["lens"][slot].numpy()[:B]
                    self._pack(ids, lens, rows, S, h_ids, h_lens)
                    stats["slot_wait_s"] += t1 - t0
                    stats["pack_s"] += time.perf_counter() - t1
                    dt = N.F32 | (0 if normalise else 0x100)
                    t2 = time.perf_counter()
                    N.check(N.lib().icd_encoder_forward(self._h, h_ids.ctypes.data, h_lens.ctypes.data, B, S,
                                                        d_sorted[row0:row0 + B].data_ptr(), dt,
                                                        C.c_void_p(stream.cuda_stream), 0), "icd_encoder_forward")
                    f["in_ev"][slot].record(stream)
                    stats["launch_s"] += time.perf_counter() - t2
                    stats["h2d_bytes"] += B * S * 4 + B * 4
                    stats["batches"] += 1
                    perm[row0:row0 + B] = rows
                    row0 += B
                    slot ^= 1
                # un-sort on the device, copy back through the pinned slot of this chunk
                if pending is not None and (pending[0] & 1) == (ci & 1):
                    finish(pending)
                    pending = None
                t3 = time.perf_counter()
                inv = f["inv"][ci & 1].numpy()           # free again: chunk ci-2 was finished an iteration ago
                inv[perm] = np.arange(m)
                f["d_inv"][:m].copy_(f["inv"][ci & 1][:m], non_blocking=True)
                if to_device:
                    torch.index_select(d_sorted[:m], 0, f["d_inv"][:m], out=out_dev[lo:hi])
                    f["out_ev"][ci & 1].record(stream)      # the pinned `inv` slot is free once this has run
                    if ci >= 1:
                        f["out_ev"][(ci - 1) & 1].synchronize()
                    continue
                f["out"][ci & 1][:m].copy_(d_sorted[:m].index_select(0, f["d_inv"][:m]), non_blocking=True)
                f["out_ev"][ci & 1].record(stream)
                stats["unsort_s"] += time.perf_counter() - t3
                if pending is not None:
                    finish(pending)
                pending = (ci, lo, hi)
            if pending is not None:
                finish(pending)
            if to_device:
                stream.synchronize()
        stats["total_s"] = time.perf_counter() - t_all
        stats["tokenizer"] = self._tokenizer_kind()
        self.last_stats = stats
        return out_dev if to_device else out

    def forward_ids(self, ids, lens, normalise: bool = True, out=None, stream: int = 0, sync: bool = True):
        """ids [B,S] int32, lens [B] int32 (numpy host or torch host/device) -> [B,hidden] float32."""
        B, S = int(ids.shape[0]), int(ids.shape[1])
        if out is None:
            if N._is_torch(ids) and ids.is_cuda:
                import torch
                out = torch.empty((B, self.cfg.hidden), dtype=torch.float32, device=ids.device)
            else:
                out = np.empty((B, self.cfg.hidden), np.float32)
        dt = N.vec_dtype(out) | (0 if normalise else 0x100)
        with self._lock:
            N.check(N.lib().icd_encoder_forward(self._h, N.buf_ptr(ids), N.buf_ptr(lens), B, S, N.buf_ptr(out), dt,
                                                C.c_void_p(stream), 1 if sync else 0), "icd_encoder_forward")
        return out

    def set_token_head(self, weight: np.ndarray, bias: np.ndarray) -> None:
        """classifier.weight [labels, hidden] / classifier.bias [labels] of a BertForTokenClassification."""
        weight = np.ascontiguousarray(weight, np.float32)
        bias = np.ascontiguousarray(bias, np.float32)
        if weight.ndim != 2 or weight.shape[1] != self.cfg.hidden or bias.shape != (weight.shape[0],):
            raise ValueError("token head must be weight [labels, hidden] and bias [labels]")
        N.check(N.lib().icd_encoder_set_token_head(self._h, N.buf_ptr(weight), N.buf_ptr(bias), int(weight.shape[0])),
                "icd_encoder_set_token_head")
        self.num_labels = int(weight.shape[0])

    def token_logits(self, ids, lens, out=None, stream: int = 0, sync: bool = True):
        """ids [B,S] int32, lens [B] int32 -> per-token logits [B,S,labels] float32 (set_token_head first)."""
        B, S = int(ids.shape[0]), int(ids.shape[1])
        L = getattr(self, "num_labels", 0)
        if L <= 0:
            raise N.NativeError("no token head set on this encoder")
        if out is None:
            if N._is_torch(ids) and ids.is_cuda:
                import torch
                out = torch.empty((B, S, L), dtype=torch.float32, device=ids.device)
            else:
                out = np.empty((B, S, L), np.float32)
        with self._lock:
            N.check(N.lib().icd_encoder_token_logits(self._h, N.buf_ptr(ids), N.buf_ptr(lens), B, S, N.buf_ptr(out),
                                                     C.c_void_p(stream), 1 if sync else 0), "icd_encoder_token_logits")
        return out

    def read_hidden(self, tokens: int) -> np.ndarray:
        out = np.empty((tokens, self.cfg.hidden), np.float32)
        N.check(N.lib().icd_encoder_read_hidden(self._h, 0, N.buf_ptr(out), out.size), "icd_encoder_read_hidden")
        return out


def _device_index(device) -> int:
    if device is None:
        return 0
    if isinstance(device, int):
        return device
    s = str(device)
    if s in ("cuda", "auto"):
        return 0
    if s.startswith("cuda:"):
        return int(s.split(":")[1])
    raise N.NativeError(f"EncoderEngine runs on CUDA devices only (got device={device!r}); there is no CPU fallback")


def bert_tokenizer_from_vocab(vocab_path: str, do_lower_case: bool = True):
    """BertTokenizerFast over a vocab.txt.  transformers >= 5 takes the vocabulary as `vocab=` (a token -> id dict)
    and silently ignores `vocab_file=` (leaving a 5-token vocabulary that maps every character to [UNK]);
    transformers 4 takes `vocab_file=`.  Either way the result is checked against the file."""
    from transformers import BertTokenizerFast
    with open(vocab_path, encoding="utf-8") as fh:
        tokens = [line.rstrip("\n") for line in fh]
    while tokens and tokens[-1] == "":
        tokens.pop()
    vocab = {t: i for i, t in enumerate(tokens)}
    tok = None
    for kwargs in ({"vocab": vocab}, {"vocab_file": vocab_path}):
        try:
            cand = BertTokenizerFast(do_lower_case=do_lower_case, **kwargs)
        except Exception:
            continue
        if cand.vocab_size == len(vocab):
            tok = cand
            break
    if tok is None:
        raise RuntimeError(f"could not build a BERT tokenizer over {vocab_path} ({len(vocab)} entries)")
    return tok


def load_tokenizer(path: str):
    """The model directory's own tokenizer; falls back to BertTokenizerFast over vocab.txt."""
    from transformers import AutoTokenizer
    vocab_path = os.path.join(path, "vocab.txt")
    try:
        if os.path.exists(os.path.join(path, "tokenizer_config.json")) or os.path.exists(os.path.join(path, "tokenizer.json")):
            tok = AutoTokenizer.from_pretrained(path, local_files_only=True)
            if tok.vocab_size > 5 or not os.path.exists(vocab_path):   # a 5-token vocabulary = the file was ignored
                return tok
    except Exception:
        pass
    return bert_tokenizer_from_vocab(vocab_path)
