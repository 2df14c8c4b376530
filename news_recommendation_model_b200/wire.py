"""Compact wire format for impressions (SURVEY.md section 8f, rows N3 / N4) — an ADDITIONAL entry point next to the
reference's packed float64 tensors, which `UserModel.forward` keeps accepting unchanged.

`tool/process_data.py:195-252` stores, for every click of every impression, the full 80-number article record as
float64 (640 B per history row, 200 rows per impression, ids as doubles).  74 of those numbers (and the 3 columns of
`x_global`) depend on the article only; a click adds 4 time buckets, read time and scroll.  Here the article records
live ONCE in device memory (`ArticleTable`, float32 — the model casts its inputs to float32 first,
`user_invariant_interest_model.py:74-75`) and an impression travels as ids:

    history row  640 B -> 16 B   (int32 article, packed uint32 time, float32 read_time + scroll)
    candidate    648 B ->  8 B   (+ 4 B float32 label)

`expand(table, batch)` rebuilds the packed float64 tensors on the GPU (`nrm_expand_compact`, one kernel) so every
kernel behind `UserModel.forward` runs unchanged and produces bit-identical results;
`FusedTrainStep.load` accepts a `CompactBatch` directly and does the expansion inside its CUDA graph.

`from_records` converts the reference's own record lists (`process_data.py:252`, what `import_processed_data` returns)
once, on the host, into a table + compact arrays in pinned memory; `CompactDataset.batches` then yields pre-batched
pinned `CompactBatch`es; `PrefetchLoader` does the same from a background thread into a fixed pinned ring (the data-loader row N4:
no per-step collate of float64 `[B,200,80]`, no per-batch pinning)."""
from __future__ import annotations

import queue
import threading
import time
from dataclasses import dataclass
from typing import Iterator, List, Optional, Sequence

import numpy as np
import torch

from . import _lib
from .config import GLOBAL_COLS, HIST_COLS, TGT_COLS
from .engine import _ptr, _stream
from .synthetic import Batch

ARTICLE_COLS = 80           # float32 per article row: pca 64 | cat | sub 5 | sent 3 | type | global 3 | pad 3
_ART_FEATS = 74             # packed columns 4..77
_YEAR_MAX, _MONTH_MAX, _DAY_MAX, _HOUR_MAX = 0xfff, 0xf, 0x1f, 0x1f


def pack_time(t: np.ndarray) -> np.ndarray:
    """[..., 4] integer time buckets (years, months, days, hours; tool/normalization.py:31-39) -> uint32."""
    t = np.asarray(t)
    ti = t.astype(np.int64)
    if (ti != t).any() or (ti < 0).any() or (ti[..., 0] > _YEAR_MAX).any() or (ti[..., 1] > _MONTH_MAX).any() \
            or (ti[..., 2] > _DAY_MAX).any() or (ti[..., 3] > _HOUR_MAX).any():
        raise ValueError('time buckets must be integers within (4095, 15, 31, 31)')
    return (ti[..., 0] | (ti[..., 1] << 12) | (ti[..., 2] << 16) | (ti[..., 3] << 21)).astype(np.uint32)


@dataclass
class ArticleTable:
    rows: torch.Tensor        # [n_articles, 80] float32, row 0 all-zero

    def to(self, device):
        return ArticleTable(self.rows.to(device))

    @property
    def n(self) -> int:
        return int(self.rows.shape[0])


@dataclass
class CompactBatch:
    impression_id: torch.Tensor   # [B] int64
    user_id: torch.Tensor         # [B] int64
    hist_article: torch.Tensor    # [B,H] int32 (0 = pad row)
    hist_time: torch.Tensor       # [B,H] int32 holding the packed uint32
    hist_click: torch.Tensor      # [B,H,2] float32
    cand_article: torch.Tensor    # [B,C] int32 (0 = pad candidate)
    cand_time: torch.Tensor       # [B,C] int32 holding the packed uint32
    label: torch.Tensor           # [B,C] float32
    empty_num: torch.Tensor       # [B] int64

    def to(self, device, non_blocking=False):
        return CompactBatch(*[getattr(self, f).to(device, non_blocking=non_blocking) for f in self.__dataclass_fields__])

    def pin(self):
        return CompactBatch(*[getattr(self, f).pin_memory() for f in self.__dataclass_fields__])

    def input_bytes(self) -> int:
        return sum(t.numel() * t.element_size() for t in (self.hist_article, self.hist_time, self.hist_click, self.cand_article,
                                                          self.cand_time, self.label, self.user_id))

    @property
    def shape(self):
        return int(self.hist_article.shape[0]), int(self.hist_article.shape[1]), int(self.cand_article.shape[1])


def expand_into(table: ArticleTable, cb: CompactBatch, xh: torch.Tensor, xt: torch.Tensor, xg: torch.Tensor,
                label: Optional[torch.Tensor]) -> None:
    """Enqueue `nrm_expand_compact` on the current stream: device CompactBatch -> packed float64 tensors (preallocated)."""
    B, H, C = cb.shape
    dev = xh.device
    if not (table.rows.is_cuda and cb.hist_article.is_cuda):
        raise _lib.NrmError('wire.expand runs on CUDA tensors only (no CPU fallback)')
    for t, shape, dt in ((xh, (B, H, HIST_COLS), torch.float64), (xt, (B, C, TGT_COLS), torch.float64), (xg, (B, C, GLOBAL_COLS), torch.float64)):
        if tuple(t.shape) != shape or t.dtype != dt or not t.is_contiguous():
            raise ValueError('expand_into: output tensors must be contiguous float64 [B,H,80] / [B,C,78] / [B,C,3]')
    if table.rows.dtype != torch.float32 or table.rows.shape[1] != ARTICLE_COLS or not table.rows.is_contiguous():
        raise ValueError('article table must be contiguous float32 [n, 80]')
    for t, dt in ((cb.hist_article, torch.int32), (cb.hist_time, torch.int32), (cb.hist_click, torch.float32), (cb.cand_article, torch.int32),
                  (cb.cand_time, torch.int32), (cb.label, torch.float32)):
        if t.dtype != dt or not t.is_contiguous():
            raise ValueError('CompactBatch tensors must be contiguous int32 / float32 as documented')
    _lib.check(_lib.load().nrm_expand_compact(_ptr(table.rows), table.n, _ptr(cb.hist_article), _ptr(cb.hist_time), _ptr(cb.hist_click),
                                              _ptr(cb.cand_article), _ptr(cb.cand_time), _ptr(cb.label) if label is not None else None,
                                              B, H, C, _ptr(xh), _ptr(xt), _ptr(xg), _ptr(label),
                                              _stream(dev)), 'nrm_expand_compact')


def expand(table: ArticleTable, cb: CompactBatch) -> Batch:
    """Device CompactBatch -> device `Batch` in the reference's packed layout (what `UserModel.forward` / `.loss` take)."""
    B, H, C = cb.shape
    dev = cb.hist_article.device
    xh = torch.empty(B, H, HIST_COLS, dtype=torch.float64, device=dev)
    xt = torch.empty(B, C, TGT_COLS, dtype=torch.float64, device=dev)
    xg = torch.empty(B, C, GLOBAL_COLS, dtype=torch.float64, device=dev)
    label = torch.empty(B, C, dtype=torch.float64, device=dev)
    expand_into(table, cb, xh, xt, xg, label)
    label_id = torch.where(cb.cand_article > 0, cb.cand_article.to(torch.float64), torch.full_like(cb.cand_article, -1, dtype=torch.float64))
    return Batch(cb.impression_id, cb.user_id, xh, xt, xg, label, label_id, cb.empty_num)


# ---------------------------------------------------------------------------------------------------------
# host side: the reference's records -> table + compact arrays (done once per dataset)
# ---------------------------------------------------------------------------------------------------------
class CompactDataset:
    """All impressions of a dataset in the compact format, in pinned host memory."""

    def __init__(self, table: ArticleTable, data: CompactBatch):
        self.table, self.data = table, data

    def __len__(self) -> int:
        return int(self.data.hist_article.shape[0])

    def select(self, idx) -> CompactBatch:
        idx = torch.as_tensor(idx, dtype=torch.int64)
        return CompactBatch(*[getattr(self.data, f).index_select(0, idx) for f in self.data.__dataclass_fields__])

    def batches(self, batch_size: int, shuffle: bool = False, seed: int = 0, drop_last: bool = False, pin: bool = True
                ) -> Iterator[CompactBatch]:
        """Pre-batched (optionally shuffled, as `train.py:37-40`'s DataLoader) pinned CompactBatches."""
        n = len(self)
        order = torch.randperm(n, generator=torch.Generator().manual_seed(seed)) if shuffle else torch.arange(n)
        for s in range(0, n, batch_size):
            idx = order[s:s + batch_size]
            if drop_last and idx.numel() < batch_size:
                return
            b = self.select(idx)
            yield b.pin() if pin else b


class PrefetchLoader:
    """The data-loader row N4 as a pipeline: a background thread gathers the next batches of a `CompactDataset` into a FIXED ring
    of pinned host buffers (allocated once: no `cudaHostAlloc` per batch, the cost that makes `pin_memory()` per batch slower than
    the training step itself) while the GPU trains on the current one.  Replaces `torch.utils.data.DataLoader(list, batch_size,
    shuffle=True)` + default collate of float64 `[B,200,80]` records (train.py:37-40).

        loader = PrefetchLoader(ds, batch_size, shuffle=True)      # once: the pinned ring is allocated here
        for cb in loader.set_epoch(epoch):                       # cb: pinned CompactBatch view of a ring slot (the last one may be shorter)
            handle = step.step(cb)              # FusedTrainStep.load enqueues the H2D copies and releases the slot when they are done

    A slot is recycled once its consumer has released it: `FusedTrainStep.load` does so with the event of its copy stream;
    any other consumer may call `loader.release(cb, event)` after enqueuing its copies, or do nothing, in which case the slot is
    released when the NEXT batch is requested, with an event recorded on the current stream at that moment."""

    def __init__(self, dataset: CompactDataset, batch_size: int, shuffle: bool = False, seed: int = 0, drop_last: bool = False,
                 depth: int = 4, pin: bool = True):
        if depth < 2:
            raise ValueError('PrefetchLoader needs a ring of at least 2 slots')
        self.ds, self.batch_size, self.shuffle, self.seed, self.drop_last, self.depth = dataset, batch_size, shuffle, seed, drop_last, depth
        d = dataset.data
        self.fields = list(d.__dataclass_fields__)
        pin = pin and torch.cuda.is_available()               # CPU-only hosts (unit tests): plain buffers, same logic

        def buf(f):
            t = torch.empty((batch_size,) + tuple(getattr(d, f).shape[1:]), dtype=getattr(d, f).dtype)
            return t.pin_memory() if pin else t
        self.ring = [CompactBatch(*[buf(f) for f in self.fields]) for _ in range(depth)]
        self._src = {f: getattr(d, f).numpy() for f in self.fields}                       # numpy views (no copies)
        self._dst = [{f: getattr(b, f).numpy() for f in self.fields} for b in self.ring]
        self._free: 'queue.Queue' = queue.Queue()
        self._full: 'queue.Queue' = queue.Queue()
        self._events = [None] * depth
        self._thread: Optional[threading.Thread] = None
        self._pending_slot: Optional[int] = None
        self._lock = threading.Lock()

    def set_epoch(self, seed: int) -> 'PrefetchLoader':
        """Shuffle seed of the next pass (the ring is allocated once; iterate the same loader every epoch)."""
        self.seed = seed
        return self

    def __len__(self) -> int:
        n = len(self.ds)
        return n // self.batch_size if self.drop_last else (n + self.batch_size - 1) // self.batch_size

    def _worker(self, order: torch.Tensor):
        n = order.numel()
        try:
            for s in range(0, n, self.batch_size):
                idx = order[s:s + self.batch_size]
                if self.drop_last and idx.numel() < self.batch_size:
                    break
                slot = self._free.get()
                if slot is None:
                    return
                ev = self._events[slot]
                if ev is not None:
                    # the consumer's H2D copies out of this slot have finished.  Polling, not cudaEventSynchronize: another thread may
                    # be capturing a CUDA graph, during which synchronising calls are not permitted
                    while not ev.query():
                        time.sleep(20e-6)
                    self._events[slot] = None
                rows = int(idx.numel())
                idx_np = idx.numpy()
                for f in self.fields:                         # numpy gathers (GIL released) straight into the pinned slot
                    np.take(self._src[f], idx_np, axis=0, out=self._dst[slot][f][:rows], mode='clip')
                self._full.put((slot, rows))
        finally:
            self._full.put(None)

    def __iter__(self) -> Iterator[CompactBatch]:
        if self._thread is not None:
            raise RuntimeError('PrefetchLoader: one pass at a time')
        n = len(self.ds)
        order = torch.randperm(n, generator=torch.Generator().manual_seed(self.seed)) if self.shuffle else torch.arange(n)
        while not self._free.empty():
            self._free.get_nowait()
        for i in range(self.depth):
            self._free.put(i)
        self._thread = threading.Thread(target=self._worker, args=(order,), daemon=True)
        self._thread.start()
        try:
            while True:
                item = self._full.get()
                self._release_pending()
                if item is None:
                    break
                slot, rows = item
                buf = self.ring[slot]
                cb = CompactBatch(*[getattr(buf, f)[:rows] for f in self.fields])
                cb._loader, cb._slot = self, slot
                self._pending_slot = slot
                yield cb
        finally:
            self._release_pending()
            self._free.put(None)                              # unblock a worker that waits for a slot
            self._thread.join()
            self._thread = None

    def release(self, cb: CompactBatch, event=None) -> None:
        """The copies out of `cb`'s pinned slot are covered by `event` (default: an event recorded now on the current stream)."""
        slot = getattr(cb, '_slot', None)
        if slot is None or getattr(cb, '_loader', None) is not self:
            return
        with self._lock:
            if self._pending_slot != slot:
                return                                        # already released
            self._pending_slot = None
        if event is None and torch.cuda.is_available():
            event = torch.cuda.Event()
            event.record()
        self._events[slot] = event
        self._free.put(slot)

    def _release_pending(self):
        slot = self._pending_slot
        if slot is not None:
            cb = CompactBatch(*[getattr(self.ring[slot], f) for f in self.fields])
            cb._loader, cb._slot = self, slot
            self.release(cb)


def _zstd_decompress(buf: bytes) -> bytes:
    """One zstd frame -> bytes, with whichever codec this environment has: `zstandard` (what the reference imports,
    tool/process_data.py:16) or the zstd codec bundled with pyarrow."""
    try:
        import zstandard
        return zstandard.ZstdDecompressor().decompress(buf)
    except ImportError:
        pass
    try:
        import pyarrow as pa
    except ImportError as exc:
        raise ImportError('reading a processed-data volume needs `zstandard` or `pyarrow` (zstd codec)') from exc
    with pa.CompressedInputStream(pa.BufferReader(buf), 'zstd') as stream:
        return stream.read()


def _zstd_compress(buf: bytes, level: int = 11) -> bytes:
    try:
        import zstandard
        return zstandard.ZstdCompressor(level=level).compress(buf)
    except ImportError:
        import pyarrow as pa
        return pa.Codec('zstd', compression_level=level).compress(buf, asbytes=True)


def load_processed_volume(path: str) -> list:
    """`tool/process_data.py:import_processed_data` (lines 449-453): one zstd frame holding the pickled record list of a volume
    (`process_data.py:252` layout).  Pickle executes code: only open volumes you produced yourself, as with the reference."""
    import pickle
    with open(path, 'rb') as f:
        return pickle.loads(_zstd_decompress(f.read()))


def save_processed_volume(records, path: str) -> None:
    """`tool/process_data.py:export_processed_data` (lines 455-462): the inverse of `load_processed_volume`, readable by the reference."""
    import pickle
    with open(path, 'wb') as f:
        f.write(_zstd_compress(pickle.dumps(list(records))))


def from_volumes(paths: Sequence[str], pin: bool = False) -> CompactDataset:
    """All impressions of the given processed-data volumes as one compact dataset (one article table over all of them)."""
    records = []
    for p in paths:
        records.extend(load_processed_volume(p))
    return from_records(records, pin=pin)


def from_records(records: Sequence[Sequence], pin: bool = False) -> CompactDataset:
    """`records`: the list `tool/process_data.py:252` builds and `import_processed_data` returns —
    [impression_id, user_id, history [H,80], inview [C,78], global [C,3], label [C], label_id [C], empty_num] per impression,
    all impressions padded to the same H and C.  Article rows are de-duplicated by VALUE (their 74 feature columns, plus
    the 3 global statistics for candidates), so no article id is needed; all-zero rows map to table row 0."""
    B = len(records)
    hist = np.stack([np.asarray(r[2], dtype=np.float64) for r in records])            # [B,H,80]
    cand = np.stack([np.asarray(r[3], dtype=np.float64) for r in records])            # [B,C,78]
    glob = np.stack([np.asarray(r[4], dtype=np.float64) for r in records])            # [B,C,3]
    H, C = hist.shape[1], cand.shape[1]
    feats = np.zeros((B * H + B * C, ARTICLE_COLS), dtype=np.float32)
    feats[:B * H, :_ART_FEATS] = hist[:, :, 4:4 + _ART_FEATS].reshape(B * H, _ART_FEATS)
    feats[B * H:, :_ART_FEATS] = cand[:, :, 4:4 + _ART_FEATS].reshape(B * C, _ART_FEATS)
    feats[B * H:, _ART_FEATS:_ART_FEATS + 3] = glob.reshape(B * C, 3)
    feats += 0.0                                                                      # -0.0 -> +0.0 so that equal values have equal bytes
    rows, inverse = np.unique(feats, axis=0, return_inverse=True)
    inverse = np.asarray(inverse).ravel()
    zero = np.flatnonzero(~rows.any(axis=1))
    if zero.size:                                                                     # move the all-zero row to index 0
        z = int(zero[0])
        new_index = np.arange(rows.shape[0], dtype=np.int64)
        new_index[:z] += 1
        new_index[z] = 0
        rows = np.concatenate((rows[z:z + 1], rows[:z], rows[z + 1:]))
    else:
        new_index = np.arange(rows.shape[0], dtype=np.int64) + 1
        rows = np.concatenate((np.zeros((1, ARTICLE_COLS), np.float32), rows))
    ids = new_index[inverse].astype(np.int32)
    # all-zero packed rows (ETL padding) keep time 0 / click 0 and point at the pad article
    t = torch.from_numpy
    cb = CompactBatch(
        t(np.array([int(np.asarray(r[0])) for r in records], dtype=np.int64)),
        t(np.array([int(np.asarray(r[1])) for r in records], dtype=np.int64)),
        t(ids[:B * H].reshape(B, H).copy()),
        t(pack_time(hist[:, :, 0:4]).view(np.int32).reshape(B, H).copy()),
        t(hist[:, :, 78:80].astype(np.float32)),
        t(ids[B * H:].reshape(B, C).copy()),
        t(pack_time(cand[:, :, 0:4]).view(np.int32).reshape(B, C).copy()),
        t(np.stack([np.asarray(r[5], dtype=np.float32) for r in records])),
        t(np.array([int(np.asarray(r[7])) for r in records], dtype=np.int64)))
    table = ArticleTable(t(np.ascontiguousarray(rows)))
    if pin:
        cb, table = cb.pin(), ArticleTable(table.rows.pin_memory())
    return CompactDataset(table, cb)


# ---------------------------------------------------------------------------------------------------------
# synthetic EB-NeRD-shaped data in the compact format (bench.py, tests)
# ---------------------------------------------------------------------------------------------------------
def make_article_table(n_articles: int = 125_541, seed: int = 7) -> ArticleTable:
    """`n_articles` random article records (EB-NeRD large has 125 541 articles) + the pad article at row 0."""
    from .synthetic import _item_rows
    rng = np.random.default_rng(seed)
    packed = _item_rows(rng, n_articles, TGT_COLS, True)
    rows = np.zeros((n_articles + 1, ARTICLE_COLS), dtype=np.float32)
    rows[1:, :_ART_FEATS] = packed[:, 4:4 + _ART_FEATS]
    rows[1:, _ART_FEATS:_ART_FEATS + 3] = (rng.random((n_articles, 3)) * 0.05).astype(np.float32)
    return ArticleTable(torch.from_numpy(rows))


def make_compact_batch(table: ArticleTable, batch: int, history: int, candidates: int, *, seed: int = 1234, user_num: int = 1000,
                       variable_history: bool = False, variable_candidates: bool = False) -> CompactBatch:
    """Same conventions as `synthetic.make_batch`, drawn as article ids into `table`."""
    rng = np.random.default_rng(seed)
    B, H, C = batch, history, candidates
    n = table.n

    def times(m):
        return pack_time(np.stack([rng.integers(0, 3, m), rng.integers(0, 13, m), rng.integers(0, 31, m), rng.integers(0, 24, m)], axis=-1))
    ha = rng.integers(1, n, (B, H)).astype(np.int32)
    ht = times(B * H).reshape(B, H)
    hc = rng.random((B, H, 2)).astype(np.float32)
    ca = rng.integers(1, n, (B, C)).astype(np.int32)
    ct = times(B * C).reshape(B, C)
    if variable_history:
        pad_h = np.arange(H)[None, :] >= rng.integers(1, H + 1, B)[:, None]
        ha[pad_h] = 0; ht[pad_h] = 0; hc[pad_h] = 0
    if variable_candidates:
        n_c = np.minimum(np.clip(np.round(np.exp(rng.normal(np.log(11.0), 0.6, B))), 5, C).astype(np.int64), C)
    else:
        n_c = np.full(B, C, dtype=np.int64)
    pad = np.arange(C)[None, :] >= n_c[:, None]
    ca[pad] = 0; ct[pad] = 0
    label = np.zeros((B, C), dtype=np.float32)
    label[np.arange(B), (rng.random(B) * n_c).astype(np.int64)] = 1.0
    t = torch.from_numpy
    return CompactBatch(t(rng.integers(1, 1 << 30, B).astype(np.int64)), t(rng.integers(0, user_num + 1, B).astype(np.int64)),
                        t(ha), t(ht.view(np.int32).copy()), t(hc), t(ca), t(ct.view(np.int32).copy()), t(label),
                        t(pad.sum(1).astype(np.int64)))
