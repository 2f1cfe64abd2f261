"""Exact fingerprint search on the device (faiss ``IndexFlatL2``) and eval.py's sequence-level hit rates.

``FingerprintIndex`` keeps a database of fingerprints resident on one GPU - the fp32 rows, their fp16 hi / lo planes
and squared norms (about 1 KiB per row at d = 128) - and answers ``search(q, k)`` with the k nearest rows in squared L2
distance through ``grafp_search_fwd``: the k-NN kernel's tensor-core Gram and fused top-k, run over key slices of the
database in parallel and merged.  ``evaluate_sequences`` computes the top-1 / near / top-3 / top-10 rates of the
reference's eval.py on such an index with one search over every query row it needs.  Approximate indexes (IVF, PQ)
are not implemented.
"""
from __future__ import annotations

import os
from typing import Iterable, Sequence, Tuple, Union

import numpy as np
import torch

from . import _native

NORM_LIMIT = 1.0 + 1e-4   # largest row norm the fp16 plane split and the selection thresholds allow
_STAGING_ROWS = 1 << 16   # rows per host -> device chunk


def _stream(device: torch.device) -> int:
    return torch.cuda.current_stream(device).cuda_stream


def _check_d(d: int) -> None:
    if d % 8 != 0 or not 64 <= d <= 256:
        raise ValueError(f"grafp_b200.search: d = {d} is not supported (a multiple of 8 in [64, 256])")


def _check_norms(x: torch.Tensor, what: str) -> None:
    """Raise ValueError if a row's L2 norm exceeds NORM_LIMIT (or is NaN); synchronises with the device."""
    if x.shape[0] == 0:
        return
    bad = ~(torch.linalg.vector_norm(x, dim=1) <= NORM_LIMIT)
    if bool(bad.any()):
        i = int(torch.nonzero(bad)[0, 0])
        raise ValueError(f"grafp_b200.FingerprintIndex.{what}: row {i} has L2 norm above {NORM_LIMIT} (or is not finite); "
                         "rows must be L2-normalised fingerprints")


class FingerprintIndex:
    """Exact squared-L2 index over fingerprints of dimension ``d`` held on ``device`` (faiss ``IndexFlatL2``).

    Precondition: every database and query row has L2 norm <= 1 + 1e-4, which unit-norm fingerprints satisfy.  ``add``
    and ``search`` check it and raise ValueError otherwise; the check synchronises with the device.

    ``d`` must be a multiple of 8 in [64, 256], ``k`` at most 128.  The index lives on a CUDA device; queries must be
    CUDA tensors (there is no CPU path), database rows may come from any device or from numpy / ``np.memmap``.
    """

    def __init__(self, d: int, device: Union[str, torch.device, None] = None):
        _check_d(int(d))
        device = torch.device("cuda") if device is None else torch.device(device)
        if device.type != "cuda":
            raise RuntimeError("grafp_b200.FingerprintIndex: the index lives on a CUDA device (there is no CPU path)")
        if device.index is None:
            device = torch.device("cuda", torch.cuda.current_device())
        self.d = int(d)
        self.device = device
        self._n = 0
        self._rows = torch.empty((0, self.d), dtype=torch.float32, device=device)
        self._hi = torch.empty((0, self.d), dtype=torch.float16, device=device)
        self._lo = torch.empty((0, self.d), dtype=torch.float16, device=device)
        self._sq = torch.empty((0,), dtype=torch.float32, device=device)
        self._staging = [None, None]
        self._staged = [None, None]

    @property
    def ntotal(self) -> int:
        """Number of database rows."""
        return self._n

    @property
    def rows(self) -> torch.Tensor:
        """The fp32 database rows (ntotal, d) on the device (a view; do not modify)."""
        return self._rows[:self._n]

    def _reserve(self, n: int) -> None:
        cap = self._rows.shape[0]
        if n <= cap:
            return
        cap = max(n, cap + cap // 2, 1024)
        with torch.cuda.device(self.device):
            for name, dt in (("_rows", torch.float32), ("_hi", torch.float16), ("_lo", torch.float16)):
                old = getattr(self, name)
                new = torch.empty((cap, self.d), dtype=dt, device=self.device)
                new[:self._n].copy_(old[:self._n])
                setattr(self, name, new)
            sq = torch.empty((cap,), dtype=torch.float32, device=self.device)
            sq[:self._n].copy_(self._sq[:self._n])
            self._sq = sq

    def _append_device(self, x: torch.Tensor) -> None:
        m = int(x.shape[0])
        if m == 0:
            return
        _check_norms(x, "add")
        self._reserve(self._n + m)
        n0 = self._n
        rows = self._rows[n0:n0 + m]
        rows.copy_(x)
        lib = _native.load()
        with torch.cuda.device(self.device):
            rc = lib.grafp_search_prepare(rows.data_ptr(), m, self.d, self._hi[n0].data_ptr(), self._lo[n0].data_ptr(),
                                          self._sq[n0:].data_ptr(), _stream(self.device))
        _native.check(rc, "FingerprintIndex.add")
        self._n = n0 + m

    def _host_chunks(self, x) -> Iterable[torch.Tensor]:
        """Device copies of host rows, chunk by chunk through two pinned staging buffers."""
        n = int(x.shape[0])
        for i, r0 in enumerate(range(0, n, _STAGING_ROWS)):
            slot = i & 1
            if self._staging[slot] is None:
                self._staging[slot] = torch.empty((_STAGING_ROWS, self.d), dtype=torch.float32).pin_memory()
            if self._staged[slot] is not None:
                self._staged[slot].synchronize()   # the copy out of this buffer two chunks ago has finished
            part = x[r0:r0 + _STAGING_ROWS]
            src = torch.from_numpy(np.ascontiguousarray(part, dtype=np.float32)) if isinstance(part, np.ndarray) \
                else part.detach().to(torch.float32)
            m = int(src.shape[0])
            buf = self._staging[slot][:m]
            buf.copy_(src)
            dev = torch.empty((m, self.d), dtype=torch.float32, device=self.device)
            dev.copy_(buf, non_blocking=True)
            ev = torch.cuda.Event()
            ev.record(torch.cuda.current_stream(self.device))
            self._staged[slot] = ev
            yield dev

    def add(self, x) -> None:
        """Append rows x (n, d): a torch tensor on any device, or a numpy array / ``np.memmap`` (read chunk by chunk,
        never held whole in host memory).  Rows are numbered in call order.  Raises ValueError for a row of norm above
        1 + 1e-4 (this synchronises); rows of earlier chunks of the same call stay added."""
        if x.ndim != 2 or int(x.shape[1]) != self.d:
            raise ValueError(f"grafp_b200.FingerprintIndex.add: expected (n, {self.d}) rows, got {tuple(x.shape)}")
        if isinstance(x, torch.Tensor) and x.is_cuda:
            self._append_device(x.detach().to(device=self.device, dtype=torch.float32))
            return
        if not isinstance(x, (torch.Tensor, np.ndarray)):
            raise TypeError(f"grafp_b200.FingerprintIndex.add: expected a torch tensor or numpy array, got {type(x)}")
        for dev in self._host_chunks(x):
            self._append_device(dev)

    def search(self, q: torch.Tensor, k: int) -> Tuple[torch.Tensor, torch.Tensor]:
        """(D, I): for every query row the k nearest database rows, as ``faiss.IndexFlatL2.search`` returns them.

        D (n_q, k) float32 squared L2 distances, computed as (|q|^2 + (-2 q.x)) + |x|^2 in fp32; I (n_q, k) int64 row
        ids.  Each row is in ascending (distance, id) order: equal distances keep the lower id.  The result of a query
        does not depend on the other queries of the batch, except that for k <= 3 on unit-norm rows two keys whose
        distances differ by less than about 1e-6 (the spread of the rows' computed |x|^2) may come back in either
        order or either one may be picked.  q must be a CUDA tensor; raises ValueError for a row of
        norm above 1 + 1e-4 (this synchronises) or k outside [1, min(128, ntotal)].
        """
        if not isinstance(q, torch.Tensor) or not q.is_cuda:
            raise RuntimeError("grafp_b200.FingerprintIndex.search: queries must be CUDA tensors (there is no CPU path)")
        if q.dim() != 2 or q.shape[1] != self.d:
            raise ValueError(f"grafp_b200.FingerprintIndex.search: expected (n_q, {self.d}) queries, got {tuple(q.shape)}")
        k = int(k)
        if not 1 <= k <= min(_native.KNN_MAX_K, self._n):
            raise ValueError(f"grafp_b200.FingerprintIndex.search: k = {k} must be in [1, min({_native.KNN_MAX_K}, "
                             f"ntotal = {self._n})]")
        q = q.detach().to(device=self.device, dtype=torch.float32).contiguous()
        n_q = int(q.shape[0])
        D = torch.empty((n_q, k), dtype=torch.float32, device=self.device)
        I = torch.empty((n_q, k), dtype=torch.int64, device=self.device)
        if n_q == 0:
            return D, I
        _check_norms(q, "search")
        lib = _native.load()
        with torch.cuda.device(self.device):   # the workspace size depends on the device's SM count
            need = lib.grafp_search_workspace_bytes(n_q, self._n, self.d, k)
            if need == 0:
                raise RuntimeError("grafp_b200.FingerprintIndex.search: " + lib.grafp_last_error().decode("utf-8", "replace"))
            ws = torch.empty((need,), dtype=torch.uint8, device=self.device)
            rc = lib.grafp_search_fwd(q.data_ptr(), n_q, self._hi.data_ptr(), self._lo.data_ptr(), self._sq.data_ptr(),
                                      self._n, self.d, k, I.data_ptr(), D.data_ptr(), ws.data_ptr(), need,
                                      _stream(self.device))
        _native.check(rc, "FingerprintIndex.search")
        return D, I


def load_index(sources: Sequence[Tuple[str, str]], device: Union[str, torch.device, None] = None) -> FingerprintIndex:
    """Index of the databases ``[(dir, name), ...]`` written by ``FingerprintWriter`` or by the reference
    (``<dir>/<name>.mm`` + ``<name>_shape.npy``), appended in list order - e.g. ``[(d, "dummy_db"), (d, "db")]`` as
    eval.py stacks them.  Each memmap is read in chunks."""
    from .inference import load_fingerprint_db
    index = None
    for source_dir, name in sources:
        data, shape = load_fingerprint_db(source_dir, name)
        if index is None:
            index = FingerprintIndex(int(shape[1]), device)
        index.add(data)
        del data
    if index is None:
        raise ValueError("grafp_b200.load_index: no sources given")
    return index


def resolve_test_ids(test_ids, n_query: int, seq_lens: Sequence[int]) -> np.ndarray:
    """``"all"`` -> arange(n_query - max(seq_lens)); a ``.npy`` path -> its contents; else the given ids (int64)."""
    if isinstance(test_ids, str):
        if test_ids == "all":
            return np.arange(max(n_query - max(seq_lens), 0), dtype=np.int64)
        if test_ids.endswith(".npy") and os.path.isfile(test_ids):
            return np.asarray(np.load(test_ids), dtype=np.int64).reshape(-1)
        raise ValueError(f"grafp_b200.evaluate_sequences: test_ids {test_ids!r} is neither 'all' nor a .npy file")
    ids = np.asarray(test_ids, dtype=np.int64).reshape(-1)
    if ids.size and (ids.min() < 0 or ids.max() >= n_query):
        raise ValueError(f"grafp_b200.evaluate_sequences: test ids must lie in [0, {n_query})")
    return ids


_RATES = ("top1_exact", "top1_near", "top3_exact", "top10_exact")


def evaluate_sequences(index: FingerprintIndex, query, test_ids, seq_lens: Sequence[int] = (1, 3, 5, 9, 11, 19),
                       k_probe: int = 20, gt_offset: int = 0, chunk: int = 256) -> dict:
    """Sequence-level hit rates of the reference's eval.py on an exact index.

    For test id t and length L, with gt = t + gt_offset and R the index rows:
      1. Q = query[t : t + L] (numpy slice semantics: shorter at the end of the queries);
      2. the exact top-``k_probe`` ids of every row of Q;
      3. row o's ids minus o, those >= 0, sorted and deduplicated, are the candidates c;
      4. score(c) = mean over o < m of Q[o] . R[c + o], m = min(len(Q), ntotal - c), products summed in fp32 as
         (a * b).sum(-1), so the result does not depend on the TF32 switches;
      5. candidates by descending score - equal scores keep the lower id (the reference's argsort leaves that order
         unspecified) - the first 10 are the prediction;
      6. flags: top1_exact pred[0] == gt, top1_near |pred[0] - gt| <= 1, top3_exact gt in pred[:3], top10_exact gt in
         pred[:10].
    One search covers every query row the test ids need; candidates and scores are batched on the device, ``chunk``
    test ids at a time.

    Returns {"top1_exact", "top1_near", "top3_exact", "top10_exact": rates in percent (float64, one per length),
    "hits": {same names: bool (n_ids, n_lens)}, "seq_lens", "test_ids"}.
    """
    dev = index.device
    if isinstance(query, np.ndarray):
        query = torch.from_numpy(np.ascontiguousarray(query, dtype=np.float32))
    if not isinstance(query, torch.Tensor) or query.dim() != 2 or query.shape[1] != index.d:
        raise ValueError(f"grafp_b200.evaluate_sequences: expected (n, {index.d}) query rows")
    seq_lens = [int(v) for v in seq_lens]
    if not seq_lens or min(seq_lens) < 1:
        raise ValueError("grafp_b200.evaluate_sequences: seq_lens must be positive")
    nq = int(query.shape[0])
    ids = resolve_test_ids(test_ids, nq, seq_lens)
    L_max = max(seq_lens)
    n_ids, n_lens = len(ids), len(seq_lens)
    hits = {name: np.zeros((n_ids, n_lens), dtype=bool) for name in _RATES}
    if n_ids:
        # the query rows some test id reads, searched once
        need = np.zeros(nq + 1, dtype=np.int64)
        np.add.at(need, ids, 1)
        np.add.at(need, np.minimum(ids + L_max, nq), -1)
        rows = np.nonzero(np.cumsum(need)[:nq] > 0)[0]
        pos = torch.full((nq,), -1, dtype=torch.int64, device=dev)
        pos[torch.from_numpy(rows).to(dev)] = torch.arange(len(rows), device=dev)
        q_dev = query.detach().to(device=dev, dtype=torch.float32)
        _, probe = index.search(q_dev[torch.from_numpy(rows).to(dev)].contiguous(), k_probe)
        R, n_db = index.rows, index.ntotal
        ids_dev = torch.from_numpy(ids).to(dev)
        big = torch.iinfo(torch.int64).max
        for li, L in enumerate(seq_lens):
            offs = torch.arange(L, device=dev)
            for c0 in range(0, n_ids, chunk):
                t = ids_dev[c0:c0 + chunk]                                  # (B,)
                r = t[:, None] + offs[None, :]                              # (B, L) query rows
                live = r < nq
                lq = live.sum(1)                                            # len(Q)
                rc = torch.where(live, r, torch.zeros_like(r))
                cand = probe[pos[rc]] - offs[None, :, None]                 # (B, L, k_probe)
                cand = torch.where(live[:, :, None] & (cand >= 0), cand, torch.full_like(cand, big))
                cand = torch.sort(cand.reshape(len(t), -1), dim=1).values   # ascending ids, invalid last
                dup = torch.zeros_like(cand, dtype=torch.bool)
                dup[:, 1:] = cand[:, 1:] == cand[:, :-1]
                valid = (cand != big) & ~dup
                c = torch.where(valid, cand, torch.zeros_like(cand))
                m = torch.minimum(lq[:, None], n_db - c)                    # rows that enter the mean
                acc = torch.zeros(c.shape, dtype=torch.float32, device=dev)
                for o in range(L):
                    use = valid & (o < m)
                    qo = q_dev[rc[:, o]]                                    # (B, d)
                    ro = R[torch.where(use, c + o, torch.zeros_like(c))]    # (B, n_cand, d)
                    acc += torch.where(use, (ro * qo[:, None, :]).sum(-1), torch.zeros_like(acc))
                score = torch.where(valid, acc / m.clamp(min=1).to(torch.float32), torch.full_like(acc, -float("inf")))
                order = torch.sort(score, dim=1, descending=True, stable=True).indices[:, :10]
                pred = torch.where(torch.gather(valid, 1, order), torch.gather(cand, 1, order), torch.full_like(order, -big))
                gt = (t + gt_offset)[:, None]
                sl = slice(c0, c0 + len(t))
                hits["top1_exact"][sl, li] = (pred[:, 0:1] == gt)[:, 0].cpu().numpy()
                hits["top1_near"][sl, li] = ((pred[:, 0:1] - gt).abs() <= 1)[:, 0].cpu().numpy()
                hits["top3_exact"][sl, li] = (pred[:, :3] == gt).any(1).cpu().numpy()
                hits["top10_exact"][sl, li] = (pred[:, :10] == gt).any(1).cpu().numpy()
    out = {name: (100.0 * hits[name].mean(0) if n_ids else np.zeros(n_lens)) for name in _RATES}
    out.update(hits=hits, seq_lens=list(seq_lens), test_ids=ids)
    return out
