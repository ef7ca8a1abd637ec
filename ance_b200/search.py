"""faiss.IndexFlatIP-shaped front end of the sm_100a flat inner-product search.

Mirrors the three calls the reference makes (drivers/run_ann_data_gen.py:269-276,303):

    cpu_index = faiss.IndexFlatIP(dim); cpu_index.add(passage_embedding)
    _, I = cpu_index.search(query_embedding, top_k)

``IndexFlatIP`` accepts numpy arrays (host, as the reference passes) or CUDA torch tensors (no
copy).  The multi-GPU form of SURVEY.md §8(e) — rows stay on the rank that encoded them, queries are
all-gathered once, per-shard top-k lists are merged on the host with ``merge_topk_host`` — lives in
``ance_b200.drivers.run_ann_data_gen.sharded_search``.
There is no CPU fallback: without libance_b200.so and an sm_100 GPU every call raises.
"""
from __future__ import annotations

import ctypes as C
from typing import Optional, Tuple

import numpy as np
import torch

from . import _lib

#: largest k a search accepts (ance_index_search / ance_index_search_exact; faiss's GPU flat index has the same limit)
MAX_K = 2048


def _as_f32_cuda(x, device) -> torch.Tensor:
    if isinstance(x, np.ndarray):
        if x.dtype != np.float32:
            raise TypeError(f"expected float32 (as faiss does), got {x.dtype}")
        x = torch.from_numpy(np.ascontiguousarray(x))
    if not isinstance(x, torch.Tensor):
        raise TypeError(f"expected numpy array or torch tensor, got {type(x)}")
    if x.dtype != torch.float32:
        raise TypeError(f"expected float32, got {x.dtype}")
    if x.dim() != 2:
        raise ValueError(f"expected a 2-D array, got shape {tuple(x.shape)}")
    if x.device.type != "cuda":
        x = x.pin_memory() if x.numel() else x
        x = x.to(device, non_blocking=True)
    return x.contiguous()


class IndexFlatIP:
    """Exact maximum-inner-product search over fp32 rows resident in HBM."""

    def __init__(self, d: int, capacity: int = 0, device: Optional[torch.device] = None,
                 operand: str = "auto", storage: Optional[torch.Tensor] = None):
        """operand: 16-bit format of the coarse tensor-core pass — "fp16" (certificate error bound ~8x tighter than bf16:
        fewer candidates to rescore), "bf16" (any fp32 range), or "auto" = fp16, switching the whole index to bf16 the
        first time a row or a query does not fit the fp16 range.  Results are exact either way.
        storage: a CUDA fp32 tensor [capacity, d] to use as the index's row storage (kept alive by the index).  Rows
        written into `storage[i:i+n]` by their producer and then passed to add() are added without a copy."""
        if not torch.cuda.is_available():
            raise _lib.AnceError("ance_b200.IndexFlatIP needs a CUDA device (sm_100); there is no CPU fallback")
        self._lib = _lib.load()
        self.d = int(d)
        self.device = torch.device(device) if device is not None else torch.device("cuda", torch.cuda.current_device())
        self.auto_operand = operand == "auto"
        self.operand = {"bf16": _lib.ANCE_FMT_BF16, "fp16": _lib.ANCE_FMT_FP16, "auto": _lib.ANCE_FMT_FP16}[operand]
        self._h = None
        self._capacity = 0
        self.ntotal = 0
        self.storage = None
        if storage is not None:
            if (storage.device.type != "cuda" or storage.dtype != torch.float32 or storage.dim() != 2
                    or storage.shape[1] != self.d or not storage.is_contiguous()):
                raise ValueError("storage must be a contiguous CUDA float32 tensor [capacity, d]")
            self.device = storage.device
            self.storage = storage
            capacity = storage.shape[0]
        if capacity:
            self._create(int(capacity))

    # -- storage -----------------------------------------------------------------------------------
    def _create(self, capacity: int):
        h = C.c_void_p()
        with torch.cuda.device(self.device):
            if self.storage is not None:
                _lib.check(self._lib.ance_index_create_over(self.d, capacity, self.operand, self.storage.data_ptr(),
                                                            C.byref(h)))
            else:
                _lib.check(self._lib.ance_index_create(self.d, capacity, self.operand, C.byref(h)))
        self._h = h
        self._capacity = capacity

    def __del__(self):
        try:
            if self._h is not None:
                self._lib.ance_index_destroy(self._h)
                self._h = None
        except Exception:
            pass

    def reset(self):
        if self._h is not None:
            _lib.check(self._lib.ance_index_reset(self._h))
        self.ntotal = 0

    def set_param(self, name: str, value: float):
        if self._h is None:
            raise _lib.AnceError("set_param before add(): create the index with a capacity")
        _lib.check(self._lib.ance_index_set_param(self._h, name.encode(), float(value)))

    def add(self, x):
        """IndexFlatIP.add: append rows.  Without a preset capacity the first add() sizes the index
        (the reference adds the whole corpus in one call, run_ann_data_gen.py:271)."""
        n = int(x.shape[0])
        if n == 0:
            return
        if x.shape[1] != self.d:
            raise ValueError(f"dimension mismatch: index {self.d}, rows {x.shape[1]}")
        if self._h is None:
            self._create(n)
        if self.ntotal + n > self._capacity:
            raise _lib.AnceError(f"index capacity {self._capacity} exceeded ({self.ntotal} + {n}); "
                                 "pass capacity= at construction")
        with torch.cuda.device(self.device):
            step = 1 << 20 if not (isinstance(x, torch.Tensor) and x.device.type == "cuda") else n
            for s in range(0, n, step):
                xs = _as_f32_cuda(x[s:s + step], self.device)
                _lib.check(self._lib.ance_index_add(self._h, xs.data_ptr(), xs.shape[0], _lib.current_stream()))
                self.ntotal += xs.shape[0]
            if step != n:   # host input: the pinned staging tensors must outlive their copies
                torch.cuda.current_stream().synchronize()

    def prepare(self):
        """Build the coarse pass's 16-bit operands from all rows added so far (centred on their mean, rounded to the
        operand format).  search() does it on demand; calling it keeps the cost out of the first search."""
        if self._h is not None and self.ntotal:
            with torch.cuda.device(self.device):
                _lib.check(self._lib.ance_index_prepare(self._h, _lib.current_stream()))

    # -- search ------------------------------------------------------------------------------------
    def search_device(self, q: torch.Tensor, k: int, row_offset: int = 0, exact: bool = False
                      ) -> Tuple[torch.Tensor, torch.Tensor]:
        """Q [nq, d] fp32 CUDA -> (D [nq, k] fp32, I [nq, k] int64), both CUDA, stream-ordered.  1 <= k <= MAX_K."""
        if int(k) > MAX_K:
            # checked here too: an empty index or query batch never reaches the library, which refuses such a k
            raise _lib.AnceError(f"k = {k} exceeds the largest supported k, {MAX_K}")
        nq = int(q.shape[0])
        D = torch.empty((nq, k), dtype=torch.float32, device=self.device)
        I = torch.empty((nq, k), dtype=torch.int64, device=self.device)
        if nq == 0:
            return D, I
        if self._h is None or self.ntotal == 0:
            D.fill_(torch.finfo(torch.float32).min)
            I.fill_(-1)
            return D, I
        fn = self._lib.ance_index_search_exact if exact else self._lib.ance_index_search
        with torch.cuda.device(self.device):
            rc = fn(self._h, q.data_ptr(), nq, int(k), D.data_ptr(), I.data_ptr(), int(row_offset),
                    _lib.current_stream())
            if rc == _lib.ANCE_ERR_UNSUPPORTED and self.auto_operand and self.operand == _lib.ANCE_FMT_FP16:
                # a row or a query left the fp16 range: re-round the index to bf16 (from its fp32 rows) and retry once;
                # inf / NaN in the data fails again and raises
                self.set_param("operand_fmt", _lib.ANCE_FMT_BF16)
                self.operand = _lib.ANCE_FMT_BF16
                rc = fn(self._h, q.data_ptr(), nq, int(k), D.data_ptr(), I.data_ptr(), int(row_offset),
                        _lib.current_stream())
            _lib.check(rc)
        return D, I

    def search(self, x, k: int):
        """IndexFlatIP.search: returns (D, I) as numpy arrays for numpy input (the reference's
        usage) or CUDA tensors for CUDA input."""
        was_numpy = isinstance(x, np.ndarray)
        if x.shape[1] != self.d:
            raise ValueError(f"dimension mismatch: index {self.d}, queries {x.shape[1]}")
        with torch.cuda.device(self.device):
            q = _as_f32_cuda(x, self.device)
            D, I = self.search_device(q, k)
            if was_numpy or x.device.type != "cuda":
                D, I = D.cpu(), I.cpu()
                return (D.numpy(), I.numpy()) if was_numpy else (D, I)
            return D, I

    def stats(self) -> dict:
        s = _lib.SearchStats()
        _lib.check(self._lib.ance_index_last_stats(self._h, C.byref(s)))
        return {n: getattr(s, n) for n, _ in s._fields_}


def merge_topk_host(Ds, Is, k: int, n_threads: int = 0, out=None):
    """Host k-way merge of per-shard (D, I) numpy arrays [nq, k] -> (D, I) [nq, k].  out: optional (D_out, I_out) arrays to
    write into (reused buffers: a fresh 6 MB result costs more in first-touch page faults than the merge itself)."""
    lib = _lib.load()
    n = len(Ds)
    if n == 0 or n != len(Is):
        raise ValueError("need the same non-zero number of D and I shards")
    Ds = [np.ascontiguousarray(d, dtype=np.float32) for d in Ds]
    Is = [np.ascontiguousarray(i, dtype=np.int64) for i in Is]
    nq = Ds[0].shape[0]
    for d, i in zip(Ds, Is):
        if d.shape != (nq, k) or i.shape != (nq, k):
            raise ValueError(f"every shard must be [{nq}, {k}]")
    if out is not None:
        Do, Io = out
        if Do.shape != (nq, k) or Io.shape != (nq, k) or Do.dtype != np.float32 or Io.dtype != np.int64 \
                or not Do.flags.c_contiguous or not Io.flags.c_contiguous:
            raise ValueError("out must be C-contiguous (float32 [nq, k], int64 [nq, k])")
    else:
        Do = np.empty((nq, k), dtype=np.float32)
        Io = np.empty((nq, k), dtype=np.int64)
    dp = (C.c_void_p * n)(*[d.ctypes.data for d in Ds])
    ip = (C.c_void_p * n)(*[i.ctypes.data for i in Is])
    _lib.check(lib.ance_merge_topk_host(dp, ip, n, nq, k, Do.ctypes.data, Io.ctypes.data, n_threads))
    return Do, Io


def omp_set_num_threads(n: int) -> None:
    """faiss.omp_set_num_threads (run_ann_data_gen.py:269): meaningless on the GPU, kept so that
    ``from ance_b200 import search as faiss`` is a drop-in for the reference's call sites."""
    return None
