"""B200-native ANN refresher — drop-in for the reference's drivers/run_ann_data_gen.py.

Same CLI flags, same inputs (`training_dir/checkpoint-N/` with scheduler.pt, `data_dir/{passages,
train-query,dev-query}` token caches + qrels) and same outputs (`output_dir/ann_training_data_N`,
`ann_ndcg_N`, `--inference` dumps), so it runs under the unmodified trainer (drivers/run_ann.py
picks the files up at run_ann.py:182-228).  What changes is where the work happens:

  reference (run_ann_data_gen.py)                       here
  ---------------------------------------------------   ------------------------------------------------
  per-record Python dataloader, batch 16 (199-202)      StridedBatchReader: memmap + numpy stride, pinned
  HF eager fp32 forward, D2H every batch (175-180)      libance_b200 encoder (tcgen05 GEMMs, fused attention);
                                                        embeddings stay in this rank's HBM
  np.save / np.load gather to rank 0 (util.py:87-146)   rows never move; ONE all-gather of query embeddings
  faiss.IndexFlatIP on rank 0, 16 threads (269-303)     per-shard sm_100a flat-IP top-k + host k-way merge
  Python loops for negatives / NDCG (339-440)           numpy (ance_b200/postprocess.py)

Row numbering is the reference's: rank r encodes records r, r+W, ...; global row = (rows of ranks
< r) + local row, i.e. the order barrier_array_merge produces (util.py:129-144); MaxP rows are
chunk-major per `per_gpu_eval_batch_size` batch (run_ann_data_gen.py:183-186).
"""
from __future__ import annotations

import argparse
import csv
import logging
import os
import random
import time
from typing import Callable, Dict, List, Optional, Tuple

import numpy as np
import torch
import torch.distributed as dist

from ..data import EmbeddingCache, StridedBatchReader
from ..models import MSMarcoConfigDict
from .. import postprocess
from ..search import MAX_K

logger = logging.getLogger(__name__)


# =============================================================================================
# bookkeeping (same behaviour as the reference helpers)
# =============================================================================================
def get_checkpoint_no(checkpoint_path: str) -> int:
    """utils/util.py:224-226."""
    import re
    nums = re.findall(r"\d+", checkpoint_path)
    return int(nums[-1]) if len(nums) > 0 else 0


def get_latest_ann_data(ann_data_path: str):
    """utils/util.py:229-243."""
    import json
    prefix = "ann_ndcg_"
    if not os.path.exists(ann_data_path):
        return -1, None, None
    files = list(next(os.walk(ann_data_path))[2])
    nos = [int(s[len(prefix):]) for s in files if s[:len(prefix)] == prefix and s[len(prefix):].isdigit()]
    if len(nos) > 0:
        no = max(nos)
        with open(os.path.join(ann_data_path, prefix + str(no)), "r") as f:
            ndcg_json = json.load(f)
        return no, os.path.join(ann_data_path, "ann_training_data_" + str(no)), ndcg_json
    return -1, None, None


def is_first_worker() -> bool:
    """utils/util.py:216-217."""
    return not dist.is_available() or not dist.is_initialized() or dist.get_rank() == 0


def _world() -> Tuple[int, int]:
    if dist.is_available() and dist.is_initialized():
        return dist.get_world_size(), dist.get_rank()
    return 1, 0


def get_latest_checkpoint(args):
    """run_ann_data_gen.py:55-71: newest `checkpoint-N` dir that already holds scheduler.pt."""
    if not os.path.exists(args.training_dir):
        return args.init_model_dir, 0
    subdirectories = list(next(os.walk(args.training_dir))[1])
    nums = [get_checkpoint_no(s) for s in subdirectories
            if os.path.exists(os.path.join(args.training_dir, s, "scheduler.pt"))]
    if len(nums) > 0:
        return os.path.join(args.training_dir, "checkpoint-" + str(max(nums))) + "/", max(nums)
    return args.init_model_dir, 0


def load_positive_ids(args):
    """run_ann_data_gen.py:74-100."""
    training_query_positive_id: Dict[int, int] = {}
    with open(os.path.join(args.data_dir, "train-qrel.tsv"), "r", encoding="utf8") as f:
        for [topicid, docid, rel] in csv.reader(f, delimiter="\t"):
            assert rel == "1"
            training_query_positive_id[int(topicid)] = int(docid)
    dev_query_positive_id: Dict[int, Dict[int, int]] = {}
    with open(os.path.join(args.data_dir, "dev-qrel.tsv"), "r", encoding="utf8") as f:
        for [topicid, docid, rel] in csv.reader(f, delimiter="\t"):
            dev_query_positive_id.setdefault(int(topicid), {})[int(docid)] = int(rel)
    return training_query_positive_id, dev_query_positive_id


# =============================================================================================
# model + encoding
# =============================================================================================
def load_model(args, checkpoint_path):
    """run_ann_data_gen.py:103-136.  No DDP wrapper: every rank loads the checkpoint itself (the
    reference wraps only to get `.module`); the tokenizer is never used on this path."""
    args.model_type = args.model_type.lower()
    configObj = MSMarcoConfigDict[args.model_type]
    args.model_name_or_path = checkpoint_path
    config = configObj.config_class.from_pretrained(
        args.config_name if args.config_name else args.model_name_or_path, num_labels=2, finetuning_task="MSMarco",
        cache_dir=args.cache_dir if args.cache_dir else None)
    model = configObj.model_class.from_pretrained(
        args.model_name_or_path, from_tf=bool(".ckpt" in args.model_name_or_path), config=config,
        cache_dir=args.cache_dir if args.cache_dir else None)
    model.to(args.device)
    model.eval()
    return config, None, model


def rows_from_batches(emb: torch.Tensor, idx: np.ndarray, batch: int) -> Tuple[torch.Tensor, np.ndarray]:
    """[n, C, d] chunk embeddings of n consecutive local records -> the reference's row layout:
    per `batch` documents, chunk-major (run_ann_data_gen.py:183-186)."""
    n, C, d = emb.shape
    rows, ids = [], []
    full = (n // batch) * batch
    if full:
        e = emb[:full].reshape(full // batch, batch, C, d).permute(0, 2, 1, 3).reshape(full * C, d)
        i = np.broadcast_to(idx[:full].reshape(full // batch, 1, batch), (full // batch, C, batch)).reshape(-1)
        rows.append(e)
        ids.append(i)
    if full < n:
        r = n - full
        rows.append(emb[full:].permute(1, 0, 2).reshape(r * C, d))
        ids.append(np.broadcast_to(idx[full:][None, :], (C, r)).reshape(-1))
    return torch.cat(rows, dim=0), np.concatenate(ids)


class B200Backend:
    """Encode + search on this rank's GPU through libance_b200."""

    def __init__(self, args, model, mask_mode: str = "lens"):
        self.args = args
        self.model = model
        self.device = args.device
        self.mask_mode = mask_mode  # "lens": 1^len 0^(L-len) (msmarco_data.py:282); "nonzero": ids != 0 (DPR_data.py:283)

    def encode(self, cache_path: str, is_query: bool, build_index: bool = False):
        """This rank's records of one token cache -> (rows [n_rows, 768] fp32 CUDA, embedding2id int64), or
        (IndexFlatIP, rows, embedding2id) with build_index.

        The rows of a rank are ONE pre-sized device tensor: every super-batch is encoded straight into its slice, and with
        build_index that tensor IS the index's fp32 storage (ance_index_create_over), each slice being added in place as
        soon as it is written.  The corpus therefore exists once in fp32 (+ once in 16 bits for the coarse pass) instead
        of the reference's per-batch arrays + concatenation + faiss copy (run_ann_data_gen.py:160-193,271)."""
        args = self.args
        W, rank = _world()
        cache = EmbeddingCache(cache_path)
        L = cache.embedding_size
        multi = (not is_query) and hasattr(self.model, "encode_lens_multi_chunk") and L > 512
        C = (L // 512) if multi else 1
        B = args.per_gpu_eval_batch_size
        # super-batch = what one encoder pass holds.  Only the MaxP row layout depends on the reference's batch size
        # (chunk-major per `per_gpu_eval_batch_size` documents, run_ann_data_gen.py:183-186): there it must be a multiple
        # of B; elsewhere B has no effect on the result and the pass is filled completely (592 x 128 tokens = whole waves
        # of 256-row GEMM tiles on 148 SMs).
        per = max(B, (args.encode_batch_tokens // L) // B * B) if multi else max(1, args.encode_batch_tokens // L)
        bucketed = self.mask_mode != "nonzero" and not multi and getattr(args, "length_buckets", True)
        varlen = bucketed and L <= 128 and getattr(args, "varlen", True) and hasattr(self.model, "encode_lens_varlen")
        if bucketed:
            per *= 8   # every length bucket of a super-batch should still fill the GPU (the encoder re-splits by tokens)
        reader = StridedBatchReader(cache, per, rank=rank, world_size=W)
        n_rows = reader.n_local * C
        dim = 768
        rows = torch.empty((max(n_rows, 1), dim), dtype=torch.float32, device=self.device)[:n_rows]
        index = None
        if build_index:
            from ..search import IndexFlatIP
            index = IndexFlatIP(dim, device=self.device, operand=args.search_operand,
                                storage=rows if n_rows else None, capacity=0 if n_rows else 1)
        ids_out: List[np.ndarray] = []
        pos = 0
        with torch.no_grad():
            for ids, lens, idx in reader:
                ids_d = ids.to(self.device, non_blocking=True)
                lens_d = lens.to(self.device, non_blocking=True)
                out = rows[pos:pos + ids.shape[0] * C]
                if self.mask_mode == "nonzero":
                    fn = self.model.query_emb if is_query else self.model.body_emb
                    out.copy_(fn(ids_d, ids_d != 0))
                    i = idx.numpy()
                elif multi:
                    e = self.model.encode_lens_multi_chunk(ids_d, lens_d)
                    e, i = rows_from_batches(e, idx.numpy(), B)
                    out.copy_(e)
                elif varlen:
                    self.model.encode_lens_varlen(ids_d, lens_d, lens_host=lens, out=out, align=getattr(args, "varlen_align", 1))
                    i = idx.numpy()
                elif bucketed:
                    self.model.encode_lens_bucketed(ids_d, lens_d, out=out)
                    i = idx.numpy()
                else:
                    self.model.encode_lens(ids_d, lens_d, out=out)
                    i = idx.numpy()
                if index is not None:
                    index.add(out)     # in place: the slice already IS index storage (no copy; operands are built by prepare())
                ids_out.append(i)
                pos += out.shape[0]
        if hasattr(self.model, "check_inputs"):
            self.model.check_inputs()   # out-of-vocabulary ids: fail like the reference's embedding lookup does
        emb2id = np.concatenate(ids_out) if ids_out else np.empty((0,), dtype=np.int64)
        return (index, rows, emb2id) if build_index else (rows, emb2id)

    def make_local_search(self, passages) -> Callable:
        """passages: an IndexFlatIP built by encode(build_index=True), or a [n, 768] CUDA tensor (copied into a new one)."""
        from ..search import IndexFlatIP
        if isinstance(passages, IndexFlatIP):
            index = passages
        else:
            index = IndexFlatIP(passages.shape[1], capacity=max(1, passages.shape[0]), device=self.device,
                                operand=self.args.search_operand)
            index.add(passages)
        self.index = index
        index.prepare()     # centred 16-bit operands of all rows (otherwise done inside the first search)
        return lambda q, k, row_offset: index.search_device(q, k, row_offset=row_offset)


# =============================================================================================
# sharded search: all-gather queries, per-shard top-k, host merge (SURVEY.md §8e)
# =============================================================================================
def _shard_sizes(n_local: int, device) -> List[int]:
    W, _ = _world()
    if W == 1:
        return [n_local]
    t = torch.tensor([n_local], dtype=torch.int64, device=device)
    out = [torch.zeros_like(t) for _ in range(W)]
    dist.all_gather(out, t)
    return [int(x.item()) for x in out]


def all_gather_rows(x: torch.Tensor) -> torch.Tensor:
    """Concatenate every rank's rows in rank order (= the merged order of util.py:129-144)."""
    W, _ = _world()
    if W == 1:
        return x
    sizes = _shard_sizes(x.shape[0], x.device)
    mx = max(sizes)
    pad = torch.zeros((mx, x.shape[1]), dtype=x.dtype, device=x.device)
    pad[:x.shape[0]] = x
    out = torch.empty((W * mx, x.shape[1]), dtype=x.dtype, device=x.device)
    dist.all_gather_into_tensor(out, pad)
    return torch.cat([out[r * mx:r * mx + sizes[r]] for r in range(W)], dim=0)


def all_gather_ids(ids: np.ndarray, device) -> np.ndarray:
    t = torch.from_numpy(np.ascontiguousarray(ids, dtype=np.int64)).to(device)
    return all_gather_rows(t[:, None])[:, 0].cpu().numpy()


#: queries per search block: four full waves of the coarse kernel on a B200 (74 CTA pairs x 256 query rows each).  One wave
#: per block (18,944) left ~28 ms of per-call latency (stream sync for the tier counters, all-to-all, staging) for every
#: 32 ms of kernels when the corpus is spread over 8 GPUs; the merge of a block still overlaps the next block's search.
QUERY_BLOCK = 75776


class _Staging:
    """Pinned host staging for one in-flight block (reused: a block's buffers are free again once its merge is done)."""

    def __init__(self, rows: int, k: int, with_scores: bool, pin: bool):
        self.D = torch.empty((rows, k), dtype=torch.float32, pin_memory=pin) if with_scores else None
        self.I = torch.empty((rows, k), dtype=torch.int64, pin_memory=pin)
        self.merged = None      # (D, I) numpy scratch of the merge of this slot's block, reused across blocks
        self.job = None


_STAGING_CACHE: Dict[tuple, list] = {}     # (rows, k, with_scores, pinned) -> sets of two buffers, kept across calls
_MERGE_POOL = None


class _StagingSet:
    def __init__(self, rows: int, k: int, with_scores: bool, pin: bool):
        self.slots = [_Staging(rows, k, with_scores, pin) for _ in range(2)]
        self.busy = False


def _staging(rows: int, k: int, with_scores: bool, pin: bool) -> "_StagingSet":
    """A free set of two staging buffers of this shape (a search in flight owns its set until `finish()`)."""
    key = (rows, k, with_scores, pin)
    sets = _STAGING_CACHE.setdefault(key, [])
    if len(_STAGING_CACHE) > 8:
        for kk in [kk for kk in _STAGING_CACHE if kk != key and not any(x.busy for x in _STAGING_CACHE[kk])]:
            del _STAGING_CACHE[kk]
    for ss in sets:
        if not ss.busy:
            break
    else:
        ss = _StagingSet(rows, k, with_scores, pin)
        sets.append(ss)
    ss.busy = True
    for st in ss.slots:
        st.job = None
    return ss


def _merge_pool():
    global _MERGE_POOL
    if _MERGE_POOL is None:
        from concurrent.futures import ThreadPoolExecutor
        _MERGE_POOL = ThreadPoolExecutor(max_workers=1)
    return _MERGE_POOL


class PendingSearch:
    """A sharded search whose device work, all-to-alls, device->host copies and merges have been issued; `finish()` waits
    for the merges and does the final gather.  Between the two the caller may enqueue more device work (bench.py encodes the
    next slice while the previous slice's lists are merged on the host).  Every rank must call `finish()` once, in the same
    order relative to its other collectives."""

    def __init__(self, **kw):
        self.__dict__.update(kw)

    def finish(self, gather_to_rank0: bool = True):
        for st in self.sset.slots:
            if st.job is not None:
                st.job.result()
                st.job = None
        self.sset.busy = False
        W, rank, nq, QB, part, k, dev, I_own = self.W, self.rank, self.nq, self.QB, self.part, self.k, self.dev, self.I_own
        if not gather_to_rank0:
            return I_own, self.q_own
        if W == 1:
            return I_own
        # final assembly on rank 0 (post-processing and the output files are rank 0's, run_ann_data_gen.py:265-336):
        # nq x k labels in total, 1/W of what a gather of the per-shard lists would move
        n_blocks = (nq + QB - 1) // QB
        mine = torch.full((n_blocks * part, k), -1, dtype=torch.int64)
        mine[:I_own.shape[0]] = torch.from_numpy(I_own)
        mine = mine.to(dev)
        if rank == 0:
            parts = [torch.empty_like(mine) for _ in range(W)]
            dist.gather(mine, parts, dst=0)
            out = np.empty((nq, k), dtype=np.int64)
            for r in range(W):
                pr = parts[r].cpu().numpy()
                row = 0
                for b0 in range(0, nq, QB):
                    nv = max(0, min(part, min(QB, nq - b0) - r * part))
                    out[b0 + r * part:b0 + r * part + nv] = pr[row:row + nv]
                    row += nv
            return out
        dist.gather(mine, None, dst=0)
        return None


def sharded_search_start(local_search: Callable, n_local_rows: int, queries_all: torch.Tensor, k: int,
                         merge_threads: int = 0, query_block: int = QUERY_BLOCK, row_offset: Optional[int] = None
                         ) -> PendingSearch:
    """Issue a sharded search (see `sharded_search`) and return without waiting for the host merges."""
    from ..search import merge_topk_host
    W, rank = _world()
    dev = queries_all.device
    cuda = dev.type == "cuda"
    offset = int(row_offset) if row_offset is not None else int(sum(_shard_sizes(n_local_rows, dev)[:rank]))
    nq = int(queries_all.shape[0])
    if k > 512:
        # above k = 512 the block shrinks so that QB * k stays at most query_block * 512: the two pinned staging slots
        # would otherwise grow with k (3.7 GB at k = 2048 and the default block)
        query_block = max(1, query_block * 512 // k)
    QB = max(W, (max(1, min(query_block, nq)) + W - 1) // W * W)      # a multiple of W: equal all-to-all splits
    part = QB // W
    side = torch.cuda.Stream(device=dev) if cuda else None
    sset = _staging(QB, k, W > 1, cuda)
    stage = sset.slots
    pool = _merge_pool()
    # the queries this rank owns: `part` of every block (all of it when W == 1); their merged labels are written straight
    # into one result array (no per-block temporaries)
    owned = [(b0 + rank * part, max(0, min(part, min(QB, nq - b0) - rank * part))) if W > 1 else (b0, min(QB, nq - b0))
             for b0 in range(0, nq, QB)]
    starts = np.concatenate([[0], np.cumsum([n for _, n in owned])]).astype(np.int64)
    I_own = np.empty((int(starts[-1]), k), dtype=np.int64)
    q_own = (np.concatenate([np.arange(q0, q0 + n, dtype=np.int64) for q0, n in owned]) if owned
             else np.empty((0,), dtype=np.int64))

    def finish_block(st: _Staging, ev, bi: int):
        if ev is not None:
            ev.synchronize()
        n_valid = owned[bi][1]
        dst = I_own[starts[bi]:starts[bi] + n_valid]
        if W == 1:
            dst[:] = st.I[:n_valid].numpy()
        elif n_valid:
            Dv, Iv = st.D.numpy().reshape(W, part, k), st.I.numpy().reshape(W, part, k)
            if st.merged is None:
                st.merged = np.empty((part, k), dtype=np.float32)       # merged scores: scratch, only the labels are kept
            merge_topk_host([Dv[s, :n_valid] for s in range(W)], [Iv[s, :n_valid] for s in range(W)], k, merge_threads,
                            out=(st.merged[:n_valid], dst))

    for bi, b0 in enumerate(range(0, nq, QB)):
        nb = min(QB, nq - b0)
        D, I = local_search(queries_all[b0:b0 + nb].contiguous(), k, offset)
        if nb < QB and W > 1:
            # ragged last block: pad the RESULTS (not the queries: an all-zero query ties with every row, which no
            # certificate can resolve, and would be sent to the brute force) so that the all-to-all splits are equal
            D = torch.cat([D, D.new_full((QB - nb, k), torch.finfo(torch.float32).min)], dim=0)
            I = torch.cat([I, I.new_full((QB - nb, k), -1)], dim=0)
        st = stage[bi % 2]
        if st.job is not None:
            st.job.result()        # the staging buffers are free again
        if W > 1:
            Dr, Ir = torch.empty_like(D), torch.empty_like(I)
            dist.all_to_all_single(Dr, D)          # Dr[s*part:(s+1)*part] = shard s's lists for my part of the block
            dist.all_to_all_single(Ir, I)
        else:
            Dr, Ir = None, I
        ev = None
        if cuda:
            side.wait_stream(torch.cuda.current_stream(dev))
            with torch.cuda.stream(side):
                if Dr is not None:
                    st.D.copy_(Dr, non_blocking=True)
                    Dr.record_stream(side)
                st.I[:Ir.shape[0]].copy_(Ir, non_blocking=True)
                Ir.record_stream(side)
                ev = torch.cuda.Event()
                ev.record(side)
        else:
            if Dr is not None:
                st.D.copy_(Dr)
            st.I[:Ir.shape[0]].copy_(Ir)
        st.job = pool.submit(finish_block, st, ev, bi)
    return PendingSearch(sset=sset, W=W, rank=rank, nq=nq, QB=QB, part=part, k=k, dev=dev, I_own=I_own, q_own=q_own)


def sharded_search(local_search: Callable, n_local_rows: int, queries_all: torch.Tensor, k: int,
                   merge_threads: int = 0, query_block: int = QUERY_BLOCK, gather_to_rank0: bool = True,
                   row_offset: Optional[int] = None) -> Optional[np.ndarray]:
    """Every rank searches its own rows for ALL queries; the per-shard top-k lists of a query are merged on the rank
    that OWNS the query, so the merge (and its device->host copy) is spread over all ranks instead of serialised on
    rank 0, and it overlaps the search of the next query block:

        for each block of `query_block` queries                        (device work on the current stream)
            D, I = local_search(block)                                   per-shard top-k, labels already global
            all_to_all(D), all_to_all(I)                                 rank r receives the W lists of ITS 1/W of the block
            async D2H into pinned staging  ->  host k-way merge (C++, worker thread)      || next block's search

    Returns I [nq, k] (global rows, merged order) on rank 0 and None elsewhere; with gather_to_rank0=False every rank
    gets the merged lists of the queries it owns as (I_own [n_own, k], own_query_numbers).  row_offset: global number
    of this rank's first row (= rows of the ranks before it); computed with one small all-gather when not given."""
    return sharded_search_start(local_search, n_local_rows, queries_all, k, merge_threads, query_block,
                                row_offset).finish(gather_to_rank0)


# =============================================================================================
# one refresh
# =============================================================================================
def _dump(args, prefix: str, emb: torch.Tensor, emb2id: np.ndarray):
    """`--inference` dumps under the reference's names (util.py:108-113, run_ann_data_gen.py:213-226)."""
    _, rank = _world()
    os.makedirs(args.output_dir, exist_ok=True)
    np.save(os.path.join(args.output_dir, "{}_emb_p__data_obj_{}.npy".format(prefix, rank)), emb.cpu().numpy(),
            allow_pickle=False)
    np.save(os.path.join(args.output_dir, "{}_embid_p__data_obj_{}.npy".format(prefix, rank)), emb2id,
            allow_pickle=False)


def generate_new_ann(args, output_num, checkpoint_path, training_query_positive_id, dev_query_positive_id,
                     latest_step_num, backend=None):
    """run_ann_data_gen.py:231-336."""
    t_start = time.time()
    detail: Dict[str, float] = {}

    def lap(name, t0):
        if torch.cuda.is_available():
            torch.cuda.synchronize()
        detail[name] = time.time() - t0
        return time.time()

    if backend is None:
        _, _, model = load_model(args, checkpoint_path)
        backend = B200Backend(args, model)
    step = str(latest_step_num)

    t = time.time()
    logger.info("***** inference of dev query *****")
    dev_emb, dev_ids = backend.encode(os.path.join(args.data_dir, "dev-query"), True)
    t = lap("encode_dev_query_s", t)
    logger.info("***** inference of passages *****")
    index, p_emb, p_ids = backend.encode(os.path.join(args.data_dir, "passages"), False, build_index=True)
    t = lap("encode_passages_s", t)
    logger.info("***** Done passage inference *****")
    if args.inference:
        _dump(args, "dev_query_" + step + "_", dev_emb, dev_ids)
        _dump(args, "passage_" + step + "_", p_emb, p_ids)
        return None
    logger.info("***** inference of train query *****")
    q_emb, q_ids = backend.encode(os.path.join(args.data_dir, "train-query"), True)
    t = lap("encode_train_query_s", t)
    t_enc = time.time()

    device = p_emb.device
    local_search = backend.make_local_search(index)
    passage_embedding2id = all_gather_ids(p_ids, device)
    dev_all, dev_query_embedding2id = all_gather_rows(dev_emb), all_gather_ids(dev_ids, device)
    q_all, query_embedding2id = all_gather_rows(q_emb), all_gather_ids(q_ids, device)
    t = lap("all_gather_s", t)

    row_offset = int(sum(_shard_sizes(p_emb.shape[0], device)[:_world()[1]]))
    dev_I = sharded_search(local_search, p_emb.shape[0], dev_all, 100, row_offset=row_offset)   # run_ann_data_gen.py:276
    t = lap("search_dev_s", t)
    q_start, q_end = postprocess.query_chunk(q_all.shape[0], output_num, args.ann_chunk_factor)
    q_all, query_embedding2id = q_all[q_start:q_end], query_embedding2id[q_start:q_end]
    logger.info("Chunked {} query from {}".format(q_end - q_start, q_emb.shape[0]))
    I = sharded_search(local_search, p_emb.shape[0], q_all.contiguous(), args.topk_training, row_offset=row_offset)  # :303
    t = lap("search_train_s", t)
    t_search = time.time()
    if not is_first_worker():
        return None

    dev_ndcg, num_queries_dev = postprocess.eval_dev_query(dev_query_embedding2id, passage_embedding2id,
                                                           dev_query_positive_id, dev_I)
    print("Rank:" + str(getattr(args, "rank", 0)) + " --- ANN NDCG@10:" + str(dev_ndcg))
    t = lap("post_ndcg_s", t)
    sampler = "reference" if args.reference_sampling else "fast"
    arrays = sampler == "fast"        # array form + native line writer; the reference sampler keeps the dict / Python path
    negatives, mrr, nq = postprocess.generate_negatives(
        query_embedding2id, passage_embedding2id, training_query_positive_id, I, args.negative_sample,
        select_topk=args.ann_measure_topk_mrr, sampler=sampler, seed=args.seed, as_arrays=arrays)
    if args.ann_measure_topk_mrr:
        print("Rank:" + str(getattr(args, "rank", 0)) + " --- ANN MRR:" + str(mrr / max(nq, 1)))
    t = lap("post_negatives_s", t)
    logger.info("***** Construct ANN Triplet *****")
    os.makedirs(args.output_dir, exist_ok=True)
    data_path = os.path.join(args.output_dir, "ann_training_data_" + str(output_num))
    if arrays:
        postprocess.write_training_data_arrays(data_path, query_embedding2id, training_query_positive_id, negatives[0],
                                               negatives[1], seed=args.seed)
    else:
        postprocess.write_training_data(data_path, query_embedding2id, training_query_positive_id, negatives,
                                        sampler=sampler, seed=args.seed)
    postprocess.write_ndcg(os.path.join(args.output_dir, "ann_ndcg_" + str(output_num)), dev_ndcg, checkpoint_path)
    lap("post_write_s", t)
    args.last_refresh_timing = {"encode_s": t_enc - t_start, "search_s": t_search - t_enc, "post_s": time.time() - t_search,
                                "detail": detail, "search_stats": index.stats() if index.ntotal else None}
    logger.info("refresh %d: encode %.1fs search %.1fs post %.1fs", output_num, t_enc - t_start, t_search - t_enc,
                time.time() - t_search)
    return dev_ndcg, num_queries_dev


# =============================================================================================
# CLI (flags of run_ann_data_gen.py:443-627, plus three B200 knobs at the end)
# =============================================================================================
def topk_training_arg(value: str) -> int:
    """argparse type of --topk_training: checked when the arguments are parsed, not after the corpus has been encoded."""
    k = int(value)
    if not 1 <= k <= MAX_K:
        raise argparse.ArgumentTypeError("must be in [1, %d] (the largest k the search supports), got %d" % (MAX_K, k))
    return k


def get_arguments(argv=None):
    p = argparse.ArgumentParser()
    p.add_argument("--data_dir", default=None, type=str, required=True)
    p.add_argument("--training_dir", default=None, type=str, required=True)
    p.add_argument("--init_model_dir", default=None, type=str, required=True)
    p.add_argument("--last_checkpoint_dir", default="", type=str)
    p.add_argument("--model_type", default=None, type=str, required=True,
                   help="Model type selected in the list: " + ", ".join(MSMarcoConfigDict.keys()))
    p.add_argument("--output_dir", default=None, type=str, required=True)
    p.add_argument("--cache_dir", default=None, type=str, required=True)
    p.add_argument("--end_output_num", default=-1, type=int)
    p.add_argument("--max_seq_length", default=128, type=int)
    p.add_argument("--max_query_length", default=64, type=int)
    p.add_argument("--max_doc_character", default=10000, type=int)
    p.add_argument("--per_gpu_eval_batch_size", default=128, type=int)
    p.add_argument("--ann_chunk_factor", default=5, type=int)
    p.add_argument("--topk_training", default=500, type=topk_training_arg,
                   help="neighbours searched per training query, 1 .. %d" % MAX_K)
    p.add_argument("--negative_sample", default=5, type=int)
    p.add_argument("--ann_measure_topk_mrr", default=False, action="store_true")
    p.add_argument("--only_keep_latest_embedding_file", default=False, action="store_true")
    p.add_argument("--no_cuda", action="store_true")
    p.add_argument("--local_rank", type=int, default=-1)
    p.add_argument("--server_ip", type=str, default="")
    p.add_argument("--server_port", type=str, default="")
    p.add_argument("--inference", default=False, action="store_true")
    p.add_argument("--config_name", default="", type=str)
    p.add_argument("--tokenizer_name", default="", type=str)
    # B200 knobs (not in the reference)
    p.add_argument("--search_operand", default="auto", choices=["auto", "fp16", "bf16"],
                   help="16-bit operand format of the coarse tensor-core pass (results are exact either way); auto = fp16, "
                        "falling back to bf16 when a row or a query leaves the fp16 range")
    p.add_argument("--encode_batch_tokens", default=75776, type=int, help="tokens per encoder launch sequence")
    p.add_argument("--reference_sampling", default=False, action="store_true",
                   help="draw the negative-sampling order from Python's `random` exactly as the reference does")
    p.add_argument("--seed", default=None, type=int, help="seed for the sampling order (reference: unseeded)")
    p.add_argument("--poll_seconds", default=60, type=int)
    p.add_argument("--varlen_align", default=1, type=int, choices=[1, 16],
                   help="16: every sequence starts at a multiple of 16 rows of its attention tile, which makes its embedding "
                        "bit-identical to the padded forward and independent of batch composition / world size; 1 (default) "
                        "packs ~12 %% more real tokens per tile, embeddings agree to fp32 summation order")
    p.add_argument("--no_varlen", dest="varlen", action="store_false",
                   help="L <= 128 caches: group sequences into padded length buckets instead of packing whole sequences of any "
                        "length into 128-token attention tiles (same embeddings up to fp32 summation order)")
    p.add_argument("--no_length_buckets", dest="length_buckets", action="store_false",
                   help="encode every sequence at the cache's full padded length (the reference's behaviour); by default "
                        "sequences are grouped by the smallest supported padded length, which yields the same embeddings")
    return p.parse_args(argv)


def set_env(args):
    """run_ann_data_gen.py:630-660.  torchrun exports LOCAL_RANK; the legacy launcher passes --local_rank."""
    if args.local_rank == -1 and "LOCAL_RANK" in os.environ and int(os.environ.get("WORLD_SIZE", "1")) > 1:
        args.local_rank = int(os.environ["LOCAL_RANK"])
    if args.no_cuda or not torch.cuda.is_available():
        raise RuntimeError("ance_b200 has no CPU fallback: the refresher needs an sm_100 GPU (drop --no_cuda)")
    if args.local_rank == -1:
        args.device = torch.device("cuda", torch.cuda.current_device())
        args.n_gpu = 1
    else:
        torch.cuda.set_device(args.local_rank)
        args.device = torch.device("cuda", args.local_rank)
        if not dist.is_initialized():
            dist.init_process_group(backend="nccl")
        args.n_gpu = 1
        args.world_size = dist.get_world_size()
    args.rank = _world()[1]
    _warm_collectives(args.device)
    logging.basicConfig(format="%(asctime)s - %(levelname)s - %(name)s -   %(message)s", datefmt="%m/%d/%Y %H:%M:%S",
                        level=logging.INFO if args.local_rank in [-1, 0] else logging.WARN)
    if args.seed is not None:
        random.seed(args.seed)


def _warm_collectives(device) -> None:
    """Process start-up, like the reference's DDP wrap (run_ann_data_gen.py:128-135): the first all-gather / all-to-all
    on an NCCL communicator sets up its rings and the peer-to-peer channels of every pair of ranks (seconds on 8 GPUs).
    Done once here so that it is not billed to the first refresh's search."""
    W, _ = _world()
    if W == 1:
        return
    x = torch.zeros((W, 8), dtype=torch.float32, device=device)
    y = torch.empty((W * W, 8), dtype=torch.float32, device=device)
    dist.all_gather_into_tensor(y, x)
    z = torch.empty_like(x)
    dist.all_to_all_single(z, x)
    zi = torch.empty((W, 8), dtype=torch.int64, device=device)
    dist.all_to_all_single(zi, torch.zeros_like(zi))
    dist.gather(x, [torch.empty_like(x) for _ in range(W)] if _world()[1] == 0 else None, dst=0)
    if device.type == "cuda":
        torch.cuda.synchronize(device)


def ann_data_gen(args, backend=None):
    """run_ann_data_gen.py:663-702."""
    last_checkpoint = args.last_checkpoint_dir
    ann_no, _, _ = get_latest_ann_data(args.output_dir)
    output_num = ann_no + 1
    logger.info("starting output number %d", output_num)
    if is_first_worker():
        os.makedirs(args.output_dir, exist_ok=True)
        os.makedirs(args.cache_dir, exist_ok=True)
    training_positive_id, dev_positive_id = load_positive_ids(args)
    while args.end_output_num == -1 or output_num <= args.end_output_num:
        next_checkpoint, latest_step_num = get_latest_checkpoint(args)
        if args.only_keep_latest_embedding_file:
            latest_step_num = 0
        if next_checkpoint == last_checkpoint:
            time.sleep(args.poll_seconds)
        else:
            logger.info("start generate ann data number %d", output_num)
            logger.info("next checkpoint at " + next_checkpoint)
            generate_new_ann(args, output_num, next_checkpoint, training_positive_id, dev_positive_id, latest_step_num,
                             backend=backend)
            if args.inference:
                break
            logger.info("finished generating ann data number %d", output_num)
            output_num += 1
            last_checkpoint = next_checkpoint
        if dist.is_available() and dist.is_initialized():
            dist.barrier()


def main(argv=None):
    args = get_arguments(argv)
    set_env(args)
    ann_data_gen(args)


if __name__ == "__main__":
    main()
