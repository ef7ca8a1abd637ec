"""Offline evaluation of `--inference` dumps — the metrics half of SURVEY.md §8(f) row 4.

Replaces cells 8-13 of the reference's `evaluation/Calculate Metrics.ipynb` (and the sharded MRR of
utils/eval_mrr.py:127-203): load the per-rank dumps the refresher writes under the reference's names, then

  full-rank   `faiss.IndexFlatIP(dim).add(passage_embedding); search(dev_query_embedding, topN)`   (cell 13)
              -> ance_b200.search.IndexFlatIP on the GPU (exact top-N, deterministic tie order)
  rerank      per query, an exact ranking of its first-stage (BM25) candidates only               (cell 11)
              -> canonical scores (fp32 inputs, fp64 accumulate) of the candidate rows, (score desc, row asc)
  metrics     the notebook's EvalDevQuery (cell 8): NDCG@10, MAP@10, MRR (trec recip_rank), recall@topN, hole rate@10,
              hole rate, and MS MARCO MRR@10 (utils/msmarco_eval.py:109-139)

The trec_eval measures come from pytrec_eval in the notebook (unpinned, not installed here); they are restated from
trec_eval's definitions: gain = relevance label, discount log2(rank + 1), ideal ranking over the judged documents;
num_rel = judged documents with label > 0.  Rankings use score = -rank as the notebook does, so there are no ties.
"""
from __future__ import annotations

import math
import os
from typing import Dict, List, Optional, Sequence, Tuple

import numpy as np

from .postprocess import _first_occurrence, ndcg_cut

MaxMRRRank = 10   # utils/msmarco_eval.py:12


def load_dumps(output_dir: str, prefix: str, max_ranks: int = 64) -> Tuple[np.ndarray, np.ndarray]:
    """Concatenate `{prefix}_emb_p__data_obj_{rank}.npy` / `{prefix}_embid_p__data_obj_{rank}.npy` over ranks 0, 1, ...
    (the merged order of utils/util.py:129-144; notebook cell 9 — which looks for `.pb` pickles the reference never
    writes, SURVEY.md §8(f)4: `.npy` is what `barrier_array_merge` and this package's `--inference` produce).
    prefix e.g. "dev_query_0_" / "passage_0_"."""
    embs, ids = [], []
    for r in range(max_ranks):
        pe = os.path.join(output_dir, "{}_emb_p__data_obj_{}.npy".format(prefix, r))
        pi = os.path.join(output_dir, "{}_embid_p__data_obj_{}.npy".format(prefix, r))
        if not (os.path.exists(pe) and os.path.exists(pi)):
            break
        embs.append(np.load(pe, mmap_mode="r"))
        ids.append(np.load(pi))
    if not embs:
        raise FileNotFoundError("no dumps named {}_emb_p__data_obj_*.npy under {}".format(prefix, output_dir))
    return np.concatenate(embs, axis=0), np.concatenate(ids, axis=0)


def msmarco_mrr(qids_to_relevant: Dict[int, Sequence[int]], qids_to_ranked: Dict[int, Sequence[int]]) -> float:
    """utils/msmarco_eval.py:109-139: MRR@10 = sum over ranked queries with judgements of 1 / (rank of the first relevant
    passage within the top 10), divided by the number of JUDGED queries."""
    total, seen = 0.0, 0
    for qid, cand in qids_to_ranked.items():
        rel = qids_to_relevant.get(qid)
        if rel is None:
            continue
        seen += 1
        rel = set(rel)
        for i in range(min(MaxMRRRank, len(cand))):
            if cand[i] in rel:
                total += 1.0 / (i + 1)
                break
    if seen == 0:
        raise IOError("No matching QIDs found. Are you sure you are scoring the evaluation set?")
    return total / len(qids_to_relevant)


def eval_dev_query_full(query_embedding2id: np.ndarray, passage_embedding2id: np.ndarray,
                        dev_query_positive_id: Dict[int, Dict[int, int]], I_nearest_neighbor, topN: int) -> Dict[str, float]:
    """The notebook's EvalDevQuery (cell 8).  I_nearest_neighbor: [nq, >= topN] row labels, or a list of per-query label
    arrays (rerank: as many as the query has candidates).  Duplicate pids (several vectors per document) keep their
    first occurrence.  Queries are scored if they have an entry in dev_query_positive_id (pytrec_eval evaluates the
    intersection of run and qrel)."""
    p2id = np.asarray(passage_embedding2id).reshape(-1)
    qids = np.asarray(query_embedding2id).reshape(-1)
    ranked_lists: Dict[int, np.ndarray] = {}
    total = labeled = a_total = a_labeled = 0
    for r in range(len(I_nearest_neighbor)):
        lab = np.asarray(I_nearest_neighbor[r])[:topN]
        if lab.size and (lab < 0).any():
            raise IndexError("search returned -1 labels (fewer rows than topN)")
        pids = p2id[lab]
        ranked = pids[_first_occurrence(pids[None, :])[0]] if pids.size else pids
        qid = int(qids[r])
        ranked_lists[qid] = ranked     # duplicate qids: last wins, as the notebook's dict assignment does
        pos = dev_query_positive_id.get(qid, {})
        unjudged = np.fromiter((int(p) not in pos for p in ranked), dtype=bool, count=len(ranked))
        a_total += len(ranked)
        a_labeled += int(unjudged.sum())
        total += min(10, len(ranked))
        labeled += int(unjudged[:10].sum())
    ndcg = Map = mrr = recall = 0.0
    n = 0
    for qid, ranked in ranked_lists.items():
        qrel = dev_query_positive_id.get(qid)
        if qrel is None:
            continue
        n += 1
        num_rel = sum(1 for v in qrel.values() if v > 0)
        ndcg += ndcg_cut(ranked, qrel, 10)
        hits, ap, rr, found = 0, 0.0, 0.0, 0
        for i, p in enumerate(ranked.tolist()):
            if qrel.get(int(p), 0) > 0:
                found += 1
                if rr == 0.0:
                    rr = 1.0 / (i + 1)
                if i < 10:
                    hits += 1
                    ap += hits / (i + 1)
        Map += ap / num_rel if num_rel else 0.0
        mrr += rr
        recall += found / num_rel if num_rel else 0.0
    if n == 0:
        raise ZeroDivisionError("no dev query has a qrel")
    relevant = {int(q): [p for p, v in d.items() if p > 0] for q, d in dev_query_positive_id.items()}   # notebook: `if pid>0`
    padded = {q: (r.tolist() + [0] * 1000)[:1000] for q, r in ranked_lists.items()}
    return {"ndcg@10": ndcg / n, "eval_query_cnt": n, "map@10": Map / n, "mrr": mrr / n, "recall@%d" % topN: recall / n,
            "hole_rate@10": labeled / total if total else math.nan, "hole_rate": a_labeled / a_total if a_total else math.nan,
            "ms_mrr@10": msmarco_mrr(relevant, padded)}


def full_rank(dev_query_embedding: np.ndarray, passage_embedding: np.ndarray, topN: int, device=None,
              block_rows: int = 1 << 20) -> np.ndarray:
    """Notebook cell 13 on the GPU: exact top-N labels of every dev query over the whole (merged) passage matrix.
    topN up to ance_b200.search.MAX_K (2048): the notebook's 1000 for MS MARCO passage runs as is."""
    import torch
    from .search import IndexFlatIP
    dev = device or torch.device("cuda", torch.cuda.current_device())
    index = IndexFlatIP(passage_embedding.shape[1], capacity=max(1, passage_embedding.shape[0]), device=dev)
    for s in range(0, passage_embedding.shape[0], block_rows):
        index.add(np.ascontiguousarray(passage_embedding[s:s + block_rows], dtype=np.float32))
    _, I = index.search(np.ascontiguousarray(dev_query_embedding, dtype=np.float32), topN)
    return I


def rerank(dev_query_embedding: np.ndarray, dev_query_embedding2id: np.ndarray, passage_embedding: np.ndarray,
           passage_embedding2id: np.ndarray, first_stage: Dict[int, Sequence[int]]) -> List[np.ndarray]:
    """Notebook cell 11: for each dev query an exact ranking of its first-stage candidate passages only (all index rows
    of each candidate pid, in candidate order).  Scores are canonical (fp64-accumulated); ties keep candidate order,
    which is what a flat index over the candidate subset returns for equal scores under this package's tie rule."""
    p2id = np.asarray(passage_embedding2id).reshape(-1)
    order = np.argsort(p2id, kind="stable")
    sorted_ids = p2id[order]
    out: List[np.ndarray] = []
    for i, qid in enumerate(np.asarray(dev_query_embedding2id).reshape(-1).tolist()):
        cand = np.asarray(first_stage.get(int(qid), ()), dtype=p2id.dtype)
        lo, hi = np.searchsorted(sorted_ids, cand, "left"), np.searchsorted(sorted_ids, cand, "right")
        rows = np.concatenate([order[a:b] for a, b in zip(lo.tolist(), hi.tolist())]) if cand.size else np.empty(0, np.int64)
        if rows.size == 0:
            out.append(rows.astype(np.int64))
            continue
        s = (np.asarray(passage_embedding[np.sort(rows)], dtype=np.float64) @ np.asarray(dev_query_embedding[i], dtype=np.float64))
        s = s[np.argsort(np.argsort(rows, kind="stable"), kind="stable")].astype(np.float32)   # back to candidate order
        out.append(rows[np.argsort(-s, kind="stable")].astype(np.int64))
    return out


def evaluate_dumps(output_dir: str, step: int, dev_query_positive_id: Dict[int, Dict[int, int]], topN: int = 1000,
                   first_stage: Optional[Dict[int, Sequence[int]]] = None) -> Dict[str, Dict[str, float]]:
    """Everything cells 9-13 print, from the dumps of `run_ann_data_gen --inference` at checkpoint `step`.  The default
    topN = 1000 is the notebook's full-rank depth for MS MARCO passage (Recall@1k); any topN <= 2048 is searched exactly."""
    q, q2id = load_dumps(output_dir, "dev_query_{}_".format(step))
    p, p2id = load_dumps(output_dir, "passage_{}_".format(step))
    res = {"full_rank": eval_dev_query_full(q2id, p2id, dev_query_positive_id, full_rank(q, p, min(topN, p.shape[0])), topN)}
    if first_stage:
        res["rerank"] = eval_dev_query_full(q2id, p2id, dev_query_positive_id, rerank(q, q2id, p, p2id, first_stage), topN)
    return res
