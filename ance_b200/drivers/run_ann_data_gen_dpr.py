"""B200-native ANN refresher for DPR / OpenQA — drop-in for the reference's drivers/run_ann_data_gen_dpr.py
(BASELINE config 5: 21M Wikipedia passages, BERT-base bi-encoder, top-100).

Same flags, inputs and outputs as the reference; encode and search run through libance_b200 exactly as in
drivers/run_ann_data_gen.py (see that module for the data-flow table).  Differences from the MS MARCO
refresher, all inherited from the reference:
  * checkpoints are single files `training_dir/checkpoint-N` holding a CheckpointState (46-60, 112-124);
  * four encode sets: train-query, test-query (NQ), trivia-test-query, passages (209-230); the attention
    mask is `ids != 0` (data/DPR_data.py:283);
  * two dev searches (k = 100) scored by answer-string hit@k (`validate`, 312-340), one train search over
    ALL queries (no ann_chunk_factor slicing, 252);
  * negatives = neighbours in rank order whose text lacks the answer; `neg_cnt` advances even for rejected
    candidates (301-307), so fewer than `negative_sample` negatives can result (SURVEY.md Appendix A.7);
  * `ann_ndcg_N` carries top20 / top100 / top20_trivia / top100_trivia / checkpoint (275-278).
"""
from __future__ import annotations

import argparse
import ast
import csv
import json
import logging
import os
import random
import time
from typing import Dict, List

import numpy as np
import torch
import torch.distributed as dist

from ..dpr_utils import AnswerMatcher, get_model_obj, load_mapping, load_states_from_checkpoint
from ..models import MSMarcoConfigDict
from .. import postprocess
from . import run_ann_data_gen as base
from .run_ann_data_gen import (B200Backend, all_gather_ids, all_gather_rows, get_checkpoint_no, get_latest_ann_data,
                               is_first_worker, sharded_search)

logger = logging.getLogger(__name__)


def get_latest_checkpoint(args):
    """run_ann_data_gen_dpr.py:46-60: newest FILE named checkpoint-N."""
    if not os.path.exists(args.training_dir):
        return args.init_model_dir, 0
    files = list(next(os.walk(args.training_dir))[2])
    nums = [get_checkpoint_no(s) for s in files if s.startswith("checkpoint-")]
    if len(nums) > 0:
        return os.path.join(args.training_dir, "checkpoint-" + str(max(nums))), max(nums)
    return args.init_model_dir, 0


def load_data(args):
    """run_ann_data_gen_dpr.py:63-109.  Answer lists are Python literals in the files; the reference uses
    eval(), this uses ast.literal_eval (same values, no code execution)."""
    passage_path = os.path.join(args.passage_path, "psgs_w100.tsv")
    test_qa_path = os.path.join(args.test_qa_path, "nq-test.csv")
    trivia_test_qa_path = os.path.join(args.trivia_test_qa_path, "trivia-test.csv")
    train_ann_path = os.path.join(args.data_dir, "train-ann")
    pid2offset, _ = load_mapping(args.data_dir, "pid2offset")
    passage_text, train_pos_id, train_answers, test_answers, test_answers_trivia = {}, [], [], [], []
    with open(train_ann_path, "r", encoding="utf8") as f:
        for row in csv.reader(f, delimiter="\t"):  # q_id, positive_pid, answers
            train_pos_id.append(int(row[1]))
            train_answers.append(ast.literal_eval(row[2]))
    with open(test_qa_path, "r", encoding="utf-8") as f:
        for row in csv.reader(f, delimiter="\t"):
            test_answers.append(ast.literal_eval(row[1]))
    with open(trivia_test_qa_path, "r", encoding="utf-8") as f:
        for row in csv.reader(f, delimiter="\t"):
            test_answers_trivia.append(ast.literal_eval(row[1]))
    with open(passage_path, "r", encoding="utf-8") as f:
        for row in csv.reader(f, delimiter="\t"):  # doc_id, doc_text, title
            if row[0] != "id":
                passage_text[pid2offset[int(row[0])]] = (row[1], row[2])
    return passage_text, train_pos_id, train_answers, test_answers, test_answers_trivia


def load_model(args, checkpoint_path):
    """run_ann_data_gen_dpr.py:112-132."""
    args.model_type = args.model_type.lower()
    model = MSMarcoConfigDict[args.model_type].model_class(args)
    saved_state = load_states_from_checkpoint(checkpoint_path)
    get_model_obj(model).load_state_dict(saved_state.model_dict)
    model.to(args.device)
    model.eval()
    return model


def validate(matcher: AnswerMatcher, answers, closest_docs, query_embedding2id, passage_embedding2id) -> List[float]:
    """run_ann_data_gen_dpr.py:312-340: fraction of questions with an answer-bearing passage in the top k, for
    every k = 1..n_docs."""
    n_docs = closest_docs.shape[1]
    top_k_hits = [0] * n_docs
    for qi in range(closest_docs.shape[0]):
        qid = int(query_embedding2id[qi])
        best = None
        for i, pidx in enumerate(closest_docs[qi]):
            if matcher.has_answer(answers[qid], int(passage_embedding2id[pidx])):
                best = i
                break
        if best is not None:
            for j in range(best, n_docs):
                top_k_hits[j] += 1
    return [v / len(closest_docs) for v in top_k_hits]


def generate_negatives(args, matcher: AnswerMatcher, answers, query_embedding2id, passage_embedding2id, closest_docs,
                       training_query_positive_id) -> Dict[int, List[int]]:
    """run_ann_data_gen_dpr.py:281-309 (including its `neg_cnt` quirk)."""
    out: Dict[int, List[int]] = {}
    for qi in range(closest_docs.shape[0]):
        qid = int(query_embedding2id[qi])
        pos_pid = training_query_positive_id[qid]
        negs: List[int] = []
        neg_cnt = 0
        for pidx in closest_docs[qi]:
            doc_id = int(passage_embedding2id[pidx])
            if doc_id == pos_pid:
                continue
            if doc_id in negs:
                continue
            if neg_cnt >= args.negative_sample:
                break
            if not matcher.has_answer(answers[qid], doc_id):
                negs.append(doc_id)
            neg_cnt += 1
        out[qid] = negs
    return out


def generate_new_ann(args, output_num, checkpoint_path, preloaded_data, latest_step_num, backend=None):
    """run_ann_data_gen_dpr.py:204-278."""
    t0 = time.time()
    if backend is None:
        backend = B200Backend(args, load_model(args, checkpoint_path), mask_mode="nonzero")
    d = args.data_dir
    q_emb, q_ids = backend.encode(os.path.join(d, "train-query"), True)
    dev_emb, dev_ids = backend.encode(os.path.join(d, "test-query"), True)
    tv_emb, tv_ids = backend.encode(os.path.join(d, "trivia-test-query"), True)
    index, p_emb, p_ids = backend.encode(os.path.join(d, "passages"), False, build_index=True)
    device = p_emb.device
    local_search = backend.make_local_search(index)
    passage_embedding2id = all_gather_ids(p_ids, device)
    sets = {}
    for name, (e, i) in {"train": (q_emb, q_ids), "dev": (dev_emb, dev_ids), "trivia": (tv_emb, tv_ids)}.items():
        sets[name] = (all_gather_rows(e), all_gather_ids(i, device))
    dev_I = sharded_search(local_search, p_emb.shape[0], sets["dev"][0], 100)
    tv_I = sharded_search(local_search, p_emb.shape[0], sets["trivia"][0], 100)
    I = sharded_search(local_search, p_emb.shape[0], sets["train"][0], args.topk_training)
    if not is_first_worker():
        return None
    passage_text, train_pos_id, train_answers, test_answers, test_answers_trivia = preloaded_data
    matcher = AnswerMatcher(passage_text)
    top_k_hits = validate(matcher, test_answers, dev_I, sets["dev"][1], passage_embedding2id)
    top_k_hits_trivia = validate(matcher, test_answers_trivia, tv_I, sets["trivia"][1], passage_embedding2id)
    query_embedding2id = sets["train"][1]
    negatives = generate_negatives(args, matcher, train_answers, query_embedding2id, passage_embedding2id, I,
                                   train_pos_id)
    os.makedirs(args.output_dir, exist_ok=True)
    path = os.path.join(args.output_dir, "ann_training_data_" + str(output_num))
    order = list(range(I.shape[0]))
    random.shuffle(order)  # the reference's unseeded module-level `random` (run_ann_data_gen_dpr.py:266-267)
    tmp = postprocess.staging_path(path)   # never named `ann_ndcg_*` / `ann_training_data_*`: the trainer polls this dir
    with open(tmp, "w") as f:
        for qi in order:
            qid = int(query_embedding2id[qi])
            f.write("{}\t{}\t{}\n".format(qid, train_pos_id[qid], ",".join(str(n) for n in negatives[qid])))
    os.replace(tmp, path)
    postprocess.write_json_atomic(
        os.path.join(args.output_dir, "ann_ndcg_" + str(output_num)),
        {"top20": top_k_hits[19], "top100": top_k_hits[99], "top20_trivia": top_k_hits_trivia[19],
         "top100_trivia": top_k_hits_trivia[99], "checkpoint": checkpoint_path})
    logger.info("dpr refresh %d done in %.1fs", output_num, time.time() - t0)
    return top_k_hits, top_k_hits_trivia


def get_arguments(argv=None):
    p = argparse.ArgumentParser()
    for name in ("--data_dir", "--training_dir", "--init_model_dir", "--model_type", "--output_dir", "--cache_dir"):
        p.add_argument(name, default=None, type=str, required=True)
    p.add_argument("--last_checkpoint_dir", default="", type=str)
    p.add_argument("--end_output_num", default=-1, type=int)
    p.add_argument("--max_seq_length", default=128, type=int)
    p.add_argument("--max_query_length", default=64, type=int)
    p.add_argument("--max_doc_character", default=10000, type=int)
    p.add_argument("--per_gpu_eval_batch_size", default=128, type=int)
    p.add_argument("--ann_chunk_factor", default=5, type=int)
    p.add_argument("--topk_training", default=500, type=base.topk_training_arg,
                   help="neighbours searched per training query, 1 .. %d" % base.MAX_K)
    p.add_argument("--negative_sample", default=5, type=int)
    p.add_argument("--ann_measure_topk_mrr", default=False, action="store_true")
    p.add_argument("--only_keep_latest_embedding_file", default=False, action="store_true")
    p.add_argument("--no_cuda", action="store_true")
    p.add_argument("--local_rank", type=int, default=-1)
    p.add_argument("--server_ip", type=str, default="")
    p.add_argument("--server_port", type=str, default="")
    p.add_argument("--passage_path", default=None, type=str, required=True)
    p.add_argument("--test_qa_path", default=None, type=str, required=True)
    p.add_argument("--trivia_test_qa_path", default=None, type=str, required=True)
    # B200 knobs
    p.add_argument("--search_operand", default="auto", choices=["auto", "fp16", "bf16"])
    p.add_argument("--encode_batch_tokens", default=75776, type=int)
    p.add_argument("--seed", default=None, type=int)
    p.add_argument("--poll_seconds", default=60, type=int)
    a = p.parse_args(argv)
    a.inference, a.reference_sampling = False, True
    return a


def ann_data_gen(args, backend=None):
    """run_ann_data_gen_dpr.py:536-560."""
    last_checkpoint = args.last_checkpoint_dir
    ann_no, _, _ = get_latest_ann_data(args.output_dir)
    output_num = ann_no + 1
    if is_first_worker():
        os.makedirs(args.output_dir, exist_ok=True)
        os.makedirs(args.cache_dir, exist_ok=True)
    preloaded_data = load_data(args) if is_first_worker() else None
    while args.end_output_num == -1 or output_num <= args.end_output_num:
        next_checkpoint, latest_step_num = get_latest_checkpoint(args)
        if args.only_keep_latest_embedding_file:
            latest_step_num = 0
        if next_checkpoint == last_checkpoint:
            time.sleep(args.poll_seconds)
        else:
            generate_new_ann(args, output_num, next_checkpoint, preloaded_data, latest_step_num, backend=backend)
            output_num += 1
            last_checkpoint = next_checkpoint
        if dist.is_available() and dist.is_initialized():
            dist.barrier()


def main(argv=None):
    args = get_arguments(argv)
    base.set_env(args)
    ann_data_gen(args)


if __name__ == "__main__":
    main()
