#!/usr/bin/env python
"""bench.py — ANN-refresh throughput (BASELINE.json metric) on N GPUs of one node.

One STEP = one slice of a full refresh at (about) the refresh's own passage:query mix, through the code the drop-in driver
runs (ance_b200.drivers.run_ann_data_gen):
    encode PB passages into index row storage and add them in place (quantisation + norms: `IndexFlatIP.add`)
  + encode QB train queries
  + top-k inner-product search of those queries against the RESIDENT full-size index (sharded i % N across ranks when
    N > 1: queries all-gathered, per-shard top-k, all-to-all of the lists to the rank that owns each query, host k-way merge
    there, merged labels gathered on rank 0 — `sharded_search`, the driver's own function).
value = (passages encoded + queries searched) per second, whole job; `stages` gives the two rates the metric names.

Workloads (--workload; the default is the one BASELINE.json's metric is quoted on):
  marco_psg        BASELINE configs[1]: rdot_nll RoBERTa-base, passages L=128, queries L=64, 8,841,823 x 768 index, top-200
  marco_doc_maxp   configs[3]: rdot_nll_multi_chunk, documents 2048 = 4 x 512 chunks, 12,855,340 x 768 chunk-row index, top-200
  dpr              configs[4]: DPR BiEncoder (BERT-base, CLS, no head), L=256, 21,015,324 x 768 un-normalised rows, top-100

  python bench.py --gpus 1 --steps 5 --warmup 3
  python bench.py --gpus 1 --steps 5 --warmup 3 --dump-outputs DIR   # + the last timed step's outputs as DIR/<name>.npy
  python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
         bench.py --gpus N --steps K --warmup W
  python bench.py --impl reference ...     # the reference's CPU arithmetic on the host cores (see run_reference)
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

DIM = 768
WORKLOADS = {
    "marco_psg": dict(
        title="BASELINE configs[1]: MS MARCO passage 8.8M, rdot_nll seq_len=128, encode + top-200",
        metric="ANN-refresh throughput: passages encoded/sec + queries top-200/sec, 8.8M x 768",
        unit="passages+queries/s", model="rdot_nll", L_p=128, L_q=64, chunks=1, n_index=8841823, topk=200,
        pb=37888, qb=2368, index_kind="layernorm_clustered", head=True),
    "marco_doc_maxp": dict(
        title="BASELINE configs[3]: MS MARCO document 3.2M, rdot_nll_multi_chunk (MaxP) seq_len=2048 = 4 x 512, encode + top-200 "
              "over 12,855,340 chunk rows",
        metric="ANN-refresh throughput: documents (4 x 512 tokens) encoded/sec + queries top-200/sec, 12.9M x 768",
        unit="documents+queries/s", model="rdot_nll_multi_chunk", L_p=2048, L_q=64, chunks=4, n_index=12855340, topk=200,
        pb=2368, qb=296, index_kind="layernorm_clustered", head=True),
    "dpr": dict(
        title="BASELINE configs[4]: DPR 21M Wikipedia passages, BiEncoder (BERT-base CLS) seq_len=256, encode + top-100",
        metric="ANN-refresh throughput: passages encoded/sec + queries top-100/sec, 21M x 768",
        unit="passages+queries/s", model="dpr", L_p=256, L_q=256, chunks=1, n_index=21015324, topk=100,
        pb=18944, qb=296, index_kind="dpr", head=False),
}


def flop_seq(L, head=True):          # SURVEY.md §8(d): dense, padded to L
    return 12 * (24 * 768 * 768 * L + 4 * 768 * L * L) + (2 * 768 * 768 if head else 0)


def gemm_flop_seq(L, head=True):     # the GEMM kernel's share
    return 12 * 24 * 768 * 768 * L + (2 * 768 * 768 if head else 0)


def pruned_flop_seq(L):
    """Last-layer pruning: out-proj + FFN of the last layer run on the CLS row only (result-identical), so
    18 * 768^2 * (L - 1) FLOP per sequence are NOT executed.  Fractions of peak are computed from EXECUTED flops."""
    return 18 * 768 * 768 * (L - 1)


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        j = json.load(open(p))
        return {"bf16_tflops": j.get("bf16_tflops_sustained", j.get("bf16_tflops")), "hbm_gbs": j.get("hbm_gbs"),
                "source": "MEASURED_PEAKS.json (bf16_tflops_sustained: the kernel is timed inside a long step)"}
    return {"bf16_tflops": 1400.0, "hbm_gbs": 6650.0, "source": "fallback (B200_PROFILING.md, sustained)"}


class ClockSampler(threading.Thread):
    Q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index=0):
        super().__init__(daemon=True)
        self.index, self.rows, self._stop_evt = index, [], threading.Event()

    def run(self):
        while not self._stop_evt.is_set():
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                f = [x.strip() for x in out.strip().split(",")]
                if len(f) >= 6:
                    self.rows.append(f)
            except Exception:
                pass
            self._stop_evt.wait(0.2)

    def stop(self):
        self._stop_evt.set()
        self.join(timeout=3)
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        sm = sorted(int(r[0]) for r in self.rows if r[0].isdigit())
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(r[2 + i].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None,
                "sm_max_mhz": int(self.rows[0][1]) if self.rows[0][1].isdigit() else None, "reasons": reasons,
                "samples": len(self.rows)}


def workload_config(args, wl, world):
    return {"workload": wl["title"], "index_rows": wl["n_index"], "dim": DIM, "topk": wl["topk"],
            "passages_per_step_per_gpu": args.passages_per_step, "queries_per_step_per_gpu": args.queries_per_step,
            "passage_len": wl["L_p"], "query_len": wl["L_q"],
            "parallelism": ("rows i%%%d per rank, all-gather queries, all-to-all of per-shard top-k, per-rank host merge" % world)
            if world > 1 else "single GPU",
            "search_operand": args.search_operand, "encoder_operand": args.encoder_operand,
            "l2": "inputs larger than L2 (16-bit index operands %.1f GB + fp32 rows %.1f GB; ~0.9 GB of activations per "
                  "encoder pass)" % (wl["n_index"] * DIM * 2 / 1e9 / world, wl["n_index"] * DIM * 4 / 1e9 / world)}


# =============================================================================================
# reference arm / CPU baseline: the reference's own CPU path on the host cores
#   encode: HF-RoBERTa/BERT eager fp32 arithmetic, batch 16 (commands/run_ann_data_gen.sh) — oracle/encoder_oracle.py,
#           pinned by golden vectors generated from the reference's classes
#   search: faiss.IndexFlatIP when a faiss wheel is importable on the box (BASELINE.md par. 4.2), else its arithmetic
#           restated as BASELINE.md specifies: blocked fp32 sgemm (torch.matmul -> MKL) + exact top-k, with all host
#           cores and with the 16 threads the reference pins (run_ann_data_gen.py:269) — the faster of the two is reported
# =============================================================================================
_CPU = {}


def _cpu_models(wl):
    key = wl["model"]
    if key not in _CPU:
        from ance_b200.synthetic import random_roberta_state_dict
        from oracle.encoder_oracle import BiEncoderOracle, RobertaDotOracle
        if wl["model"] == "dpr":
            sd = {**random_roberta_state_dict(seed=0, vocab=30522, max_pos=512, head=False, prefix="question_model."),
                  **random_roberta_state_dict(seed=1, vocab=30522, max_pos=512, head=False, prefix="ctx_model.")}
            _CPU[key] = BiEncoderOracle(sd)
        else:
            _CPU[key] = RobertaDotOracle(random_roberta_state_dict(seed=0))
    return _CPU[key]


def synth_tokens(n, L, seed, wl):
    """Full-length synthetic token ids (the roofline regime, SURVEY.md §8d): int32 [n, L], position 0 = <s>/[CLS]."""
    g = torch.Generator().manual_seed(seed)
    hi = 30522 if wl["model"] == "dpr" else 50265
    ids = torch.randint(3, hi, (n, L), generator=g, dtype=torch.int32)
    ids[:, 0] = 101 if wl["model"] == "dpr" else 0
    return ids


def cpu_search_topk(P: torch.Tensor, Q: torch.Tensor, k: int, threads: int, p_block: int = 65536):
    """Blocked fp32 sgemm + exact top-k with a running merge (the faiss IndexFlatIP arithmetic)."""
    torch.set_num_threads(threads)
    best_d = torch.full((Q.shape[0], k), -float("inf"))
    best_i = torch.full((Q.shape[0], k), -1, dtype=torch.int64)
    for s in range(0, P.shape[0], p_block):
        S = Q @ P[s:s + p_block].T
        d, i = torch.topk(S, min(k, S.shape[1]), dim=1)
        d, i = torch.cat([best_d, d], 1), torch.cat([best_i, i + s], 1)
        best_d, sel = torch.topk(d, k, dim=1)
        best_i = torch.gather(i, 1, sel)
    return best_d, best_i


def _pick_threads(fn, thread_sets):
    """Time `fn` once per candidate thread count on a small probe and return the fastest (small fp32 GEMMs stop scaling —
    and regress — far below the 128+ hardware threads of a B200 host, so "all cores" is not automatically the best the
    reference's CPU path can do; both it and the reference's own 16 (run_ann_data_gen.py:269) are tried)."""
    best_t, best_th = None, thread_sets[0]
    for th in thread_sets:
        torch.set_num_threads(th)
        fn()   # warm-up at this thread count
        t0 = time.time()
        fn()
        dt = time.time() - t0
        if best_t is None or dt < best_t:
            best_t, best_th = dt, th
    torch.set_num_threads(best_th)
    return best_th


def cpu_step_sample(wl, n_p, n_q, search_q, search_rows, want_outputs=False):
    """Time a bounded sample of one step on the CPU.  Returns rates (units/s; the search rate is scaled linearly in the
    row count to the workload's index size), what was used, and optionally the sample's inputs / outputs for the
    parity block of the B200 arm."""
    cores = os.cpu_count() or 1
    thread_sets = sorted({cores, min(cores, 64), min(cores, 16)}, reverse=True)
    orc = _cpu_models(wl)
    setup_t0 = time.time()
    L_p, L_q, C = wl["L_p"], wl["L_q"], wl["chunks"]
    p_ids, q_ids = synth_tokens(n_p, L_p, 11, wl), synth_tokens(n_q, L_q, 12, wl)

    def enc_p(ids):
        m = torch.ones_like(ids)
        return orc.body_emb_multi_chunk(ids, m) if C > 1 else orc.body_emb(ids, m)

    if "enc_threads" not in _CPU:
        probe = p_ids[:min(16, n_p)] if C == 1 else p_ids[:2]
        _CPU["enc_threads"] = _pick_threads(lambda: enc_p(probe), thread_sets)
    enc_threads = _CPU["enc_threads"]
    torch.set_num_threads(enc_threads)
    setup_s = time.time() - setup_t0        # thread-count probe (first call only): not part of the sample
    t_all = t0 = time.time()
    p_emb = torch.cat([enc_p(p_ids[s:s + 16]) for s in range(0, n_p, 16)])   # per_gpu_eval_batch_size of the shipped scripts
    rate_p = n_p / (time.time() - t0)
    t0 = time.time()
    q_emb = orc.query_emb(q_ids, torch.ones_like(q_ids))
    rate_q = n_q / (time.time() - t0)
    t_work = time.time() - t_all
    key = (search_rows, search_q, wl["index_kind"])
    if _CPU.get("search_key") != key:   # synthetic operands: setup, generated once per process, not timed
        rng = np.random.default_rng(0)      # (torch.randn with a CPU generator needs ~50 s for 400M values)

        def rows(n):
            x = rng.standard_normal((n, DIM), dtype=np.float32)
            if wl["index_kind"] != "dpr":
                for s0 in range(0, n, 1 << 16):
                    c = x[s0:s0 + (1 << 16)]
                    c -= c.mean(1, keepdims=True)
                    c /= c.std(1, keepdims=True)
            return torch.from_numpy(x)

        _CPU["search_key"], _CPU["search_ops"] = key, (rows(search_rows), rows(search_q))
    P, Qs = _CPU["search_ops"]
    k = wl["topk"]
    try:
        import faiss  # noqa: F401  (absent from this image; used when the box has it)
        search_kind = "faiss.IndexFlatIP"
        index = faiss.IndexFlatIP(DIM)
        index.add(P.numpy())
        if "search_threads" not in _CPU:
            best = None
            for th in thread_sets:
                faiss.omp_set_num_threads(th)
                t0 = time.time()
                index.search(Qs[:64].numpy(), k)
                dt = time.time() - t0
                if best is None or dt < best[0]:
                    best = (dt, th)
            _CPU["search_threads"] = best[1]
        s_threads = _CPU["search_threads"]
        faiss.omp_set_num_threads(s_threads)
        t0 = time.time()
        D_np, I_np = index.search(Qs.numpy(), k)
        qps_slice = search_q / (time.time() - t0)
        D_cpu, I_cpu = torch.from_numpy(D_np), torch.from_numpy(I_np)
    except ImportError:
        search_kind = "blocked fp32 sgemm (MKL) + top-k"
        if "search_threads" not in _CPU:
            n_probe = min(search_rows, 1 << 17)
            _CPU["search_threads"] = _pick_threads(lambda: cpu_search_topk(P[:n_probe], Qs[:min(256, search_q)], k, torch.get_num_threads()),
                                                   thread_sets)
        s_threads = _CPU["search_threads"]
        t0 = time.time()
        D_cpu, I_cpu = cpu_search_topk(P, Qs, k, s_threads)
        qps_slice = search_q / (time.time() - t0)
    t_work += search_q / qps_slice
    qps_full = qps_slice * search_rows / wl["n_index"]
    info = {"rate_p": rate_p, "rate_q": rate_q, "qps_full": qps_full, "seconds": t_work,
            "encode_threads": enc_threads, "search_threads": s_threads, "search_kind": search_kind, "host_cores": cores}
    if want_outputs:
        info["outputs"] = dict(p_ids=p_ids, q_ids=q_ids, p_emb=p_emb, q_emb=q_emb, P=P, Q=Qs, D=D_cpu, I=I_cpu)
    return info


# bounded samples of one step for the CPU arm: ~15-25 s of host work inside the default bench run, a few s per step of
# `--impl reference` (K + W steps must end within a few minutes)
def cpu_samples(wl):
    n_p = {"marco_psg": 192, "marco_doc_maxp": 16, "dpr": 96}[wl_name(wl)]
    base = dict(n_p=n_p, n_q=48, search_q=1024, search_rows=1 << 20)
    ref = dict(n_p=max(16, n_p // 2), n_q=32, search_q=512, search_rows=1 << 19)
    if os.environ.get("ANCE_BENCH_TINY_CPU"):   # contract tests only (tests/test_bench_contract.py)
        base = ref = dict(n_p=2, n_q=2, search_q=4, search_rows=4096)
    return base, ref


def wl_name(wl):
    return next(k for k, v in WORKLOADS.items() if v is wl)


def sample_text(wl, sm, info):
    return ("%d %s L=%d + %d queries L=%d through the oracle port of the reference's HF eager fp32 path (batch 16, %d threads); "
            "%d queries x %s rows %s (%d threads), top-%d, scaled linearly to N=%s; host has %d cores"
            % (sm["n_p"], "documents" if wl["chunks"] > 1 else "passages", wl["L_p"], sm["n_q"], wl["L_q"],
               info["encode_threads"], sm["search_q"], format(sm["search_rows"], ","), info["search_kind"],
               info["search_threads"], wl["topk"], format(wl["n_index"], ","), info["host_cores"]))


def cpu_value(pb, qb, info):
    t = pb / info["rate_p"] + qb / info["rate_q"] + qb / info["qps_full"]
    return (pb + qb) / t


def run_reference(args, wl):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    pb, qb = args.passages_per_step, args.queries_per_step
    _, ref_sample = cpu_samples(wl)
    vals, spent, info = [], 0.0, None
    for i in range(args.warmup + args.steps):
        info = cpu_step_sample(wl, **ref_sample)
        spent += info["seconds"]
        if i >= args.warmup:
            vals.append(cpu_value(pb, qb, info))
    v = float(np.mean(vals))
    sample = "per step: " + sample_text(wl, ref_sample, info) + "; extrapolated to the step's %d + %d units; %.1f s of CPU work per step" % (
        pb, qb, spent / max(1, args.warmup + args.steps))
    print(json.dumps({
        "impl": "reference", "metric": wl["metric"], "value": v, "unit": wl["unit"], "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": (pb + qb) / v * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args, wl, 1),
        "cpu_baseline": {"value": v, "unit": wl["unit"], "cores": max(info["encode_threads"], info["search_threads"]),
                         "kind": "port", "sample": sample, "passages_per_s": info["rate_p"],
                         "queries_topk_per_s": info["qps_full"]},
        "e2e": {"value": v, "unit": wl["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }))


# =============================================================================================
# B200 arm
# =============================================================================================
def build_model(wl, dev, encoder_operand):
    from ance_b200.models import BiEncoder, RobertaDot_CLF_ANN_NLL_MultiChunk, RobertaDot_NLL_LN
    from ance_b200.synthetic import random_roberta_state_dict, roberta_base_config
    if wl["model"] == "dpr":
        model = BiEncoder()
        model.load_state_dict({**random_roberta_state_dict(seed=0, vocab=30522, max_pos=512, head=False, prefix="question_model."),
                               **random_roberta_state_dict(seed=1, vocab=30522, max_pos=512, head=False, prefix="ctx_model.")})
    else:
        cls = RobertaDot_CLF_ANN_NLL_MultiChunk if wl["model"] == "rdot_nll_multi_chunk" else RobertaDot_NLL_LN
        model = cls(roberta_base_config())
        model.load_state_dict(random_roberta_state_dict(seed=0), strict=True)
    model.encoder_operand = encoder_operand
    return model.to(dev).eval()


DUMP_MAX_ROWS = 4096


def dump_outputs(out_dir, outputs):
    """Write each output as out_dir/<name>.npy: float32, labels as float64 (exact below 2**53).  An output of more than
    DUMP_MAX_ROWS rows keeps the rows np.random.default_rng(0).choice(n, DUMP_MAX_ROWS, replace=False), sorted: the same
    rows in every run, so that two builds can be compared output for output (at most ~32 MB in all)."""
    os.makedirs(out_dir, exist_ok=True)
    for name, x in outputs.items():
        x = x.cpu().numpy() if torch.is_tensor(x) else np.asarray(x)
        if x.shape[0] > DUMP_MAX_ROWS:
            x = x[np.sort(np.random.default_rng(0).choice(x.shape[0], DUMP_MAX_ROWS, replace=False))]
        np.save(os.path.join(out_dir, name + ".npy"), x.astype(np.float64 if x.dtype.kind in "iu" else np.float32))


def run_b200(args, wl):
    import torch.distributed as dist
    from ance_b200 import _lib
    from ance_b200.drivers.run_ann_data_gen import sharded_search, sharded_search_start
    from ance_b200.search import IndexFlatIP
    from ance_b200.synthetic import synth_index_rows

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (there is no CPU fallback; use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl")
    pb, qb = args.passages_per_step, args.queries_per_step
    L_p, L_q, C, k = wl["L_p"], wl["L_q"], wl["chunks"], wl["topk"]
    Lc = L_p // C                                  # tokens per encoded sequence
    model = build_model(wl, dev, args.encoder_operand)
    mask_form = wl["model"] == "dpr"               # DPR: mask = ids != 0 (DPR_data.py:283); MARCO: lengths (msmarco_data.py:282)

    # this rank's shard of the synthetic corpus, resident for the whole run
    n_index = wl["n_index"]
    n_local = len(range(rank, n_index, world))
    row_offset = sum(len(range(r, n_index, world)) for r in range(rank))   # global number of this rank's first row
    index = IndexFlatIP(DIM, capacity=n_local, device=dev, operand=args.search_operand)
    for x in synth_index_rows(n_local, DIM, dev, 1234 + rank, wl["index_kind"]):
        index.add(x)
    del x
    torch.cuda.empty_cache()
    # the step's own passages go into a scratch index of pb * C rows (in-place add, as the driver does)
    step_rows = torch.empty((pb * C, DIM), dtype=torch.float32, device=dev)
    step_index = IndexFlatIP(DIM, device=dev, operand=args.search_operand, storage=step_rows)

    # synthetic token ids: HOST pinned (e2e) and device-resident copies (value); full length = the roofline regime
    p_ids_h = synth_tokens(pb, L_p, 100 + rank, wl).pin_memory()
    q_ids_h = synth_tokens(qb, L_q, 200 + rank, wl).pin_memory()
    p_mask_h = torch.ones((pb, L_p), dtype=torch.bool).pin_memory()     # GetProcessingFn's attention_mask (bool [L])
    q_mask_h = torch.ones((qb, L_q), dtype=torch.bool).pin_memory()
    p_ids_d, q_ids_d = p_ids_h.to(dev), q_ids_h.to(dev)
    p_len_d = torch.full((pb,), L_p, dtype=torch.int32, device=dev)
    q_len_d = torch.full((qb,), L_q, dtype=torch.int32, device=dev)
    local_search = lambda q, kk, off: index.search_device(q, kk, row_offset=off)   # noqa: E731

    def encode_passages_fast(ids, lens):
        """device-resident inputs, the refresher's fast path (lengths instead of masks, rows written in place)"""
        if wl["model"] == "dpr":
            step_rows.copy_(model.body_emb(ids, ids != 0))
        elif C > 1:
            step_rows.copy_(model.encode_lens_multi_chunk(ids, lens).reshape(pb * C, DIM))
        else:
            model.encode_lens(ids, lens, out=step_rows)

    pending = []      # N > 1: the previous slice's search, issued but not yet merged / gathered
    last = {}         # what the latest step computed (--dump-outputs): its queries and, once merged, their top-k labels

    def step_value():
        step_index.reset()
        encode_passages_fast(p_ids_d, p_len_d)
        step_index.add(step_rows)          # in place: the rows were written into the index's own storage
        step_index.prepare()               # column mean + centred 16-bit operands + norm statistics of the added rows
        q = model.query_emb(q_ids_d, q_ids_d != 0) if mask_form else model.encode_lens(q_ids_d, q_len_d)
        if world == 1:
            last["query_emb"] = q
            last["topk_labels"] = sharded_search(local_search, n_local, q.contiguous(), k, row_offset=row_offset)
            return last["topk_labels"]     # numpy labels
        q_all = torch.empty((qb * world, DIM), dtype=torch.float32, device=dev)
        dist.all_gather_into_tensor(q_all, q.contiguous())
        last["query_emb"] = q_all
        # As in the driver's block loop, the host merge of this slice's lists overlaps the device work that follows: the
        # search is issued here and finished (merge waited for, labels gathered on rank 0) after the NEXT slice has been
        # enqueued; `drain()` finishes the last one inside the timed region.
        pending.append(sharded_search_start(local_search, n_local, q_all, k, row_offset=row_offset))
        if len(pending) > 1:
            last["topk_labels"] = pending.pop(0).finish()
            return last["topk_labels"]
        return None

    def drain():
        while pending:
            last["topk_labels"] = pending.pop(0).finish()

    def step_e2e():
        """The calls a user of the reference makes (run_ann_data_gen.py:172-180,269-303), host buffers in, numpy out:
        H2D of the batch's ids + mask, `model.body_emb(ids.long(), mask.long())`, `IndexFlatIP.add`,
        `model.query_emb`, `.cpu().numpy()`, `IndexFlatIP.search(numpy, k)` (N > 1: the driver's sharded search)."""
        step_index.reset()
        pi, pm = p_ids_h.to(dev, non_blocking=True), p_mask_h.to(dev, non_blocking=True)
        qi, qm = q_ids_h.to(dev, non_blocking=True), q_mask_h.to(dev, non_blocking=True)
        emb = model.body_emb(pi.long(), pm.long())
        step_index.add(emb.reshape(pb * C, DIM))
        step_index.prepare()
        q = model.query_emb(qi.long(), qm.long())
        if world > 1:
            q_all = torch.empty((qb * world, DIM), dtype=torch.float32, device=dev)
            dist.all_gather_into_tensor(q_all, q.contiguous())
            return sharded_search(local_search, n_local, q_all, k, row_offset=row_offset)
        _, I = index.search(q.cpu().numpy(), k)
        return I

    def sync():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps: int, wall: bool):
        sync()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.time()
        e0.record()
        for _ in range(steps):
            fn()
        drain()
        e1.record()
        sync()
        ms = (time.time() - t0) * 1e3 if wall else e0.elapsed_time(e1)   # e2e includes host work: wall clock
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms / steps

    warm = max(3, args.warmup)
    for _ in range(warm):
        step_value()
    drain()
    sync()
    launches0 = _lib.load().ance_launch_count()
    _lib.profile_enable(True)
    _lib.profile_read(reset=True)
    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.start()
    ms = timed(step_value, args.steps, wall=False)
    clocks = sampler.stop() if sampler else None
    prof = _lib.profile_read(reset=True)
    _lib.profile_enable(False)
    launches = _lib.load().ance_launch_count() - launches0
    if args.dump_outputs and rank == 0:    # before the e2e pass below writes its own passages into step_rows
        dump_outputs(args.dump_outputs, {"passage_emb": step_rows, "query_emb": last["query_emb"],
                                         "topk_labels": last["topk_labels"]})
    st = index.stats()
    step_e2e()
    ms_e2e = timed(step_e2e, max(2, args.steps // 2), wall=True)
    # practical figure (SURVEY.md §8d): MS-MARCO-like passage lengths ~ clipped N(76, 28), encoded as the driver does by
    # default (whole sequences packed into 128-token tiles: only real tokens are computed) and with padded length buckets.
    # Reported beside, never inside, `value`.
    ms_marco = ms_marco_bucketed = None
    if wl["model"] == "rdot_nll":
        gl = torch.Generator().manual_seed(5)
        mlens_h = torch.clamp(torch.normal(76.0, 28.0, (pb,), generator=gl).round(), 8, L_p).to(torch.int32)
        mlens = mlens_h.to(dev)

        def time_it(fn):
            for _ in range(2):
                fn()
            sync()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(2):
                fn()
            e1.record()
            sync()
            return e0.elapsed_time(e1) / 2

        ms_marco = time_it(lambda: model.encode_lens_varlen(p_ids_d, mlens, lens_host=mlens_h, out=step_rows))
        ms_marco_bucketed = time_it(lambda: model.encode_lens_bucketed(p_ids_d, mlens, out=step_rows))

    if rank != 0:
        return
    units = (pb + qb) * world
    pk = peaks()
    head = wl["head"]
    gemm_ms, gemm_n = prof["encoder_gemm"]
    seqs_p = pb * C
    pruned = args.steps * (seqs_p * pruned_flop_seq(Lc) + qb * pruned_flop_seq(L_q))
    gemm_flop = args.steps * (seqs_p * gemm_flop_seq(Lc, head) + qb * gemm_flop_seq(L_q, head)) - pruned  # executed
    gemm_tf = gemm_flop / gemm_ms / 1e9
    coarse_ms, coarse_n = prof["coarse_search"]
    coarse_tf = args.steps * 2.0 * qb * world * n_local * DIM / coarse_ms / 1e9 if coarse_ms else None
    enc_ms = gemm_ms + prof["attention"][0] + prof["norm_embed"][0]
    srch_ms = coarse_ms + prof["rescore"][0] + prof["exact"][0]     # + the queries' share of `quantize` (negligible)
    alg_flop = args.steps * (seqs_p * flop_seq(Lc, head) + qb * flop_seq(L_q, head))
    traffic = None
    tp = os.path.join(ROOT, "profiles", "r02_ncu_gemm_traffic.json")
    if not os.path.exists(tp):
        tp = os.path.join(ROOT, "profiles", "r01_ncu_gemm_traffic.json")
    if os.path.exists(tp) and wl is WORKLOADS["marco_psg"]:
        traffic = json.load(open(tp)).get("dram_bytes_per_launch")
    out = {
        "metric": wl["metric"], "value": units / ms * 1e3, "unit": wl["unit"], "n_gpus": world, "steps": args.steps,
        "warmup": warm, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": args.encoder_operand,   # 16-bit tensor-core operands and storage, fp32 accumulation / statistics
        "data": "synthetic", "config": workload_config(args, wl, world),
        "stages": {
            "passages_encoded_per_s": (pb + qb * L_q / L_p) * args.steps / enc_ms * 1e3 * world,
            "queries_topk_per_s": qb * world * args.steps / srch_ms * 1e3,
            "encode_ms_per_step": enc_ms / args.steps, "search_ms_per_step": srch_ms / args.steps,
            "index_add_ms_per_step": prof["quantize"][0] / args.steps,
            "encode_frac_of_bf16_peak": ((alg_flop - pruned) / enc_ms / 1e9) / pk["bf16_tflops"],
            "attention_share_of_encode": prof["attention"][0] / enc_ms,
            "encode_flop_per_sequence": {"algorithmic": flop_seq(Lc, head), "executed": flop_seq(Lc, head) - pruned_flop_seq(Lc)},
            "search_coarse_tflops": coarse_tf,
            "search_coarse_frac_of_bf16_peak": coarse_tf / pk["bf16_tflops"] if coarse_tf else None,
            "search_stats": st,
            "passages_per_s_marco_like_lengths": (pb / ms_marco * 1e3 * world) if ms_marco else None,   # variable-length tiles
            "passages_per_s_marco_like_lengths_bucketed": (pb / ms_marco_bucketed * 1e3 * world) if ms_marco_bucketed else None,
        },
        "roofline": {"kernel": "tc05_gemm_kernel<EpStore> (encoder linear layers)", "bound": "tensor",
                     "achieved": gemm_tf, "peak": pk["bf16_tflops"], "unit": "TFLOP/s", "frac": gemm_tf / pk["bf16_tflops"],
                     "traffic": traffic, "peak_source": pk["source"], "launches": gemm_n,
                     "avg_launch_ms": gemm_ms / max(gemm_n, 1),
                     "share_of_step": gemm_ms / (ms * args.steps)},
        "e2e": {"value": units / ms_e2e * 1e3, "unit": wl["unit"],
                "h2d_bytes_per_step": int(pb * L_p * 5 + qb * L_q * 5 + (0 if world > 1 else qb * DIM * 4)),
                "d2h_bytes_per_step": int(qb * world * k * (8 if world > 1 else 12) + (0 if world > 1 else qb * DIM * 4)),
                "path": "host ids+mask -> body_emb / query_emb (plugin calls) -> IndexFlatIP.add -> "
                        + ("all-gather + sharded_search (driver)" if world > 1 else "IndexFlatIP.search(numpy)")},
        "gpu_launches": int(launches),
        "clocks": clocks,
        "kernel_ms_per_step": {kk: v[0] / args.steps for kk, v in prof.items()},
    }
    if world == 1 and not args.no_cpu_baseline:
        base_sample, _ = cpu_samples(wl)
        info = cpu_step_sample(wl, want_outputs=True, **base_sample)
        o = info.pop("outputs")
        out["cpu_baseline"] = {
            "value": cpu_value(pb, qb, info), "unit": wl["unit"], "cores": max(info["encode_threads"], info["search_threads"]),
            "kind": "port", "sample": sample_text(wl, base_sample, info) + "; %.0f s of CPU work" % info["seconds"],
            "passages_per_s": info["rate_p"], "queries_topk_per_s": info["qps_full"], "search_kind": info["search_kind"]}
        # parity of the B200 path with the CPU arm on the very sample the CPU arm just computed (checker use of oracle/)
        with torch.no_grad():
            pi = o["p_ids"].to(dev)
            if wl["model"] == "dpr":
                pe, qe = model.body_emb(pi, pi != 0), model.query_emb(o["q_ids"].to(dev), o["q_ids"].to(dev) != 0)
            elif C > 1:
                pe = model.encode_lens_multi_chunk(pi, torch.full((pi.shape[0],), L_p, dtype=torch.int32, device=dev))
                qe = model.encode_lens(o["q_ids"].to(dev), torch.full((o["q_ids"].shape[0],), L_q, dtype=torch.int32, device=dev))
            else:
                pe = model.encode_lens(pi, torch.full((pi.shape[0],), L_p, dtype=torch.int32, device=dev))
                qe = model.encode_lens(o["q_ids"].to(dev), torch.full((o["q_ids"].shape[0],), L_q, dtype=torch.int32, device=dev))
        pe, qe = pe.reshape(-1, DIM).cpu(), qe.cpu()
        ref_p = o["p_emb"].reshape(-1, DIM)
        small = IndexFlatIP(DIM, capacity=o["P"].shape[0], device=dev, operand=args.search_operand)
        small.add(o["P"].to(dev))
        Dg, Ig = small.search(o["Q"].numpy(), k)
        same = float((torch.from_numpy(Ig) == o["I"]).all(dim=1).float().mean())
        setov = float(np.mean([len(np.intersect1d(Ig[i], o["I"][i].numpy())) for i in range(Ig.shape[0])])) / k
        out["parity"] = {
            "encoder_min_cosine_vs_fp32_reference": float(torch.nn.functional.cosine_similarity(pe, ref_p, dim=-1).min()),
            "encoder_max_abs_vs_fp32_reference": float(max((pe - ref_p).abs().max(), (qe - o["q_emb"]).abs().max())),
            "search_topk_lists_identical_frac_vs_cpu_fp32": same, "search_topk_set_overlap_vs_cpu_fp32": setov,
            "search_score_max_rel_diff": float(((torch.from_numpy(Dg) - o["D"]).abs().max() / o["D"].abs().max())),
            "note": "CPU fp32 sgemm sums in a different order than the canonical fp64-accumulated score: lists may differ "
                    "only where two scores are closer than fp32 summation noise; bit-exact parity vs the oracle is in tests/",
            "overlap_at_200_vs_fp32_encoded_corpus": _load_overlap()}
    print(json.dumps(out))


def _load_overlap():
    """The 20,480-passage overlap@200 gate is a GPU test (tests/test_gpu_encoder.py); its last committed result."""
    p = os.path.join(ROOT, "profiles", "r02_overlap_at_200.json")
    return json.load(open(p)) if os.path.exists(p) else None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=4)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="marco_psg", choices=sorted(WORKLOADS))
    ap.add_argument("--passages_per_step", type=int, default=0, help="per GPU; 0 = the workload's default")
    ap.add_argument("--queries_per_step", type=int, default=0, help="per GPU; 0 = the workload's default")
    ap.add_argument("--search_operand", default="auto", choices=["auto", "fp16", "bf16"])
    ap.add_argument("--encoder_operand", default="fp16", choices=["fp16", "bf16"])
    ap.add_argument("--no_cpu_baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one computed (passage and query embeddings, top-k "
                         "labels) as DIR/<name>.npy; the inputs are seeded, so runs with the same arguments compare")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the B200 path (--impl b200)")
    wl = WORKLOADS[args.workload]
    # defaults: marco_psg 64 encoder passes of 592 x 128 tokens + 2 of 1184 x 64 (16:1, the refresh's own 17.6:1);
    # marco_doc_maxp 64 passes of 148 x 512 (2,368 documents) + 296 queries (8:1; real 8.75:1); dpr 64 passes of 296 x 256
    args.passages_per_step = args.passages_per_step or wl["pb"]
    args.queries_per_step = args.queries_per_step or wl["qb"]
    if args.impl == "reference":
        run_reference(args, wl)
    else:
        run_b200(args, wl)


if __name__ == "__main__":
    try:
        main()
    finally:
        import torch.distributed as _dist
        if _dist.is_available() and _dist.is_initialized():
            _dist.destroy_process_group()
