"""Search throughput against k (100 .. 2048) at the MS MARCO passage size, 8,841,823 x 768.

For every operand format x query count x k: queries/s of the whole ance_index_search call (CUDA events, profiler off,
median of --reps after a warm-up), then one more call with the library's per-class device timers on (coarse pass,
rescore, quantize, exact fallback), and the tier counts and largest certificate eps from stats().  6,980 queries is the
MS MARCO dev set (the notebook's full rank at top-1000); 18,944 is one wave of the coarse kernel's CTA pairs x 256 rows.

The index rows are clustered LayerNorm-like vectors (tools/bringup_search.make_data, seeded), 27 GB of fp32 and 13.6 GB
of 16-bit operands: far larger than L2.  The card's name, power limit and max SM clock are read in the same run.

    python tools/perf_search_topk.py [--n 8841823] [--out profiles/r03_perf_search_topk.jsonl]
"""
import argparse
import json
import subprocess
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
import torch  # noqa: E402

from ance_b200 import _lib  # noqa: E402
from ance_b200.search import IndexFlatIP  # noqa: E402
from tools.bringup_search import make_data  # noqa: E402


def card():
    r = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True, timeout=30)
    f = [x.strip() for x in r.stdout.strip().split(",")]
    return {"name": f[0], "power_limit": f[1], "sm_max_clock": f[2]} if len(f) == 3 else {"nvidia_smi": r.stdout.strip()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=8841823)
    ap.add_argument("--nq", default="6980,18944")
    ap.add_argument("--k", default="100,200,500,1000,2048")
    ap.add_argument("--fmt", default="fp16,bf16")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=str(ROOT / "profiles" / "r03_perf_search_topk.jsonl"))
    a = ap.parse_args()
    nqs = [int(x) for x in a.nq.split(",")]
    ks = [int(x) for x in a.k.split(",")]
    dev = torch.device("cuda:0")
    head = {"card": card(), "torch_device": torch.cuda.get_device_name(0), "N": a.n, "dim": 768}
    out = open(a.out, "a")

    def emit(rec):
        print(json.dumps(rec), flush=True)
        out.write(json.dumps(rec) + "\n")
        out.flush()

    emit(head)
    P, Q = make_data(a.n, max(nqs), 768, "clustered", dev)
    for fmt in a.fmt.split(","):
        idx = IndexFlatIP(768, capacity=a.n, operand=fmt)
        idx.add(P)
        idx.prepare()
        for nq in nqs:
            q = Q[:nq].contiguous()
            for k in ks:
                idx.search_device(q, k)            # warm-up: workspace for this shape
                torch.cuda.synchronize()
                ms = []
                for _ in range(a.reps):
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record()
                    idx.search_device(q, k)
                    e1.record()
                    torch.cuda.synchronize()
                    ms.append(e0.elapsed_time(e1))
                st = idx.stats()
                _lib.profile_enable(True)
                _lib.profile_read(reset=True)
                idx.search_device(q, k)
                torch.cuda.synchronize()
                prof = _lib.profile_read(reset=True)
                _lib.profile_enable(False)
                med = sorted(ms)[len(ms) // 2]
                emit({"N": a.n, "nq": nq, "k": k, "fmt": fmt, "ms": med, "ms_all": ms, "qps": nq / med * 1e3,
                      "coarse_ms": prof["coarse_search"][0], "rescore_ms": prof["rescore"][0],
                      "quant_ms": prof["quantize"][0], "exact_ms": prof["exact"][0],
                      "coarse_tflops": 2.0 * nq * a.n * 768 / max(prof["coarse_search"][0], 1e-9) / 1e9,
                      "kprime": st["kprime"], "n_splits": st["n_splits"], "n_tier2": st["n_tier2"],
                      "n_uncertified": st["n_uncertified"], "n_candidates": st["n_candidates"], "max_eps": st["max_eps"]})
        del idx
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
