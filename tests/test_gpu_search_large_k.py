"""Flat inner-product search at 512 < k <= 2048 (the notebook's top-1000 full rank, `--topk_training` above 512): the
large-reservoir coarse epilogue, tier 2 and tier 3 at large k, the exact path, the host-side query blocks, and the
evaluation / refresh drivers end to end.  Every result must equal the CPU oracle bit for bit."""
import json

import numpy as np
import pytest
import torch

from oracle import flat_ip_oracle, refresh_oracle
from tests.test_gpu_search import _index, _ln_rows

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def rows60k():
    P = _ln_rows(np.random.default_rng(1234), 60000, 768)
    Q = _ln_rows(np.random.default_rng(4321), 300, 768)
    return P, Q


@pytest.fixture(scope="module")
def oracle60k(rows60k):
    P, Q = rows60k
    return flat_ip_oracle.search(P, Q, 2048)    # the top-k of every smaller k is its prefix


@pytest.mark.parametrize("operand", ["bf16", "fp16"])
@pytest.mark.parametrize("cta_group", [1, 2])
@pytest.mark.parametrize("k", [513, 1000, 2048])
def test_seeded_parity_large_k(rows60k, oracle60k, operand, cta_group, k):
    P, Q = rows60k
    idx = _index(P, operand, cta_group=cta_group)
    D, I = idx.search(Q, k)
    Do, Io = oracle60k
    assert (I == Io[:, :k]).all(), f"{(I != Io[:, :k]).any(1).sum()} queries differ"
    assert (D == Do[:, :k]).all()
    st = idx.stats()
    assert st["nq"] == 300 and st["kprime"] >= k
    assert P.shape[0] >= 4 * st["kprime"]          # the tensor-core path ran, not the small-index brute force
    # ... and certified every query: a large-reservoir compaction that kept too few candidates or set its threshold too
    # high would still give the oracle's answer, through the brute force
    assert st["n_uncertified"] == 0, st


def test_duplicates_and_ties_at_the_k_boundary():
    k = 1000
    rng = np.random.default_rng(5)
    P = _ln_rows(rng, 30000, 768)
    P[20000:20600] = P[0:600]          # exact duplicates -> exact score ties, many of them around rank k
    Q = _ln_rows(np.random.default_rng(6), 64, 768)
    Q[:40] = P[0:40] + 0.01 * Q[:40]
    idx = _index(P)
    D, I = idx.search(Q, k)
    Do, Io = flat_ip_oracle.search(P, Q, k)
    assert (I == Io).all() and (D == Do).all()
    for q in range(40):
        a, b = np.where(I[q] == q)[0], np.where(I[q] == 20000 + q)[0]
        assert len(a) == 1 and len(b) == 1 and b[0] == a[0] + 1   # tie: smaller row first
    assert idx.stats()["kprime"] >= k


def test_tier2_forced_at_k_1000(rows60k, oracle60k):
    """k' just above k (1024 at k = 1000) and one row range per query tile: the tier-1 certificate fails for many queries,
    and tier 2 (reservoir 4096, k' 2016) reruns them from their own thresholds."""
    P, Q = rows60k
    k = 1000
    idx = _index(P, "bf16", kprime=1024, n_splits=1)
    D, I = idx.search(Q, k)
    Do, Io = oracle60k
    assert (I == Io[:, :k]).all() and (D == Do[:, :k]).all()
    st = idx.stats()
    assert st["kprime"] == 1024 and st["n_tier2"] > 0, st
    assert st["n_uncertified"] == 0, st            # tier 2 certified every query tier 1 could not


def test_tier3_forced_at_k_1000():
    """24,576 identical rows at the top of every ranking: neither coarse pass can separate them, so the exact brute force
    answers, ties in ascending row order.  One row range per query tile at tier 1 (with eleven, every range keeps nearly
    all of its rows and the certificate passes there); tier 2 splits the rows into four ranges of 6,144 ties each, more
    than its 4096-entry reservoir holds, so it overflows, is compacted and cannot certify either."""
    k = 1000
    base = _ln_rows(np.random.default_rng(8), 1, 768)
    P = _ln_rows(np.random.default_rng(80), 32768, 768)
    tied = np.arange(P.shape[0]) % 4 != 0
    P[tied] = base
    Q = (base + 0.05 * _ln_rows(np.random.default_rng(9), 32, 768)).astype(np.float32)
    idx = _index(P, n_splits=1)
    D, I = idx.search(Q, k)
    Do, Io = flat_ip_oracle.search_bruteforce(P, Q, k)
    assert (I == Io).all() and (D == Do).all()
    assert tied[I].all() and (np.diff(I, axis=1) > 0).all()
    st = idx.stats()
    assert st["n_tier2"] > 0 and st["n_uncertified"] > 0, st


def test_exact_path_small_index_and_padding_at_k_2048():
    k = 2048
    Q = _ln_rows(np.random.default_rng(13), 100, 768)
    # the validation path (exact=True) on an index the tensor-core path would serve
    P = _ln_rows(np.random.default_rng(12), 30000, 768)
    D, I = _index(P).search_device(torch.from_numpy(Q).cuda(), k, exact=True)
    Do, Io = flat_ip_oracle.search(P, Q, k)
    assert (I.cpu().numpy() == Io).all() and (D.cpu().numpy() == Do).all()
    # k <= n < 4 k': the small-index branch of search() (brute force)
    Ps = _ln_rows(np.random.default_rng(14), 5000, 768)
    idx = _index(Ps)
    D, I = idx.search(Q, k)
    Do, Io = flat_ip_oracle.search(Ps, Q, k)
    assert (I == Io).all() and (D == Do).all()
    assert idx.stats()["n_uncertified"] == 100
    # n < k: labels -1 and scores -FLT_MAX after the n rows
    Pt = _ln_rows(np.random.default_rng(15), 1500, 768)
    D, I = _index(Pt).search(Q, k)
    Do, Io = flat_ip_oracle.search_bruteforce(Pt, Q, k)
    assert (I == Io).all() and (D == Do).all()
    assert (I[:, 1500:] == -1).all() and (D[:, 1500:] == np.finfo(np.float32).min).all()


def test_k_above_2048_is_refused_and_the_index_still_works(rows60k):
    from ance_b200._lib import AnceError
    P, Q = rows60k
    idx = _index(P)
    D0, I0 = idx.search(Q, 200)
    with pytest.raises(AnceError, match="2048"):
        idx.search(Q, 2049)
    with pytest.raises(AnceError, match="2048"):
        idx.search_device(torch.from_numpy(Q).cuda(), 2049, exact=True)
    with pytest.raises(AnceError, match="2048"):      # also where the library is never called
        idx.search(Q[:0], 2049)
    from ance_b200.search import IndexFlatIP
    with pytest.raises(AnceError, match="2048"):
        IndexFlatIP(768).search(Q, 2049)
    D1, I1 = idx.search(Q, 200)
    assert (I1 == I0).all() and (D1 == D0).all()
    Do, Io = flat_ip_oracle.search(P, Q, 200)
    assert (I1 == Io).all() and (D1 == Do).all()


def test_sharded_at_k_1000_on_one_gpu():
    """4 row shards with row offsets and the host merge at k = 1000, then sharded_search with one rank and a query block
    that the k > 512 rule shrinks (256 -> 131 queries: three blocks)."""
    from ance_b200.drivers import run_ann_data_gen as drv
    from ance_b200.search import merge_topk_host
    P = _ln_rows(np.random.default_rng(14), 40001, 768)
    Q = _ln_rows(np.random.default_rng(15), 300, 768)
    W, k = 4, 1000
    order = np.concatenate([np.arange(r, P.shape[0], W) for r in range(W)])
    Pm = P[order]
    Dg, Ig = flat_ip_oracle.search(Pm, Q, k)
    Ds, Is, off = [], [], 0
    qd = torch.from_numpy(Q).cuda()
    for r in range(W):
        n = len(range(r, P.shape[0], W))
        D, I = _index(Pm[off:off + n]).search_device(qd, k, row_offset=off)
        Ds.append(D.cpu().numpy())
        Is.append(I.cpu().numpy())
        off += n
    Dm, Im = merge_topk_host(Ds, Is, k)
    assert (Im == Ig).all() and (Dm == Dg).all()
    idx = _index(Pm)

    def local_search(q, kk, row_offset):
        return idx.search_device(q, kk, row_offset=row_offset)

    ps = drv.sharded_search_start(local_search, Pm.shape[0], qd, k, query_block=256, row_offset=0)
    assert ps.QB == 131
    assert (ps.finish() == Ig).all()


def test_offline_evaluation_default_top_1000_and_topk_training_1000(tmp_path):
    """`evaluate_dumps` with its default topN = 1000 on `--inference` dumps of a corpus larger than 4 k', against the
    notebook loop on the oracle's top-1000; a refresh with `--topk_training 1000` against the post-processing oracle on
    the oracle's top-1000; `--topk_training 4096` refused before anything is encoded."""
    from ance_b200 import evaluation as ev
    from ance_b200.drivers import run_ann_data_gen as drv
    from tests.test_evaluation import _notebook_eval
    from tests.test_gpu_driver import _argv, _make_world
    import random
    data, ckpt, caches, train_pos, dev_pos, *_ = _make_world(tmp_path, n_p=6000, n_q=120, n_dev=40)
    bad = tmp_path / "refused"
    with pytest.raises(SystemExit):
        drv.main(_argv(data, ckpt, bad, tmp_path, extra=("--topk_training", "4096")))
    assert not bad.exists()
    out = tmp_path / "ann"
    drv.main(_argv(data, ckpt, out, tmp_path, extra=("--inference",)))
    q, q2id = ev.load_dumps(str(out), "dev_query_0_")
    p, p2id = ev.load_dumps(str(out), "passage_0_")
    assert p.shape == (6000, 768) and p.shape[0] > 4 * 1440    # k' of fp16 operands at k = 1000
    _, Io = flat_ip_oracle.search(np.ascontiguousarray(p), np.ascontiguousarray(q), 1000)
    res = ev.evaluate_dumps(str(out), 0, dev_pos)
    want = _notebook_eval(q2id, p2id, dev_pos, Io, 1000)
    assert "recall@1000" in res["full_rank"]
    for key, v in want.items():
        assert res["full_rank"][key] == pytest.approx(v, abs=1e-12), key
    # a refresh that searches 1000 neighbours per training query
    out2 = tmp_path / "ann2"
    drv.main(_argv(data, ckpt, out2, tmp_path, extra=("--topk_training", "1000")))
    text = open(out2 / "ann_training_data_0").read()
    args = drv.get_arguments(_argv(data, ckpt, out2, tmp_path))
    drv.set_env(args)
    _, _, model = drv.load_model(args, str(ckpt))
    be = drv.B200Backend(args, model)
    P, p2id = be.encode(str(data / "passages"), False)
    Qt, q2id = be.encode(str(data / "train-query"), True)
    _, I = flat_ip_oracle.search(P.cpu().numpy(), Qt.cpu().numpy(), 1000)
    rng = random.Random(0)
    negs, _, _ = refresh_oracle.generate_negatives(q2id, p2id, train_pos, I, set(q2id.tolist()), 5, False, rng)
    want_text = "".join(refresh_oracle.training_data_lines(q2id, train_pos, negs, set(q2id.tolist()), rng))
    assert text == want_text
    assert 0.0 <= json.load(open(out2 / "ann_ndcg_0"))["ndcg"] <= 1.0
