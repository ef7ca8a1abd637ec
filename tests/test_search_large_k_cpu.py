"""CPU side of k up to 2048: the two oracles at large k, the drivers' `--topk_training` check, and the sharded search's
query-block rule for k > 512 under a two-rank gloo group."""
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from oracle import flat_ip_oracle


@pytest.mark.parametrize("k", [1000, 2048])
@pytest.mark.parametrize("n", [700, 1800, 5000])
def test_python_and_c_oracles_agree_at_large_k(k, n):
    rng = np.random.default_rng(n + k)
    P = rng.standard_normal((n, 48)).astype(np.float32)
    P[n // 2:n // 2 + 40] = P[:40]                      # exact ties
    Q = rng.standard_normal((12, 48)).astype(np.float32)
    Db, Ib = flat_ip_oracle.search_bruteforce(P, Q, k)
    Dc, Ic = flat_ip_oracle.search_c(P, Q, k)
    Ds, Is = flat_ip_oracle.search(P, Q, k)
    assert (Ic == Ib).all() and (Dc == Db).all()
    assert (Is == Ib).all() and (Ds == Db).all()
    if n < k:
        assert (Ib[:, n:] == -1).all() and (Db[:, n:] == np.finfo(np.float32).min).all()


_REQUIRED = ["--data_dir", "d", "--training_dir", "t", "--init_model_dir", "i", "--model_type", "rdot_nll",
             "--output_dir", "o", "--cache_dir", "c"]
_DPR_EXTRA = ["--passage_path", "p", "--test_qa_path", "q", "--trivia_test_qa_path", "tq"]


@pytest.mark.parametrize("dpr", [False, True])
def test_topk_training_is_checked_when_parsing(dpr, capsys):
    from ance_b200.drivers import run_ann_data_gen as drv
    from ance_b200.drivers import run_ann_data_gen_dpr as drv_dpr
    from ance_b200.search import MAX_K
    parse = drv_dpr.get_arguments if dpr else drv.get_arguments
    argv = _REQUIRED + (_DPR_EXTRA if dpr else [])
    assert MAX_K == 2048
    assert parse(argv).topk_training == 500
    for k in (1, 1000, 2048):
        assert parse(argv + ["--topk_training", str(k)]).topk_training == k
    for bad in ("2049", "4096", "0", "-3"):
        with pytest.raises(SystemExit):
            parse(argv + ["--topk_training", bad])
        assert "2048" in capsys.readouterr().err


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _worker(rank, world, port, tmpdir):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        from ance_b200.drivers import run_ann_data_gen as drv
        n_p, n_q, k = 2600, 46, 1000
        rng = np.random.default_rng(17)
        P = rng.standard_normal((n_p, 24)).astype(np.float32)
        Q = rng.standard_normal((n_q, 24)).astype(np.float32)
        P[1500:1530] = P[7:37]                      # ties that straddle shards
        mine = np.arange(rank, n_p, world)
        p_loc = P[mine]
        p2id = drv.all_gather_ids(mine, torch.device("cpu"))
        q_all = torch.from_numpy(Q)

        def local_search(q, kk, row_offset):
            D, I = flat_ip_oracle.search_bruteforce(p_loc, q.numpy(), kk)
            return torch.from_numpy(D), torch.from_numpy(np.where(I >= 0, I + row_offset, -1))

        one = drv.sharded_search_start(local_search, p_loc.shape[0], q_all, k, query_block=1 << 20)
        assert one.QB == 46                          # 2^20 * 512 // 1000 queries: one block
        I_one = one.finish()
        shrunk = drv.sharded_search_start(local_search, p_loc.shape[0], q_all, k, query_block=40)
        assert shrunk.QB == 20                       # 40 * 512 // 1000 = 20: three blocks, the last one ragged
        I_blk = shrunk.finish()
        small = drv.sharded_search_start(local_search, p_loc.shape[0], q_all, 100, query_block=40)
        assert small.QB == 40                        # k <= 512: the block is what the caller asked for
        small.finish()
        if rank == 0:
            _, Ig = flat_ip_oracle.search_bruteforce(P[p2id], Q, k)
            assert (I_one == Ig).all() and (I_blk == I_one).all()
            np.save(os.path.join(tmpdir, "ok.npy"), np.ones(1))
    finally:
        dist.destroy_process_group()


def test_sharded_search_large_k_gloo(tmp_path):
    mp.spawn(_worker, args=(2, _free_port(), str(tmp_path)), nprocs=2, join=True)
    assert (tmp_path / "ok.npy").exists()
