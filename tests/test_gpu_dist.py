"""GPU, world_size 2, NCCL on one box (skipped with fewer than two GPUs): the sharded ALS fit (row shards + factor
all-gather after every half-step) and the item-sharded hybrid scoring (extrema all-reduce, all-to-all of the
per-shard lists, merge) through the native kernels, against the single-GPU result and the CPU oracle.

SURVEY.md section 4 item 4: "1-GPU result == N-GPU result".  Long rows are sliced differently on a shard than on
the whole matrix, which changes the fp32 summation order of their partial sums, so factors agree to rounding
(rel-L2 <= 1e-5 after 3 sweeps), not bit for bit; against the fp64 oracle the usual 1e-3 / 1e-4 bounds hold.
Run with:  python -m pytest tests/test_gpu_dist.py -m gpu -q   (on a box with two or more GPUs)
"""
import os
import socket

import numpy as np
import pytest
import torch
import torch.multiprocessing as mp

from oracle import als_oracle, c_oracle, hybrid_oracle
from tests.util import rel_l2

pytestmark = pytest.mark.gpu


def _free_port():
    s = socket.socket(); s.bind(("127.0.0.1", 0)); p = s.getsockname()[1]; s.close()
    return p


def _worker(rank, world, port, case, out_dir):
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"; os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    import hybrid_als_twotower_recommender_b200  # noqa: F401
    from hybrid_als_twotower_recommender_b200 import als_engine, scoring
    z = np.load(case)
    U, I, k = int(z["U"]), int(z["I"]), int(z["k"])
    implicit = bool(z["implicit"]) if "implicit" in z.files else False
    eng = als_engine.AlsEngine(z["u"], z["i"], z["r"], U, I, k, 0.1, implicit=implicit, alpha=float(z["alpha"]) if implicit else 1.0,
                               device=dev, dist_rank=rank, world=world, seg_len=int(z["seg"]))
    eng.set_user_factors(z["X0"])
    if implicit:      # fit only: the implicit engine has no RMSE of its own, scoring is covered by the explicit cases
        X, Y = eng.fit(2)
        np.savez(os.path.join(out_dir, f"rank{rank}.npz"), X=X.cpu().numpy(), Y=Y.cpu().numpy())
        dist.barrier()
        dist.destroy_process_group()
        return
    if bool(z["graphs"]):
        assert eng.enable_graphs(), "graph capture of a half-step incl. its NCCL all-gather"
    X, Y = eng.fit(3)
    rmse = eng.rmse(z["u"], z["i"], z["r"])
    # item-sharded scoring on fixed operands (independent of the fit, so that the comparison is exact)
    ib, ie = scoring.shard_items(int(z["Is"]), rank, world)
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    sc = scoring.HybridScorer(t(z["Ua"]), t(z["Ia"][ib:ie]), t(z["Ut"]), t(z["It"][ib:ie]), item_offset=ib,
                              dist_rank=rank, world=world)
    fi, fs = sc.recommend(int(z["topk"]), 0.8, 0.2)
    np.savez(os.path.join(out_dir, f"rank{rank}.npz"), X=X.cpu().numpy(), Y=Y.cpu().numpy(), rmse=rmse,
             fi=fi.cpu().numpy(), fs=fs.cpu().numpy(), ub=eng.user_bounds, ibn=eng.item_bounds)
    dist.barrier()
    dist.destroy_process_group()


def _single(case):
    import hybrid_als_twotower_recommender_b200  # noqa: F401
    from hybrid_als_twotower_recommender_b200 import als_engine, scoring
    z = np.load(case)
    U, I, k = int(z["U"]), int(z["I"]), int(z["k"])
    eng = als_engine.AlsEngine(z["u"], z["i"], z["r"], U, I, k, 0.1, seg_len=int(z["seg"]))
    eng.set_user_factors(z["X0"])
    X, Y = eng.fit(3)
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
    sc = scoring.HybridScorer(t(z["Ua"]), t(z["Ia"]), t(z["Ut"]), t(z["It"]))
    idx, s = sc.recommend(int(z["topk"]), 0.8, 0.2)
    return X.cpu().numpy(), Y.cpu().numpy(), eng.rmse(z["u"], z["i"], z["r"]), idx.cpu().numpy(), s.cpu().numpy()


# (CUDA-graph capture of the half-steps with their all-gathers is exercised by bench.py at N > 1; under mp.spawn the
# capture of an NCCL collective did not return on the test box, so it is not repeated here.)
@pytest.mark.parametrize("k,graphs", [(64, False), (128, False)])
def test_two_gpu_fit_and_scoring_match_one_gpu_and_oracle(tmp_path, k, graphs):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs on one box")
    rng = np.random.default_rng(40 + k)
    U, I, nnz = 5000, 800, 160_000
    p = 1.0 / np.arange(1, I + 1); p /= p.sum()
    u, i = rng.integers(0, U, nnz), rng.choice(I, nnz, p=p)
    r = rng.integers(1, 6, nnz).astype(np.float32)
    X0 = als_oracle.init_factors(U, k, 3)
    Us, Is, ka, kt, topk = 700, 9000, 128, 50, 100          # scoring operands: tensor-core path on every shard
    Ua, Ia = rng.normal(0, ka ** -0.5, (Us, ka)).astype(np.float32), rng.normal(0, 1, (Is, ka)).astype(np.float32)
    Ut, It = rng.normal(0, 1, (Us, kt)).astype(np.float32), rng.normal(0, 1, (Is, kt)).astype(np.float32)
    case = str(tmp_path / "case.npz")
    np.savez(case, u=u, i=i, r=r, U=U, I=I, k=k, X0=X0, seg=1024, graphs=graphs, Ua=Ua, Ia=Ia, Ut=Ut, It=It, Is=Is,
             topk=topk)
    mp.spawn(_worker, args=(2, _free_port(), case, str(tmp_path)), nprocs=2, join=True)
    outs = [np.load(tmp_path / f"rank{q}.npz") for q in range(2)]
    # every rank holds the same full factor matrices after the all-gathers
    assert np.array_equal(outs[0]["X"], outs[1]["X"]) and np.array_equal(outs[0]["Y"], outs[1]["Y"])
    assert outs[0]["ub"][-1] == U and outs[0]["ibn"][-1] == I and 0 < outs[0]["ub"][1] < U
    X1, Y1, rmse1, idx1, s1 = _single(case)
    assert rel_l2(outs[0]["X"], X1) <= 1e-5 and rel_l2(outs[0]["Y"], Y1) <= 1e-5
    assert abs(float(outs[0]["rmse"]) - rmse1) <= 1e-5
    Xo, Yo = als_oracle.als_fit(u, i, r, U, I, k, 3, 0.1, X0, half_step=c_oracle.als_half_step)
    assert rel_l2(outs[0]["X"], Xo) <= 1e-3 and rel_l2(outs[0]["Y"], Yo) <= 1e-3
    assert abs(float(outs[0]["rmse"]) - als_oracle.rmse(Xo, Yo, u, i, r)) <= 1e-4
    # scoring: rank q owns the merged lists of the q-th half of the users
    per = (Us + 1) // 2
    assert outs[0]["fi"].shape == (per, topk)
    got_i = np.concatenate([outs[0]["fi"], outs[1]["fi"]])[:Us]
    got_s = np.concatenate([outs[0]["fs"], outs[1]["fs"]])[:Us]
    # both paths end in exact fp32 scores, but a user the bf16 bound cannot prove is re-run by the CUDA-core kernel,
    # whose sequential fmaf differs from the warp-shuffle sum in the last bit -- and which users those are depends on
    # the shard.  Lists must agree except where two neighbouring scores are within that last bit.
    assert np.allclose(got_s, s1, atol=1e-6)
    diff = got_i != idx1
    assert diff.mean() < 2e-3, diff.mean()
    assert np.abs(got_s[diff] - s1[diff]).max(initial=0.0) <= 2e-6
    wi, ws = hybrid_oracle.hybrid_topk_dense(Ua, Ia, Ut, It, 0.8, 0.2, topk)
    assert np.allclose(got_s, ws, atol=1e-5) and (got_i == wi).mean() > 0.995


def test_two_gpu_implicit_rank128_matches_one_gpu_and_oracle(tmp_path):
    """Config 4's path at N > 1: Hu-Koren half-steps on the tensor cores (rank 128), tensor-core Gram on every rank,
    fp32 factor all-gather.  Two sweeps vs the single-GPU engine and vs the fp64 oracle."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs on one box")
    import hybrid_als_twotower_recommender_b200  # noqa: F401
    from hybrid_als_twotower_recommender_b200 import als_engine
    rng = np.random.default_rng(77)
    U, I, nnz, k, alpha = 4000, 2500, 120_000, 128, 10.0
    p = 1.0 / np.arange(1, I + 1); p /= p.sum()
    u, i = rng.integers(0, U, nnz), rng.choice(I, nnz, p=p)
    r = (rng.geometric(0.4, nnz) * rng.choice([1, 1, 1, -1, 0], nnz)).astype(np.float32)
    X0 = als_oracle.init_factors(U, k, 5)
    case = str(tmp_path / "case.npz")
    np.savez(case, u=u, i=i, r=r, U=U, I=I, k=k, X0=X0, seg=1024, graphs=False, implicit=True, alpha=alpha)
    mp.spawn(_worker, args=(2, _free_port(), case, str(tmp_path)), nprocs=2, join=True)
    outs = [np.load(tmp_path / f"rank{q}.npz") for q in range(2)]
    assert np.array_equal(outs[0]["X"], outs[1]["X"]) and np.array_equal(outs[0]["Y"], outs[1]["Y"])
    eng = als_engine.AlsEngine(u, i, r, U, I, k, 0.1, implicit=True, alpha=alpha, seg_len=1024)
    eng.set_user_factors(X0)
    X1, Y1 = eng.fit(2)
    assert rel_l2(outs[0]["X"], X1.cpu().numpy()) <= 2e-5 and rel_l2(outs[0]["Y"], Y1.cpu().numpy()) <= 2e-5
    Xo, Yo = als_oracle.als_fit(u, i, r, U, I, k, 2, 0.1, X0, implicit=True, alpha=alpha,
                                half_step=c_oracle.als_half_step)
    assert rel_l2(outs[0]["X"], Xo) <= 1e-3 and rel_l2(outs[0]["Y"], Yo) <= 1e-3
