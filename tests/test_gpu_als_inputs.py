"""GPU: the ALS half-step on ratings bf16 cannot represent and on rows cut at the chunk / MMA boundaries, through every
kernel the library can select, against the fp64 C oracle; the split-form entry point; the Gram against an entrywise
error bound.

The tensor-core kernels carry a rating as bf16(r) + bf16(r - bf16(r)); integer ratings make the low part zero, so
every route here also runs the non-integer kinds of tests.util.draw_ratings.  Each route case checks with
torch.profiler which kernels ran, so a change to the dispatch cannot quietly turn it into a duplicate of another case.
Tolerances as in test_gpu_als.py -- explicit: rel-L2 <= 2e-5 and max-abs <= 1e-4 * max|x| (here without the absolute
floor of 1: an explicit half-step is linear in the ratings); implicit: IMPL_TOL.

HALS_FORCE_SIMT is read once per process, so the CUDA-core kernels at ranks 64 / 128 run in a child process
(this module run as a script); everything else runs in-process.
"""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from oracle import als_oracle, c_oracle
from tests.test_gpu_als import HS_ABS, HS_REL, IMPL_TOL, _mods, _nat, assert_close, gpu_half_step
from tests.util import RATING_KINDS, RATING_SCALE, assert_ran, bf16_exact, draw_ratings, launched_kernels

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# Destination rows of the boundary matrix: empty rows; 1 rating; around the 16-rating MMA step and the 32-rating chunk
# (a row's last chunk is the one with cnt <= 32); rows longer than SEG, cut into equal slices except a shorter last one
# (97 -> 49 + 48, 1100 -> 11 x 92 + 88; 1700 -> 18 slices: the slot pre-sum of rows with more than 16).
ROW_LENS = (0, 1, 15, 16, 17, 0, 31, 32, 33, 63, 64, 65, 0, 97, 128, 151, 300, 1100, 1700, 0)
N_ROWS, N_SRC, SEG = len(ROW_LENS), 300, 96
EMPTY = np.array([n == 0 for n in ROW_LENS])
REG = 0.1
IMPL_REG, IMPL_ALPHA = 0.05, 40.0
MAIN_KERNELS = ("als_ws64_kernel", "als_ws128_kernel", "als_tc64_kernel", "als_tc128_kernel", "als_build_solve_kernel")


def boundary_case(kind, k):
    """(dst rows, src cols, ratings, source factors) of the boundary matrix, in shuffled COO order."""
    rng = np.random.default_rng(3)
    rows = np.repeat(np.arange(N_ROWS), ROW_LENS)
    cols = rng.integers(0, N_SRC, rows.size)
    start = np.concatenate([[0], np.cumsum(ROW_LENS)])
    cols[start[1]] = N_SRC - 1                                  # the last source row
    cols[start[2]] = 0
    cols[start[4]: start[4] + 5] = cols[start[4]]               # duplicate (row, column) pairs ...
    cols[start[8] + 32] = cols[start[8]]                        # ... one of them alone in the row's last chunk
    r = draw_ratings(kind, rows.size, np.random.default_rng(RATING_KINDS.index(kind)))
    if kind != "int":
        assert (~bf16_exact(r)).mean() > 0.5, "most ratings must need the low bf16 part"
    perm = rng.permutation(rows.size)
    return rows[perm], cols[perm], r[perm], als_oracle.init_factors(N_SRC, k, 7)


def oracle_half_step(rows, cols, r, X, implicit=False):
    rp, ci, v = als_oracle.coo_to_csr(rows, cols, r, N_ROWS)
    if implicit:
        return c_oracle.als_half_step(rp, ci, v, X, IMPL_REG, implicit=True, alpha=IMPL_ALPHA)
    return c_oracle.als_half_step(rp, ci, v, X, REG)


def implicit_alpha(kind):
    # the confidence c = alpha |r| stays in the range IMPL_TOL is stated for, whatever the ratings' scale
    return IMPL_ALPHA / RATING_SCALE.get(kind, 1.0)


def check_plan(plan):
    assert plan.n_long == 6 and int(plan.host["long_nseg"][: plan.n_long].max()) > 16
    it = plan.host
    sl = it["item_slot"][: plan.n_items] >= 0
    lens = it["item_len"][: plan.n_items][sl]
    assert lens.min() < lens.max(), "some sliced row must end in a shorter slice"


def check_main_kernel(names, kernels):
    assert_ran(names, *kernels, absent=[m for m in MAIN_KERNELS if not kernels[0].startswith(m)])


# route -> (rank, plan with packed ratings, kernels that must run; the first is the main kernel)
EXPLICIT_ROUTES = {
    "ws64": (64, True, ("als_ws64_kernel", "als_slot_group_sum_kernel", "als_reduce_solve64_warp_kernel")),
    "ws128": (128, True, ("als_ws128_kernel", "als_slot_group_sum_kernel", "als_reduce_solve128_kernel")),
    "tc64": (64, False, ("als_tc64_kernel", "als_slot_group_sum_kernel", "als_reduce_solve64_kernel")),
    "tc128": (128, False, ("als_tc128_kernel", "als_slot_group_sum_kernel", "als_reduce_solve128_kernel")),
}


@pytest.mark.parametrize("kind", RATING_KINDS)
@pytest.mark.parametrize("route", list(EXPLICIT_ROUTES))
def test_explicit_tensor_core_route_matches_oracle(route, kind):
    """ws64 / ws128: the default plan.  tc64 / tc128: a plan without packed ratings (the round-1 kernels split the
    fp32 ratings themselves).  A second call is bit-identical."""
    k, packed, kernels = EXPLICIT_ROUTES[route]
    rows, cols, r, X = boundary_case(kind, k)
    with launched_kernels() as names:
        got, plan = gpu_half_step(rows, cols, r, N_ROWS, X, REG, seg_len=SEG, packed=packed)
    check_main_kernel(names, kernels)
    check_plan(plan)
    assert_close(got, oracle_half_step(rows, cols, r, X), floor=0.0)
    assert not got[EMPTY].any(), "rows without ratings are zero"
    again, _ = gpu_half_step(rows, cols, r, N_ROWS, X, REG, seg_len=SEG, packed=packed)
    assert np.array_equal(got, again)


# route -> (rank, plan packed for implicit feedback, kernels that must run)
IMPLICIT_ROUTES = {
    "ws64": (64, True, ("als_ws64_kernel", "als_slot_group_sum_kernel", "als_reduce_solve64_warp_kernel")),
    "ws128": (128, True, ("als_ws128_kernel", "als_slot_group_sum_kernel", "als_reduce_solve128_kernel")),
    # a plan not packed for implicit feedback: the CUDA-core kernel (include/hals_b200.h, hals_als_plan.vals_scale)
    "simt64": (64, False, ("als_build_solve_kernel<64,true,true>", "als_reduce_solve_kernel<64>")),
    "simt128": (128, False, ("als_build_solve_kernel<128,true,true>", "als_reduce_solve_kernel<128>")),
}


@pytest.mark.parametrize("kind", RATING_KINDS)
@pytest.mark.parametrize("route", list(IMPLICIT_ROUTES))
def test_implicit_route_matches_oracle(route, kind):
    k, tc, kernels = IMPLICIT_ROUTES[route]
    rows, cols, r, X = boundary_case(kind, k)
    alpha = implicit_alpha(kind)
    run = lambda: gpu_half_step(rows, cols, r, N_ROWS, X, IMPL_REG, implicit=True, alpha=alpha, seg_len=SEG,
                                plan_implicit=tc)
    with launched_kernels() as names:
        got, plan = run()
    check_main_kernel(names, kernels)
    check_plan(plan)
    rp, ci, v = als_oracle.coo_to_csr(rows, cols, r, N_ROWS)
    want = c_oracle.als_half_step(rp, ci, v, X, IMPL_REG, implicit=True, alpha=alpha)
    assert_close(got, want, **IMPL_TOL[tc])
    assert not got[EMPTY].any()
    if tc:
        assert np.array_equal(got, run()[0])


@pytest.mark.parametrize("implicit", [False, True])
def test_unaligned_source_takes_the_scalar_gather(implicit):
    """Rank 16 with the source factors one float into a larger buffer: the launcher must leave the 16-byte gather."""
    k = 16
    rows, cols, r, X = boundary_case("decimal", k)
    kw = dict(implicit=True, alpha=IMPL_ALPHA) if implicit else {}
    reg = IMPL_REG if implicit else REG
    with launched_kernels() as names:
        got, _ = gpu_half_step(rows, cols, r, N_ROWS, X, reg, seg_len=SEG, src_offset=1, **kw)
    imp = str(implicit).lower()
    assert_ran(names, f"als_build_solve_kernel<16,{imp},false>", "als_reduce_solve_kernel<16>",
               absent=(f"als_build_solve_kernel<16,{imp},true>",))
    assert_close(got, oracle_half_step(rows, cols, r, X, implicit), **(IMPL_TOL[False] if implicit else dict(floor=0.0)))


@pytest.mark.parametrize("k", [64, 128])
def test_split_half_step_contract(k):
    """hals_als_half_step_split: the same solution as hals_als_half_step, bit for bit (the same kernel; the stateless
    call only splits the source first); dst_hl holds the split of every solved row; rows without ratings are not
    touched in either output."""
    _, csr = _mods()
    nat = _nat()
    L = nat.lib()
    dev = torch.device("cuda")
    rows, cols, r, X = boundary_case("decimal", k)
    ref, _ = gpu_half_step(rows, cols, r, N_ROWS, X, REG, seg_len=SEG)
    t = lambda a: torch.as_tensor(a).to(dev)
    shard = csr.build_csr(t(rows), t(cols), t(r), N_ROWS)
    plan = csr.AlsPlanHandle(shard, k, SEG, n_src=N_SRC)
    src = t(X)
    src_hl = torch.zeros((N_SRC + 1, 2 * k), dtype=torch.bfloat16, device=dev)      # row N_SRC stays zero
    nat.check(L.hals_als_split_factors(nat.ptr(src), N_SRC, k, nat.ptr(src_hl), nat.current_stream()))
    dst = torch.full((N_ROWS, k), 7.0, dtype=torch.float32, device=dev)            # poison
    dst_hl = torch.full((N_ROWS, 2 * k), -3.0, dtype=torch.bfloat16, device=dev)
    with launched_kernels() as names:
        nat.check(L.hals_als_half_step_split(nat.ptr(shard.colidx), N_ROWS, nat.ptr(src_hl), N_SRC, nat.ptr(dst),
                                             nat.ptr(dst_hl), k, REG, plan.struct, nat.ptr(plan.workspace),
                                             plan.workspace_bytes, nat.current_stream()), "hals_als_half_step_split")
    reduce = "als_reduce_solve64_warp_kernel" if k == 64 else "als_reduce_solve128_kernel"
    assert_ran(names, f"als_ws{k}_kernel", reduce, absent=("split_bf16_kernel",))
    solved = ~EMPTY
    got = dst.cpu().numpy()
    assert np.array_equal(got[solved], ref[solved])
    assert (got[EMPTY] == 7.0).all()
    want_hl = torch.empty_like(dst_hl)
    nat.check(L.hals_als_split_factors(nat.ptr(dst), N_ROWS, k, nat.ptr(want_hl), nat.current_stream()))
    got_hl = dst_hl.view(torch.int16).cpu().numpy()
    assert np.array_equal(got_hl[solved], want_hl.view(torch.int16).cpu().numpy()[solved])
    assert (dst_hl[torch.from_numpy(EMPTY).to(dev)] == -3.0).all()


# --- Gram ------------------------------------------------------------------------------------------------------------

def gram_input(n, k):
    # columns from 2^-6 to 2^6: an entry is checked against its own scale, not the largest diagonal entry
    rng = np.random.default_rng(n * 1000 + k)
    return (rng.standard_normal((n, k)) * 2.0 ** np.linspace(-6, 6, k)).astype(np.float32)


def gpu_gram(Y):
    als_engine, _ = _mods()
    dev = torch.device("cuda")
    k = Y.shape[1]
    out = torch.empty((k, k), dtype=torch.float32, device=dev)
    ws = torch.empty(int(_nat().lib().hals_gram_workspace_bytes(k)), dtype=torch.uint8, device=dev)
    als_engine.native_gram(torch.from_numpy(Y).to(dev), out, ws)
    torch.cuda.synchronize()
    return out.cpu().numpy()


def gram_chain(n, tc):
    """Most rows one fp32 partial sum of the Gram kernels accumulates (csrc/als_misc.cu, csrc/gram_tc.cu)."""
    cdiv = lambda a, b: -(-a // b)
    if tc:
        grid = min(torch.cuda.get_device_properties(0).multi_processor_count, cdiv(n, 32), 148)
        return cdiv(cdiv(n, grid), 32) * 32
    return cdiv(n, min(max(cdiv(n, 256), 1), 592))


def assert_gram_bound(G, Y, tc):
    """|G - G64| <= c (|Y|^T |Y|) entrywise.
    Tensor cores: h = bf16(y), l = bf16(y - h), so |y - h| <= 2^-8 |y| and |y - h - l| <= 2^-16 |y|; the kernel sums
    h_i h_j + h_i l_j + l_i h_j = s_i s_j - l_i l_j (s = h + l), which misses y_i y_j by at most
    (2 * 2^-16 + 2^-16) |y_i y_j| to first order: the two split residuals and the dropped l l^T.
    Both paths: a partial sum accumulates at most m products in fp32 (<= m * 2^-24 of the sum of their magnitudes);
    the partials are added in fp64 and the result rounded once to fp32 (2^-24)."""
    Yd = Y.astype(np.float64)
    want = als_oracle.gram_f64(Y)
    mag = np.abs(Yd).T @ np.abs(Yd)
    c = (3 * 2.0 ** -16 * 1.01 if tc else 0.0) + (gram_chain(Y.shape[0], tc) + 2) * 2.0 ** -24
    ratio = np.abs(G.astype(np.float64) - want) / (c * mag)
    assert np.isfinite(G).all()
    assert ratio.max() <= 1.0, (ratio.max(), np.unravel_index(ratio.argmax(), ratio.shape))


@pytest.mark.parametrize("n", [2047, 2048, 2049, 4097])
@pytest.mark.parametrize("k", [64, 128])
def test_gram_across_the_tensor_core_switch(k, n):
    """Ranks 64 / 128 switch to gram_tc_kernel at 2048 rows; 2049 and 4097 leave a ragged tail of a 32-row stage."""
    Y = gram_input(n, k)
    with launched_kernels() as names:
        G = gpu_gram(Y)
    tc = n >= 2048
    if tc:
        assert_ran(names, f"gram_tc_kernel<{k}>", f"gram_tc_finish_kernel<{k}>", absent=("gram_partial_kernel",))
    else:
        assert_ran(names, f"gram_partial_kernel<{k}>", "gram_reduce_kernel", absent=("gram_tc_kernel",))
    assert_gram_bound(G, Y, tc)


@pytest.mark.parametrize("k", [1, 3, 33, 100])
def test_gram_cuda_core_ranks(k):
    Y = gram_input(10_000, k)
    with launched_kernels() as names:
        G = gpu_gram(Y)
    kp = 16 if k <= 16 else 32 if k <= 32 else 64 if k <= 64 else 128
    assert_ran(names, f"gram_partial_kernel<{kp}>", absent=("gram_tc_kernel",))
    assert_gram_bound(G, Y, False)


# --- HALS_FORCE_SIMT=1: the CUDA-core kernels at ranks 64 / 128, in a child process ---------------------------------

SIMT_GRAM_N = (2048, 4097, 10_000)


def _force_simt_child(out):
    """Runs with HALS_FORCE_SIMT=1: every explicit half-step of the boundary matrix and the Gram at ranks 64 / 128,
    saved (results and launched kernel names) to `out` for the parent's tests."""
    res = {}
    for k in (64, 128):
        for kind in RATING_KINDS:
            rows, cols, r, X = boundary_case(kind, k)
            with launched_kernels() as names:
                res[f"x_{k}_{kind}"], _ = gpu_half_step(rows, cols, r, N_ROWS, X, REG, seg_len=SEG)
            res[f"names_x_{k}_{kind}"] = np.array(names)
        for n in SIMT_GRAM_N:
            with launched_kernels() as names:
                res[f"g_{k}_{n}"] = gpu_gram(gram_input(n, k))
            res[f"names_g_{k}_{n}"] = np.array(names)
    np.savez(out, **res)


@pytest.fixture(scope="module")
def force_simt(tmp_path_factory):
    out = tmp_path_factory.mktemp("force_simt") / "out.npz"
    cmd = [sys.executable] + (["-s"] if sys.flags.no_user_site else []) + ["-m", "tests.test_gpu_als_inputs", str(out)]
    p = subprocess.run(cmd, cwd=ROOT, env=dict(os.environ, HALS_FORCE_SIMT="1"), capture_output=True, text=True,
                       timeout=900)
    assert p.returncode == 0, p.stdout[-4000:] + p.stderr[-4000:]
    with np.load(out) as z:
        return {n: z[n] for n in z.files}


@pytest.mark.parametrize("kind", RATING_KINDS)
@pytest.mark.parametrize("k", [64, 128])
def test_explicit_cuda_core_route_matches_oracle(force_simt, k, kind):
    check_main_kernel(list(force_simt[f"names_x_{k}_{kind}"]),
                      (f"als_build_solve_kernel<{k},false,true>", f"als_reduce_solve_kernel<{k}>"))
    rows, cols, r, X = boundary_case(kind, k)
    got = force_simt[f"x_{k}_{kind}"]
    assert_close(got, oracle_half_step(rows, cols, r, X), HS_REL, HS_ABS, floor=0.0)
    assert not got[EMPTY].any()


@pytest.mark.parametrize("n", SIMT_GRAM_N)
@pytest.mark.parametrize("k", [64, 128])
def test_cuda_core_gram_at_the_tensor_core_ranks(force_simt, k, n):
    assert_ran(list(force_simt[f"names_g_{k}_{n}"]), f"gram_partial_kernel<{k}>", absent=("gram_tc_kernel",))
    assert_gram_bound(force_simt[f"g_{k}_{n}"], gram_input(n, k), False)


if __name__ == "__main__":
    _force_simt_child(sys.argv[1])
