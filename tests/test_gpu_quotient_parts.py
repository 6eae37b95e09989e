"""The quotient by coset parts on the device (b200zk_coeff_to_extended_parts, b200zk_graph_evaluate_part,
b200zk_extended_parts_to_coeff): every part is the strided slice of the full extended coset, a program evaluated on a part is
the strided slice of its full-domain evaluation, and the recombined parts are the oracle's extended_to_coeff, byte for byte."""
import json
import os
import random
import sys

import numpy as np
import pytest

from oracle import oracle as O
from quotient_programs import C_ADD, C_MUL, R_MOD, S_ADVICE, S_FIXED, S_INTER, S_PREV, S_Y, ZETA, omega_of, random_program
from h_terms_programs import logup_terms_program, permutation_terms_program

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
THREADS = os.cpu_count() or 8


@pytest.fixture(autouse=True)
def one_stream(ctx):
    """Library and torch on one stream, so torch copies and the library's kernels are ordered."""
    import torch

    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        ctx.set_stream(s.cuda_stream)
        yield
        ctx.synchronize()
    ctx.set_stream(None)


def dev(a):
    import torch

    return torch.from_numpy(np.ascontiguousarray(a, dtype=np.uint64).view(np.int64)).cuda()


def empty(n):
    import torch

    return torch.empty((n, 4), dtype=torch.int64, device="cuda")


def host(t):
    return t.cpu().numpy().view(np.uint64)


def interleave(parts, J):
    """part-major (J parts of n) -> extended row order r + J*i"""
    return np.ascontiguousarray(np.asarray(parts).reshape(J, -1, 4).transpose(1, 0, 2).reshape(-1, 4))


@pytest.mark.parametrize("k", [1, 4, 10, 16, 20])
@pytest.mark.parametrize("log_j", [0, 1, 2, 3, 4])
def test_coeff_to_extended_parts_are_strided_coset_slices(ctx, zk, k, log_j):
    J, n = 1 << log_j, 1 << k
    dom, dom_o = zk.EvaluationDomain(ctx, J + 1, k), O.EvaluationDomain(J + 1, k)
    assert dom.extended_k == k + log_j and dom.n_parts == J
    cols = [O.fill_fr(n, 300 + 7 * k + log_j + c) for c in range(2)]
    full = [dom_o.coeff_to_extended(c, THREADS) for c in cols]
    dcols = [dev(c) for c in cols]
    for r in range(J):
        host_out = [empty(n)]  # host input, one column
        dom.coeff_to_extended_parts([cols[0]], r, host_out)
        dev_out = [empty(n), empty(n)]  # device inputs, two distinct columns in one call
        dom.coeff_to_extended_parts(dcols, r, dev_out)
        assert np.array_equal(host(host_out[0]), full[0][r::J])
        assert np.array_equal(host(dev_out[0]), full[0][r::J])
        assert np.array_equal(host(dev_out[1]), full[1][r::J])


def test_parts_at_degree_24_hash_to_the_committed_coset_digest(ctx, zk):
    """the input of test_gpu_exact_big.py::test_transforms_exact_at_degree_24, extended by parts: the four parts, interleaved,
    are the committed 2^26 coset"""
    sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
    import make_big_digests as G

    digests = json.load(open(os.path.join(ROOT, "tests", "golden", "big_digests.json")))
    k = 24
    dom = zk.EvaluationDomain(ctx, 5, k)
    J = dom.n_parts
    assert J == 4
    coeffs = dev(G.ntt_inputs(k))
    dom.lagrange_to_coeff(coeffs)
    assert G.sha(host(coeffs)) == digests["lagrange_to_coeff_24"]
    parts = empty(J << k)
    for r in range(J):
        dom.coeff_to_extended_parts([coeffs], r, [parts[r << k:(r + 1) << k]])
    assert G.sha(interleave(host(parts), J)) == digests["coeff_to_extended_26"]


def _full_and_parts(ctx, zk, k, log_j, n_fixed, n_advice, n_instance, seed):
    """random coefficient columns as full cosets (the existing path) and as per-part columns"""
    J, n = 1 << log_j, 1 << k
    dom = zk.EvaluationDomain(ctx, J + 1, k)
    rng = random.Random(seed)
    mk = lambda cnt: [dev(O.fill_fr(n, rng.randrange(1 << 30))) for _ in range(cnt)]
    coeffs = [mk(n_fixed), mk(n_advice), mk(n_instance)]
    full = [[dom.coeff_to_extended(c) for c in group] for group in coeffs]

    def part_cols(r):
        out = []
        for group in coeffs:
            bufs = [empty(n) for _ in group]
            if group:
                dom.coeff_to_extended_parts(group, r, bufs)
            out.append(bufs)
        return out

    return dom, full, part_cols


def _check_programs_by_parts(ctx, zk, k, log_j, programs, n_fixed, n_advice, n_instance, seed, n_challenges=0):
    J, n = 1 << log_j, 1 << k
    dom, full, part_cols = _full_and_parts(ctx, zk, k, log_j, n_fixed, n_advice, n_instance, seed)
    ch = O.fill_fr(max(n_challenges, 1), seed + 1)[:n_challenges]
    beta, gamma, theta, y = (O.fill_fr(1, seed + 10 + i)[0] for i in range(4))
    prev = O.fill_fr(J * n, seed + 20)
    graphs = [ctx.graph(calcs, O.frs_from_ints(consts), rots) for calcs, consts, rots in programs]
    kw = dict(challenges=ch, beta=beta, gamma=gamma, theta=theta, y=y)
    want = dev(prev)
    for g in graphs:  # the full-coset path, PreviousValue chained over the programs
        g.evaluate(want, dom.extended_k, J, fixed=full[0], advice=full[1], instance=full[2], extended_omega=dom.extended_omega, **kw)
    want = host(want)
    for r in range(J):
        fx, ad, ins = part_cols(r)
        vals = dev(prev[r::J])
        for g in graphs:
            g.evaluate_part(vals, k, dom.extended_k, r, fixed=fx, advice=ad, instance=ins, **kw)
        assert np.array_equal(host(vals), want[r::J]), f"part {r}"
    for g in graphs:
        g.release()


@pytest.mark.parametrize("seed,k,log_j", [(1, 6, 2), (2, 10, 3), (3, 3, 4), (4, 12, 1), (5, 8, 0)])
def test_graph_evaluate_part_is_the_strided_full_evaluation(ctx, zk, seed, k, log_j):
    progs = []
    for s in (seed, seed + 100):  # two programs: the second reads the first's values as PreviousValue
        calcs, constants, rotations = random_program(s, 80, 2, 3, 1, 2, 5)
        progs.append((calcs, constants, [0, 1, -1, 2, -2][:len(rotations)]))
    _check_programs_by_parts(ctx, zk, k, log_j, progs, 2, 3, 1, seed, n_challenges=2)


def test_graph_evaluate_part_runs_the_permutation_and_lookup_programs(ctx, zk):
    k, log_j = 9, 2
    n_sets, chunk, n_cols = 3, 2, 5
    perm = permutation_terms_program(n_sets, chunk, n_cols, -((1 << k) - 7))
    _check_programs_by_parts(ctx, zk, k, log_j, [perm], n_cols + 3, n_sets + n_cols, 0, 41)
    look = logup_terms_program(2)
    _check_programs_by_parts(ctx, zk, k, log_j, [look], 3, 2 + 3, 0, 42)


@pytest.mark.parametrize("k,log_j", [(8, 1), (8, 2), (6, 3), (5, 4)])
def test_extended_parts_to_coeff_matches_the_oracle(ctx, zk, k, log_j):
    J, n = 1 << log_j, 1 << k
    dom, dom_o = zk.EvaluationDomain(ctx, J + 1, k), O.EvaluationDomain(J + 1, k)
    h = O.fill_fr(J * n, 500 + k + log_j)
    w_ext, zn = omega_of(dom.extended_k), pow(ZETA, n, R_MOD)
    t_inv = [pow(zn * pow(w_ext, n * t, R_MOD) - 1, -1, R_MOD) for t in range(J)]
    h_int = O.frs_to_ints(h)
    divided = O.frs_from_ints([x * t_inv[i % J] % R_MOD for i, x in enumerate(h_int)])
    want = {False: dom_o.extended_to_coeff(h, THREADS), True: dom_o.extended_to_coeff(divided, THREADS)}
    part_major = np.ascontiguousarray(np.concatenate([h[r::J] for r in range(J)]))
    for divide in (False, True):
        for n_pieces in sorted({1, max(J - 1, 1), J}):
            parts = dev(part_major)
            out = empty(n_pieces * n)
            got = dom.extended_parts_to_coeff(parts, divide, n_pieces, out)
            assert np.array_equal(host(got), want[divide][: n_pieces * n]), (divide, n_pieces)
        parts = dev(part_major)  # in place: the pieces land at the front of the parts buffer
        got = dom.extended_parts_to_coeff(parts, divide)
        assert np.array_equal(host(got), want[divide][: J * n])


def test_invalid_part_arguments_are_rejected_and_the_context_stays_usable(ctx, zk):
    n = 16
    col, out = dev(O.fill_fr(n, 1)), empty(n)
    ptr = lambda t: zk.C.c_void_p(t.data_ptr())
    tab = lambda *ts: (zk.C.c_void_p * len(ts))(*[t.data_ptr() for t in ts])
    L = zk.lib()

    def expect(rc, words):
        assert rc == zk.E_INVALID
        msg = L.b200zk_last_error(ctx._h).decode()
        assert all(w in msg for w in words), msg

    expect(L.b200zk_coeff_to_extended_parts(ctx._h, tab(col), 1, 4, 6, 4, tab(out)), ["part 4", "J = 4"])
    expect(L.b200zk_coeff_to_extended_parts(ctx._h, tab(col), 1, 4, 3, 0, tab(out)), ["extended_k = 3"])
    expect(L.b200zk_coeff_to_extended_parts(ctx._h, tab(col), 1, 4, 29, 0, tab(out)), ["extended_k = 29"])
    expect(L.b200zk_coeff_to_extended_parts(ctx._h, tab(col), 1, 4, 9, 0, tab(out)), ["exceeds the supported maximum of 16"])
    host_out = np.zeros((n, 4), np.uint64)
    host_tab = (zk.C.c_void_p * 1)(host_out.ctypes.data)
    expect(L.b200zk_coeff_to_extended_parts(ctx._h, tab(col), 1, 4, 5, 0, host_tab), ["out[0] must be a device pointer"])
    parts = empty(4 * n)
    expect(L.b200zk_extended_parts_to_coeff(ctx._h, ptr(parts), 4, 6, 5, 1, ptr(parts)), ["n_pieces = 5"])
    expect(L.b200zk_extended_parts_to_coeff(ctx._h, ptr(parts), 4, 3, 1, 1, ptr(parts)), ["extended_k = 3"])
    expect(L.b200zk_extended_parts_to_coeff(ctx._h, ptr(parts), 4, 9, 1, 1, ptr(parts)), ["supported maximum"])
    hp = np.zeros((4 * n, 4), np.uint64)
    expect(L.b200zk_extended_parts_to_coeff(ctx._h, zk.C.c_void_p(hp.ctypes.data), 4, 6, 1, 1, ptr(parts)), ["parts must be a device pointer"])
    expect(L.b200zk_extended_parts_to_coeff(ctx._h, ptr(parts), 4, 6, 1, 1, zk.C.c_void_p(hp.ctypes.data)), ["out must be a device pointer"])
    g = ctx.graph([(C_MUL, (S_ADVICE, 0, 1), (S_PREV, 0, 0), None)], O.frs_from_ints([1]), [0, 1])
    with pytest.raises(zk.B200zkError) as ei:
        g.evaluate_part(dev(O.fill_fr(n, 3)), 4, 6, 4, advice=[col])
    assert ei.value.code == zk.E_INVALID and "part 4" in str(ei.value)
    with pytest.raises(zk.B200zkError):
        g.evaluate_part(dev(O.fill_fr(n, 3)), 4, 9, 0, advice=[col])
    g.release()
    # still usable: one valid call gives the oracle's part
    dom, dom_o = zk.EvaluationDomain(ctx, 5, 4), O.EvaluationDomain(5, 4)
    c = O.fill_fr(n, 9)
    o = [empty(n)]
    dom.coeff_to_extended_parts([c], 3, o)
    assert np.array_equal(host(o[0]), dom_o.coeff_to_extended(c)[3::4])


# ------------------------------------------------------------------------------------------------ multi-GPU
def _worker(rank, world, port, q):
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import importlib

    import torch
    import torch.distributed as dist

    zk = importlib.import_module("scroll-prover_b200")
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    ctx = zk.Context(rank)
    s = torch.cuda.Stream()
    ok = True
    with torch.cuda.stream(s):
        ctx.set_stream(s.cuda_stream)
        ctx.comm_init_torch(dist)
        k = 12
        dom = zk.EvaluationDomain(ctx, 5, k)  # J = 4
        n, J = 1 << k, dom.n_parts
        d = lambda a: torch.from_numpy(np.ascontiguousarray(a, dtype=np.uint64).view(np.int64)).cuda()
        cols = [d(O.fill_fr(n, 700 + i)) for i in range(3)]  # coefficient form, the same on every rank
        prog = [(C_MUL, (S_ADVICE, 0, 1), (S_ADVICE, 1, 2), None), (C_ADD, (S_INTER, 0, 0), (S_FIXED, 0, 0), None),
                (C_MUL, (S_PREV, 0, 0), (S_Y, 0, 0), None), (C_ADD, (S_INTER, 2, 0), (S_INTER, 1, 0), None)]
        g = ctx.graph(prog, O.frs_from_ints([0, 1]), [0, 1, -1])
        yv = O.fr_from_int(777)

        def eval_parts(buf, parts):
            for r in parts:
                pc = [torch.empty((n, 4), dtype=torch.int64, device="cuda") for _ in cols]
                dom.coeff_to_extended_parts(cols, r, pc)
                g.evaluate_part(buf[r * n:(r + 1) * n], k, dom.extended_k, r, fixed=[pc[2]], advice=[pc[0], pc[1]], y=yv)

        single = torch.zeros((J * n, 4), dtype=torch.int64, device="cuda")
        eval_parts(single, range(J))
        want = dom.extended_parts_to_coeff(single, True).cpu().numpy()
        first, cnt = zk.shard_range(J * n, rank, world)
        ok &= first % n == 0 and cnt % n == 0  # world | J: a rank's slice is whole parts
        sharded = torch.zeros((J * n, 4), dtype=torch.int64, device="cuda")
        eval_parts(sharded, range(first // n, (first + cnt) // n))
        ctx.allgather_rows(sharded, dom.extended_k)
        got = dom.extended_parts_to_coeff(sharded, True).cpu().numpy()
        ok &= bool(np.array_equal(got, want))
        ctx.synchronize()
        g.release()
    ctx.set_stream(None)
    q.put((rank, ok))
    dist.barrier()
    ctx.close()
    dist.destroy_process_group()


@pytest.mark.parametrize("world", [2, 4])
def test_parts_sharded_over_ranks_recombine_to_the_single_gpu_pieces(world):
    import torch

    if torch.cuda.device_count() < world:
        pytest.skip(f"needs {world} GPUs")
    import torch.multiprocessing as mp

    mpctx = mp.get_context("spawn")
    q = mpctx.Queue()
    port = 28700 + (os.getpid() + 11 * world) % 1000
    procs = [mpctx.Process(target=_worker, args=(r, world, port, q)) for r in range(world)]
    for p in procs:
        p.start()
    res = [q.get(timeout=900) for _ in procs]
    for p in procs:
        p.join(timeout=120)
    assert sorted(res) == [(r, True) for r in range(world)]
