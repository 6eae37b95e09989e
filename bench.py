#!/usr/bin/env python
"""bench.py — chunk-proof polynomial-arithmetic wall time on B200 (BASELINE.json metric, configs[2]).

A "step" is ONE pass of the hot path over one CHUNK PROOF's worth of synthetic columns: the KZG commits (MSM) and
NTTs that halo2's create_proof issues for the three proofs `test-chunk-prove` generates on the degree-26 SRS
(/root/reference/Makefile:41, integration/tests/chunk_tests.rs:17-24, integration/src/prove.rs:37-39):

    inner   zkEVM super-circuit,  k = 20 (INNER_DEGREE, integration/src/mock.rs:9): several hundred columns
    layer1  wide compression,     k = 24 (integration/configs/layer1.config:3-9)
    layer2  thin compression,     k = 25 (integration/configs/layer2.config:3-9; 11 MSMs by release-v0.13.1/chunk.protocol)

per layer (SURVEY.md §8(a) a5/a7, §8(d).2-3):
    C columns   x [commit_lagrange = MSM 2^k -> lagrange_to_coeff = iNTT 2^k -> coeff_to_extended = coset NTT 2^(k+2)]
    M commits   of coefficient-form polynomials (4 quotient pieces + SHPLONK)       = MSM 2^k over g
    X           coeff_to_extended of fixed / permutation polynomials (layer2 only)  = coset NTT 2^(k+2)
    1           extended_to_coeff of the quotient                                  = inverse coset NTT 2^(k+2)
The layers run one after the other (each verifies the previous proof).  Column counts of the inner proof are the
survey's estimate ("several hundred"), stated in `config`.  The real trace cannot be proved here (no Rust toolchain, no
SRS files, host witness generation out of scope), so the layer is replayed on synthetic data of that shape.

`--k K` replays ONE layer of the layer-1 shape at degree K instead (size sweeps; K = 24 is BASELINE configs[1]).

JSON keys: see DESIGN.md "Measurement".  `value` = device-resident seconds per step (inputs in HBM), `e2e` = the same
step through the public session API with HOST (pinned) witness columns, H2D inside the timed region, commitments read
back.  With --gpus N (torchrun) every layer's independent jobs are fanned out over the ranks (strong scaling; the only
exchange is one all-gather of the 96 B commitments per layer).

--impl reference times the CPU restatement of the reference's Rayon path (oracle/, all host threads): every timed
iteration runs one operation of each kind of each layer AT FULL SIZE and the step is those times multiplied by the op
counts (`extrapolated_by_op_counts`); nothing is rescaled from smaller sizes, warm-up iterations never feed the value.
The default arm never touches oracle/ outside its `cpu_baseline` leg.

--dump-outputs DIR writes what the last timed step computed, for comparing two builds output for output (the inputs are seeded, so
they are the same on every run with the same arguments): `<layer>_commitments.npy`, every job's commitment of every layer as affine
(x, y) (identity = (0, 0)), and `<last layer>_coefficients.npy`, the coefficient vectors of the last layer's transform chains, which
stay in device memory after the step, at the rows of `<last layer>_coefficient_rows.npy` (a fixed, seeded sample).  Field elements
are canonical integers as eight little-endian 32-bit limbs in float64, which is exact.  Earlier layers' coefficient vectors are
overwritten by the later layers of the same step, and the extended (coset) evaluations go to a ring of buffers that the jobs reuse,
so neither is dumped.
"""
from __future__ import annotations

import argparse
import importlib
import json
import os
import subprocess
import sys
import threading
import time
from collections import namedtuple

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

MAC32_PER_MADD = 1280  # 10 modmul x 128 MAC32 (SURVEY.md §8(d))
Q_MOD = 0x30644E72E131A029B85045B68181585D97816A916871CA8D3C208C16D87CFD47  # BN254 base field
R_MOD = 0x30644E72E131A029B85045B68181585D2833E84879B9709143E1F593F0000001  # BN254 scalar field
DUMP_COEFF_BYTES = 32 << 20  # cap on the sampled coefficient rows of --dump-outputs (8 float64 limbs = 64 B per element)

# name, k, witness-like Lagrange columns, uniform Lagrange columns, coefficient-form commits, extra coset NTTs
Layer = namedtuple("Layer", "name k wit uni coeff extra")
# inner: estimate for the zkEVM super-circuit (SURVEY.md §8(a) a5 "several hundred"): ~400 advice / lookup-multiplicity
# columns (witness-like), ~100 permutation-z / lookup-phi / random columns (uniform), 4 quotient pieces + 2 SHPLONK commits
# layer1: 15 advice + 2 lookup advice (layer1.config) -> 19 witness-like + 9 z / phi / random, 4 + 3 coefficient commits
# layer2: chunk.protocol num_witness [1,1,3] -> 5 Lagrange commits; 4 quotient pieces + 2 SHPLONK commits = 11 MSMs;
#         12 coset NTTs in all (SURVEY.md §8(d).3): the 5 witness columns + the 7 fixed / permutation polynomials
CHUNK_LAYERS = (Layer("inner", 20, 416, 96, 6, 0), Layer("layer1", 24, 19, 9, 7, 0), Layer("layer2", 25, 3, 2, 6, 7))


def layers_for(args):
    if args.k:
        return (Layer(f"degree-{args.k} layer", args.k, 19, 9, 7, 0),)
    only = [x for x in getattr(args, "only", "").split(",") if x]
    return tuple(l._replace(k=max(2, l.k - args.shrink)) for l in CHUNK_LAYERS if not only or l.name in only)


def metric_name(args) -> str:
    if args.k:
        return f"chunk-proof wall-sec (degree-{args.k} layer poly-arith replay)"
    return "chunk-proof wall-sec (degree-26 SRS: k=20+24+25 replay)" + (f" [sizes shrunk by 2^{args.shrink}]" if args.shrink else "") + \
        (f" [only {args.only}]" if getattr(args, "only", "") else "")


def workload_desc(args) -> str:
    ls = layers_for(args)
    per = "; ".join(f"{l.name} k={l.k}: {l.wit + l.uni} x (MSM 2^{l.k} + iNTT 2^{l.k} + cosetNTT 2^{l.k + 2}) + {l.coeff} MSM 2^{l.k}"
                    + (f" + {l.extra} cosetNTT 2^{l.k + 2}" if l.extra else "") + f" + 1 icosetNTT 2^{l.k + 2}" for l in ls)
    head = "configs[1] inner-prove degree-%d layer shape replay" % args.k if args.k else \
        "configs[2] test-chunk-prove (degree-26 SRS) replay, three proofs in sequence"
    return f"{head}: {per}"


# relative job costs in ms, measured on one B200 (profiles/sweep_r01.jsonl and this round's batch figures); only the
# balance of the fan-out depends on them
def _cost(kind: str, dist: str, k: int) -> float:
    s = 2.0 ** (k - 24)
    if kind in ("lmsm", "msm"):
        return (9.6 if dist == "w" else 42.0) * s * (1.0 if k >= 22 else 0.9)
    if kind == "ntt":
        return 19.5 * s
    return 16.0 * s  # coset / icoset


def make_jobs(layer: Layer):
    """(kind, scalar distribution, relative cost) for every independent unit of one layer's proof."""
    # A column's commitment (MSM) and its transforms (iNTT + coset NTT) are independent, so they are separate jobs.
    k = layer.k
    jobs = [("lmsm", "w", _cost("lmsm", "w", k))] * layer.wit + [("lmsm", "u", _cost("lmsm", "u", k))] * layer.uni   # commit_lagrange
    jobs += [("ntt", "w", _cost("ntt", "w", k))] * layer.wit + [("ntt", "u", _cost("ntt", "u", k))] * layer.uni      # lagrange_to_coeff + coeff_to_extended
    jobs += [("msm", "u", _cost("msm", "u", k))] * layer.coeff + [("coset", "u", _cost("coset", "u", k))] * layer.extra
    jobs += [("icoset", "u", _cost("icoset", "u", k))]
    return jobs


def assign_jobs(jobs, world: int):
    """LPT greedy fan-out of the independent jobs over ranks."""
    order = sorted(range(len(jobs)), key=lambda i: -jobs[i][2])
    load = [0.0] * world
    out = [[] for _ in range(world)]
    for i in order:
        r = min(range(world), key=lambda x: load[x])
        out[r].append(jobs[i])
        load[r] += jobs[i][2]
    return out


def op_counts(layer: Layer):
    """operations of one layer by kind (the multipliers of the CPU arm's per-op times)"""
    return {"msm_w": layer.wit, "msm_u": layer.uni + layer.coeff, "intt": layer.wit + layer.uni,
            "coset": layer.wit + layer.uni + layer.extra + 1}  # the quotient's inverse coset NTT costs one coset NTT


def host_threads() -> int:
    """Threads the reference's Rayon pool would get: min(logical CPUs, affinity mask, cgroup CPU quota)."""
    n = os.cpu_count() or 1
    try:
        n = min(n, len(os.sched_getaffinity(0)))
    except Exception:
        pass
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            n = min(n, max(1, int(int(q) / int(per) + 0.5)))
    except Exception:
        pass
    return n


class ClockSampler:
    def __init__(self, device: int):
        self.device, self.rows, self.proc = device, [], None

    def start(self):
        q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
            "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.device), f"--query-gpu={q}", "--format=csv,noheader,nounits",
                                          "-lms", "200"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.proc:
            self.proc.terminate()
        sm = sorted(int(float(r[0])) for r in self.rows if r and r[0].replace(".", "").isdigit())
        mx = max([int(float(r[1])) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()] or [0])
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows if len(r) >= 7 for i in range(4) if r[3 + i].lower().startswith("active")})
        loaded = [x for x in sm if x > 0.5 * (mx or 1)] or sm
        return {"sm_mhz": loaded[len(loaded) // 2] if loaded else None, "sm_max_mhz": mx or None, "reasons": reasons,
                "samples": len(sm)}


def imad_peak():
    """INT32 multiply-pipe peaks (GMAC32/s): `measured` from the tracked, clock-stamped microbenchmark record
    IMAD_PEAK.json (written by tools/imad_peak.py on a B200), `nominal` = SMs x 32 IMAD.WIDE lanes/clk x max SM clock."""
    d = json.load(open(os.path.join(ROOT, "IMAD_PEAK.json")))
    return d["montgomery_product_gmac32"], d["nominal_imad_wide_gmac32"], d


# ====================================================================================================
# reference arm / cpu_baseline: the oracle's restatement of halo2_proofs' Rayon path on the host cores
# ====================================================================================================
_CPU_INPUTS = {}


def _cpu_inputs(k: int, threads: int):
    """bases / scalars / domain for the CPU legs, generated once per size (not part of any timed region)."""
    from oracle import oracle as O  # ORACLE: allowed here only (cpu_baseline / --impl reference)

    if k not in _CPU_INPUTS:
        n = 1 << k
        _CPU_INPUTS[k] = (O.fill_points_chain(n, 7, threads), O.fill_fr(n, 1, True), O.fill_fr(n, 2, False), O.EvaluationDomain(5, k))
    return _CPU_INPUTS[k]


def cpu_layer_sample(k: int, threads: int):
    """One operation of each kind at FULL size on `threads` host threads: witness-like MSM 2^k, uniform MSM 2^k,
    iNTT 2^k, coset NTT 2^(k+2).  Returns {op: seconds}."""
    from oracle import oracle as O  # ORACLE: allowed here only (cpu_baseline / --impl reference)

    bases, sw, su, dom = _cpu_inputs(k, threads)
    t = {}
    t0 = time.perf_counter(); O.best_multiexp(sw, bases, threads); t["msm_w"] = time.perf_counter() - t0
    t0 = time.perf_counter(); O.best_multiexp(su, bases, threads); t["msm_u"] = time.perf_counter() - t0
    t0 = time.perf_counter(); coeff = dom.lagrange_to_coeff(su, threads); t["intt"] = time.perf_counter() - t0
    t0 = time.perf_counter(); dom.coeff_to_extended(coeff, threads); t["coset"] = time.perf_counter() - t0
    return t


def cpu_parallelism(threads: int):
    """how many of the nominal host threads actually run in parallel (containers are often CPU-quota limited):
    one 2^14-point MSM chunk alone vs one such chunk per thread, all at once"""
    from oracle import oracle as O  # ORACLE: allowed here only (cpu_baseline / --impl reference)

    m = 1 << 14
    bases, su = O.fill_points_chain(m, 7, threads), O.fill_fr(m, 2, False)
    reps, rb = np.tile(su, (threads, 1)), np.tile(bases, (threads, 1))
    t1 = tT = 1e30
    for _ in range(2):
        t0 = time.perf_counter(); O.best_multiexp(su, bases, 1); t1 = min(t1, time.perf_counter() - t0)
        t0 = time.perf_counter(); O.best_multiexp(reps, rb, threads); tT = min(tT, time.perf_counter() - t0)
    out = {"effective_parallelism": round(threads * t1 / tT, 1) if tT > 0 else None, "affinity": len(os.sched_getaffinity(0))}
    for f in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        if os.path.exists(f):
            out["cgroup_cpu"] = open(f).read().strip()
            break
    return out


def cpu_step_sample(layers, threads: int, bounded_k: int = 0):
    """(step seconds, per-layer detail): every layer's four operations timed once at full size, times the op counts.
    bounded_k > 0 (the product arm's in-line `cpu_baseline`, which must stay a ~30 s sample): layers with k > bounded_k are not
    timed but SCALED from the largest timed layer by their size ratio -- MSM by 2^dk, transforms by 2^dk * k / k0 -- and are
    marked `scaled_from`; `--impl reference` never does this."""
    total, detail, timed = 0.0, {}, {}
    for l in layers:
        cnt = op_counts(l)
        if bounded_k and l.k > bounded_k and timed:
            k0 = max(timed)
            f = 2.0 ** (l.k - k0)
            t = {"msm_w": timed[k0]["msm_w"] * f, "msm_u": timed[k0]["msm_u"] * f, "intt": timed[k0]["intt"] * f * l.k / k0,
                 "coset": timed[k0]["coset"] * f * (l.k + 2) / (k0 + 2)}
            extra = {"scaled_from": k0}
        else:
            t = cpu_layer_sample(l.k, threads)
            timed[l.k] = t
            extra = {}
        sec = sum(cnt[o] * t[o] for o in cnt)
        detail[l.name] = {"k": l.k, "op_s": {o: round(v, 6) for o, v in t.items()}, "op_counts": cnt, "layer_s": sec, **extra}
        total += sec
    return total, detail


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    threads = host_threads()
    layers = layers_for(args)
    for l in layers:  # inputs (and the thread pool / page faults) outside every timed region
        _cpu_inputs(l.k, threads)
    small = tuple(l._replace(k=min(l.k, 12)) for l in layers)
    for _ in range(args.warmup):  # warm-up never feeds the value: code paths and the thread pool at a small size
        cpu_step_sample(small, threads)
    budget_s, t_start, vals, detail = 240.0, time.perf_counter(), [], None
    for i in range(args.steps):
        if vals and (time.perf_counter() - t_start) + sample_wall > budget_s:
            break  # the run stays within a few minutes: fewer full-size samples, never smaller ones
        t0 = time.perf_counter()
        v, detail = cpu_step_sample(layers, threads)
        sample_wall = time.perf_counter() - t0
        vals.append(v)
    v = sum(vals) / len(vals)
    par = cpu_parallelism(threads)
    sample = ("every timed sample: 1 witness-like MSM + 1 uniform MSM + 1 iNTT 2^k + 1 coset NTT 2^(k+2) per layer at FULL size "
              "(k = %s) on %d host threads; step = op times x op counts; value = mean of %d full-size samples (of %d requested steps); "
              "warm-up at 2^12, never in the value" % ("/".join(str(l.k) for l in layers), threads, len(vals), args.steps))
    line = {"impl": "reference", "metric": metric_name(args), "value": v, "unit": "s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": v * 1e3, "higher_is_better": False, "scaling": "strong", "vs_baseline": None,
            "dtype": "u64x4 (254-bit Montgomery integers on the CPU)", "data": "synthetic",
            "config": {"workload": workload_desc(args), "k": args.k or None, "layers": [l._asdict() for l in layers]},
            "extrapolated_by_op_counts": True, "full_size_samples": len(vals), "sample_values_s": vals,
            "timed_cpu_seconds_per_sample": sample_wall,
            "cpu_baseline": {"value": v, "unit": "s", "cores": threads, "kind": "port", "sample": sample, "detail": detail,
                             "parallelism": par},
            "e2e": {"value": v, "unit": "s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))
    return 0


# ====================================================================================================
# product arm
# ====================================================================================================
def _limbs32(values) -> np.ndarray:
    """integers below 2^256 as rows of eight little-endian 32-bit limbs in float64 (exact)"""
    return np.array([[(v >> (32 * i)) & 0xFFFFFFFF for i in range(8)] for v in values], dtype=np.float64).reshape(-1, 8)


def dump_outputs(out_dir, plans, pool_coeff, suffix=""):
    """--dump-outputs: the commitments of every layer and a seeded sample of the last layer's coefficient vectors (see the module
    docstring); called right after the timed steps, while the buffers still hold the last step's results."""
    import torch

    os.makedirs(out_dir, exist_ok=True)
    mont = lambda limbs, mod: int.from_bytes(limbs.tobytes(), "little") * pow(1 << 256, -1, mod) % mod
    for pl in plans:
        xy = []
        for c in pl.get("commits", np.zeros((0, 12), np.uint64)):  # Jacobian (X, Y, Z), Montgomery form
            x, y, z = (mont(c[4 * i:4 * i + 4], Q_MOD) for i in range(3))
            zi = pow(z, -1, Q_MOD) if z else 0
            xy += [x * zi * zi % Q_MOD, y * zi * zi * zi % Q_MOD]
        np.save(os.path.join(out_dir, f"{pl['layer'].name}_commitments{suffix}.npy"), _limbs32(xy).reshape(-1, 2, 8))
    last = plans[-1]
    n, chains = last["n"], len(last["nt"])
    if chains:
        rows = np.sort(np.random.default_rng(0).choice(n, size=min(n, 1 << 16, DUMP_COEFF_BYTES // (64 * chains)), replace=False))
        coeff = pool_coeff[:chains * n * 4].view(chains, n, 4)[:, torch.from_numpy(rows).to(pool_coeff.device)]
        coeff = coeff.cpu().numpy().view(np.uint64).reshape(-1, 4)
        name = last["layer"].name
        np.save(os.path.join(out_dir, f"{name}_coefficients{suffix}.npy"), _limbs32(mont(e, R_MOD) for e in coeff).reshape(chains, -1, 8))
        np.save(os.path.join(out_dir, f"{name}_coefficient_rows{suffix}.npy"), rows.astype(np.float64))


def run_b200(args):
    import torch

    zk = importlib.import_module("scroll-prover_b200")
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the product has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    dist = None
    if world > 1:
        import torch.distributed as dist_mod

        dist = dist_mod
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    dev = torch.device("cuda", local)
    layers = layers_for(args)
    comp = torch.cuda.Stream()  # a non-default stream, so that our CUDA events bracket the library's launches
    torch.cuda.set_stream(comp)
    ctx = zk.Context(local)
    ctx.set_stream(comp.cuda_stream)
    if dist:
        ctx.comm_init_torch(dist)  # the context owns the NCCL communicator (sharded entry points)

    # ---- synthetic inputs (device-generated)
    gen = torch.Generator(device=dev).manual_seed(1234 + rank)

    def rand_limbs(cnt):
        t = torch.randint(-(2 ** 63), 2 ** 63 - 1, (cnt, 4), dtype=torch.int64, device=dev, generator=gen)
        t[:, 3] &= 0x0FFFFFFFFFFFFFFF  # < 2^252 < r: valid Montgomery limbs of a uniform-ish element
        return t

    def witness_like(cnt):
        sel = torch.rand(cnt, device=dev, generator=gen)
        small = torch.randint(0, 1 << 16, (cnt,), dtype=torch.int64, device=dev, generator=gen)
        raw = torch.zeros((cnt, 4), dtype=torch.int64, device=dev)
        raw[:, 0] = torch.where((sel >= 0.6) & (sel < 0.9), small, torch.zeros_like(small))
        r2 = zk.fr_from_int(1 << 256)  # Montgomery form of R: x * R2 * R^-1 = x*R -> to_mont
        torch.cuda.synchronize()
        mont = ctx.poly_scale(raw, r2)
        uni = rand_limbs(cnt)
        m = (sel >= 0.9).unsqueeze(1)
        torch.cuda.synchronize()
        return torch.where(m, uni, mont).contiguous()

    # ---- SRS: the degree-26 SRS downsized per layer (ParamsKZG::downsize): `g` of a smaller degree is a prefix of the
    # largest one, so ONE handle of the largest k serves every layer's coefficient-form commits; g_lagrange is per degree.
    kmax = max(l.k for l in layers)
    g = torch.empty((1 << kmax, 8), dtype=torch.int64, device=dev)
    torch.cuda.synchronize()
    ctx.g1_generator_mul_batch(rand_limbs(1 << kmax), out=g)
    srs_g = ctx.srs_register(g, zk.SRS_G)
    srs_gl = {}
    for l in layers:
        if l.k not in srs_gl:
            ctx.g1_generator_mul_batch(rand_limbs(1 << l.k), out=g[: 1 << l.k])
            srs_gl[l.k] = ctx.srs_register(g[: 1 << l.k], zk.SRS_G_LAGRANGE)
    srs_g_small = {}  # a small layer commits over its own short `g` handle (tables sized for it) rather than a 2^25 prefix
    for l in layers:
        if l.k + 4 < kmax and l.k not in srs_g_small:
            ctx.g1_generator_mul_batch(rand_limbs(1 << l.k), out=g[: 1 << l.k])
            srs_g_small[l.k] = ctx.srs_register(g[: 1 << l.k], zk.SRS_G)
    del g
    torch.cuda.empty_cache()

    # ---- per layer: this rank's jobs, inputs, output pools
    RING_IN = 64   # distinct input columns per (layer, distribution) when a layer has more columns than that
    plans = []
    pool_coeff_bytes = pool_ext_bytes = 0
    for l in layers:
        n, ek = 1 << l.k, l.k + 2
        my = assign_jobs(make_jobs(l), world)[rank]
        lm = [j for j in my if j[0] == "lmsm"]
        nt = [j for j in my if j[0] == "ntt"]
        ms = [j for j in my if j[0] == "msm"]
        cs = [j for j in my if j[0] == "coset"]
        ic = [j for j in my if j[0] == "icoset"]
        need = {"w": max(sum(1 for j in lm if j[1] == "w"), sum(1 for j in nt if j[1] == "w")),
                "u": max(sum(1 for j in lm if j[1] == "u"), sum(1 for j in nt if j[1] == "u"))}
        cols = {d: [(witness_like if d == "w" else rand_limbs)(n) for _ in range(min(need[d], RING_IN))] for d in ("w", "u")}
        coeff_in = [rand_limbs(n) for _ in range(min(2, len(ms) + len(cs)))]   # device-produced polynomials (h pieces, openings, fixed)
        hext = rand_limbs(1 << ek) if ic else None                              # device-produced quotient evaluations
        dom = zk.EvaluationDomain(ctx, 5, l.k)
        n_coeff_out = len(nt)
        pool_coeff_bytes = max(pool_coeff_bytes, n_coeff_out * n * 32)
        plans.append({"layer": l, "n": n, "ek": ek, "lm": lm, "nt": nt, "ms": ms, "cs": cs, "ic": ic, "cols": cols, "coeff_in": coeff_in,
                      "hext": hext, "dom": dom, "my": my})
    # output pools shared by the layers (they run one after the other): every transform chain keeps its OWN coefficient
    # vector (the openings need them), the extended cosets go to a ring (evaluate_h consumes them group by group)
    free_b, _ = torch.cuda.mem_get_info()
    RING_EXT_BYTES = int(min(16 << 30, max(1 << 20, 0.25 * free_b)))
    pool_coeff = torch.empty(max(pool_coeff_bytes, 32) // 8, dtype=torch.int64, device=dev)
    pool_ext = torch.empty(RING_EXT_BYTES // 8, dtype=torch.int64, device=dev)

    def job_lists(pl, src_cols):
        """this rank's share of one layer as ONE b200zk_run_column_jobs list: a column whose commitment and transforms both
        landed here is one mode-2 job (uploaded once in the e2e arm)"""
        l, n, ek = pl["layer"], pl["n"], pl["ek"]
        gl = srs_gl[l.k]
        gsrs = srs_g_small.get(l.k, srs_g)
        ext_elems = (1 << ek) * 4
        ring = max(1, pool_ext.numel() // ext_elems)
        state = {"c": 0, "e": 0}

        def coeff_out():
            o = pool_coeff[state["c"] * n * 4:(state["c"] + 1) * n * 4]
            state["c"] += 1
            return o

        def ext_out():
            o = pool_ext[(state["e"] % ring) * ext_elems:((state["e"] % ring) + 1) * ext_elems]
            state["e"] += 1
            return o

        jl = []
        for d in ("w", "u"):
            lm = [j for j in pl["lm"] if j[1] == d]
            nt = [j for j in pl["nt"] if j[1] == d]
            both = min(len(lm), len(nt))
            cs_ = src_cols[d]
            pick = lambda i: cs_[i % len(cs_)]
            jl += [(pick(i), gl, 2, coeff_out(), ext_out()) for i in range(both)]
            jl += [(pick(i), gl, 0, None, None) for i in range(both, len(lm))]
            jl += [(pick(i), None, 3, coeff_out(), ext_out()) for i in range(both, len(nt))]
        ci = pl["coeff_in"]
        jl += [(ci[i % len(ci)], gsrs, 0, None, None) for i in range(len(pl["ms"]))]
        jl += [(ci[i % len(ci)], None, 5, None, ext_out()) for i in range(len(pl["cs"]))]
        if pl["ic"]:
            jl.append((pl["hext"], None, 4, pool_ext[:ext_elems], None))
        return jl, ring

    for pl in plans:
        pl["resident"], pl["ring"] = job_lists(pl, pl["cols"])
    # ---- e2e: the witness columns (every Lagrange-form column) start in pinned HOST memory; polynomials the prover
    # produces on the device (quotient pieces, opening quotients, the quotient's evaluations) and the proving key's
    # fixed / permutation polynomials are device-resident in a session and stay so
    h2d_bytes = 0
    for pl in plans:
        host = {d: [c.cpu().pin_memory() for c in pl["cols"][d]] for d in ("w", "u")}
        pl["host_jobs"], _ = job_lists(pl, host)
        pl["h2d_bytes"] = sum(pl["n"] * 32 for j in pl["host_jobs"] if j[2] in (0, 1, 2, 3) and not j[0].is_cuda)
        h2d_bytes += pl["h2d_bytes"]
    total_jobs = sum(len(pl["resident"]) for pl in plans)
    d2h_bytes = total_jobs * 96
    commits = np.zeros((max(len(pl["resident"]) for pl in plans) + 1, 12), np.uint64)
    gather_cap = max(len(pl["resident"]) for pl in plans) + 8
    if dist:
        cap_t = torch.tensor([gather_cap], device=dev)
        dist.all_reduce(cap_t, op=dist.ReduceOp.MAX)
        gather_cap = int(cap_t.item())

    def run_layer(pl, key):
        jl = pl[key]
        if jl:
            pl["commits"] = zk.run_column_jobs(ctx, jl, pl["layer"].k, omega_inv=pl["dom"].omega_inv,
                                               extended_omega=pl["dom"].extended_omega,
                                               extended_omega_inv=pl["dom"].extended_omega_inv, extended_k=pl["ek"])
            commits[: len(jl)] = pl["commits"]
        torch.cuda.current_stream().synchronize()
        if dist:  # the next proof hashes this proof's commitments: one tiny all-gather per layer, the only exchange
            t = torch.zeros((world, gather_cap, 12), dtype=torch.int64, device=dev)
            mine = torch.zeros((gather_cap, 12), dtype=torch.int64, device=dev)
            mine[: len(jl)] = torch.from_numpy(commits[: len(jl)].view(np.int64)).to(dev)
            dist.all_gather_into_tensor(t.view(-1), mine.view(-1))

    layer_ms = {"resident": [[] for _ in plans], "host_jobs": [[] for _ in plans]}

    def step(key, record=False):
        evs = [torch.cuda.Event(enable_timing=True) for _ in range(len(plans) + 1)] if record else None
        if record:
            evs[0].record(comp)
        for i, pl in enumerate(plans):
            run_layer(pl, key)
            if record:
                evs[i + 1].record(comp)
        return evs

    def barrier():
        torch.cuda.synchronize()
        if dist:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(key, steps, warmup, profile=False):
        for _ in range(warmup):
            step(key)
        barrier()
        if profile:
            ctx.profile_enable(True)
            ctx.profile_reset()
            ctx.msm_total_adds(reset=True)
        l0 = ctx.launch_count()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        e0.record(comp)
        all_evs = [step(key, record=True) for _ in range(steps)]
        e1.record(comp)
        barrier()
        wall = time.perf_counter() - t0
        ms = e0.elapsed_time(e1)
        for evs in all_evs:
            for i in range(len(plans)):
                layer_ms[key][i].append(evs[i].elapsed_time(evs[i + 1]))
        prof = ctx.profile_read() if profile else None
        if profile:
            prof["_actual_adds"] = ctx.msm_total_adds()
            ctx.profile_enable(False)
        launches = ctx.launch_count() - l0
        tt = torch.tensor([ms], dtype=torch.float64, device=dev)
        if dist:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        return tt.item() / 1e3 / steps, wall / steps, prof, launches

    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.start()
    sec, wall, _, launches = timed("resident", args.steps, args.warmup, profile=False)
    clocks = sampler.stop() if sampler else None
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, plans, pool_coeff, f"_rank{rank}" if world > 1 else "")
    per_layer_value = [sum(v) / len(v) / 1e3 for v in layer_ms["resident"]]
    # per-kernel durations (roofline, kernel_ms_per_step) come from a separate profiled pass of the SAME step with the
    # two-stream overlap switched off: while kernels of two streams share the SMs their individual durations say nothing
    ctx.set_overlap(False)
    prof_steps = 1
    layer_ms["resident"] = [[] for _ in plans]
    _, _, prof, _ = timed("resident", prof_steps, 0, profile=True)
    ctx.set_overlap(True)
    if args.skip_e2e:
        e2e_sec, per_layer_e2e = None, None
    else:
        e2e_sec, e2e_wall, _, _ = timed("host_jobs", max(1, min(args.steps, 3)), 1)
        per_layer_e2e = [sum(v) / len(v) / 1e3 for v in layer_ms["host_jobs"]]

    # ---- units processed (whole job) for the throughput figures
    bf = lambda lg: (1 << lg) // 2 * lg
    total_bf = sum((l.wit + l.uni) * (bf(l.k) + bf(l.k + 2)) + (l.extra + 1) * bf(l.k + 2) for l in layers)
    total_points = sum((l.wit + l.uni + l.coeff) * (1 << l.k) for l in layers)

    if rank == 0:
        peak_meas, peak_nom, peak_rec = imad_peak()
        actual_adds = prof.pop("_actual_adds")
        msm_ms = sum(prof[c]["ms"] for c in prof if c.startswith("msm_"))
        acc_ms = prof["msm_accumulate"]["ms"]
        ntt_ms = prof["ntt_pass"]["ms"]
        my_bf = my_ntt_bytes = my_points = 0
        for pl in plans:
            l, n, ek = pl["layer"], pl["n"], pl["ek"]
            passes = lambda lg: (lg + 7) // 8  # this build: digits of <= 8 bits
            for j in pl["my"]:
                if j[0] == "ntt":
                    my_bf += bf(l.k) + bf(ek)
                    my_ntt_bytes += 64 * n * passes(l.k) + 64 * (1 << ek) * passes(ek)  # algorithmic: 64 B/element/pass
                elif j[0] in ("coset", "icoset"):
                    my_bf += bf(ek)
                    my_ntt_bytes += 64 * (1 << ek) * passes(ek)
                else:
                    my_points += n
        # algorithmic MAC32 of the accumulate launches = bucket additions actually performed (non-zero signed digits;
        # witness-like columns skip most of the N*W upper bound) x 1280 MAC32 per mixed add (SURVEY.md §8(d))
        acc_achieved = (actual_adds * MAC32_PER_MADD) / (acc_ms * 1e-3) / 1e9 if acc_ms else None
        traffic, traffic_note = None, None
        try:  # DRAM bytes of one msm_accumulate launch from the committed `ncu --set full` capture (uniform 2^24 MSM)
            ncu = json.load(open(os.path.join(ROOT, "profiles", "ncu_r01_v6_summary.json")))
            for e in ncu["kernels"]:
                if e["kernel"].startswith("msm_accumulate"):
                    rd, wr = float(e["dram__bytes_read.sum"].split()[0]), float(e["dram__bytes_write.sum"].split()[0])
                    traffic = (rd + wr) * 1e9
                    traffic_note = ("dram__bytes_read+write of ONE msm_accumulate launch (MSM 2^24, uniform scalars, 201 M adds) "
                                    "from profiles/ncu_r01_v6_summary.json; algorithmic bytes of that launch = 201e6 x 68 B = 13.7e9")
                    break
        except Exception:
            pass
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))) if os.path.exists(os.path.join(ROOT, "MEASURED_PEAKS.json")) else {}
        hbm_peak = peaks.get("hbm_gbs", 6650.0)
        ntt_gbs = my_ntt_bytes * prof_steps / (ntt_ms * 1e-3) / 1e9 if ntt_ms else None
        cpu = None
        if world == 1 and not args.no_cpu_baseline:
            threads = host_threads()
            cs, detail = cpu_step_sample(layers, threads, bounded_k=24)
            scaled = [n for n, d in detail.items() if "scaled_from" in d]
            cpu = {"value": cs, "unit": "s", "cores": threads, "kind": "port", "extrapolated_by_op_counts": True, "scaled_layers": scaled,
                   "sample": "bounded sample (~30 s of CPU work): per layer with k <= 24, 1 witness-like MSM + 1 uniform MSM + 1 iNTT 2^k + "
                             "1 coset NTT 2^(k+2) at full size on all host threads; step = op times x op counts; layers above 2^24 ("
                             + ", ".join(scaled) + ") are scaled from the 2^24 times by their size ratio -- the full-size figure for "
                             "every layer is what `--impl reference` measures", "detail": detail}
        st = ctx.msm_last_stats()
        line = {
            "metric": metric_name(args), "value": sec, "unit": "s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": sec * 1e3, "higher_is_better": False, "scaling": "strong", "vs_baseline": None,
            "dtype": "u32x8 (254-bit Montgomery integers)", "data": "synthetic",
            "config": {"workload": workload_desc(args), "k": args.k or None, "layers": [l._asdict() for l in layers],
                       "parallelism": f"per-layer job fan-out x{world} (no data-path collective; one 96 B/commitment all-gather per layer)",
                       "buffers": {"distinct_input_columns_per_layer_and_distribution": RING_IN,
                                   "coefficient_outputs": "one per transform chain (kept)",
                                   "extended_outputs_ring": [pl["ring"] for pl in plans]},
                       "l2": "inputs (>= 32 MiB per column, hundreds of distinct columns) exceed the 126 MB L2; no flush needed"},
            "layers_s": {pl["layer"].name: v for pl, v in zip(plans, per_layer_value)},
            "layers_e2e_s": {pl["layer"].name: v for pl, v in zip(plans, per_layer_e2e)} if per_layer_e2e else None,
            "msm_points_per_s_in_kernels_rank0": my_points * prof_steps / (msm_ms * 1e-3) if msm_ms else None,
            "ntt_butterflies_per_s": (my_bf * prof_steps) / (ntt_ms * 1e-3) if ntt_ms else None,
            "msm_actual_bucket_adds_per_step_rank0": actual_adds / prof_steps,
            "msm_g1_adds_per_s": actual_adds / (msm_ms * 1e-3) if msm_ms else None,
            "job_msm_points_per_s": total_points / sec, "job_ntt_butterflies_per_s": total_bf / sec,
            "roofline": {"bound": "int32-imad", "kernel": "msm_accumulate", "achieved": acc_achieved,
                         "peak": peak_meas, "peak_nominal": peak_nom, "unit": "GMAC32/s",
                         "frac": acc_achieved / peak_meas if acc_achieved else None,
                         "frac_of_nominal": acc_achieved / peak_nom if acc_achieved else None,
                         "peak_source": "IMAD_PEAK.json (tracked; Montgomery-product microbenchmark with its clock record; "
                                        "MEASURED_PEAKS.json has no INT32 figure): " + peak_rec.get("source", ""),
                         "traffic": traffic, "traffic_note": traffic_note,
                         "hbm": {"kernel": "ntt_pass", "achieved": ntt_gbs, "peak": hbm_peak, "unit": "GB/s",
                                 "frac": ntt_gbs / hbm_peak if ntt_gbs else None, "peak_source": "MEASURED_PEAKS.json hbm_gbs"}},
            "kernel_ms_per_step_rank0": {c: prof[c]["ms"] / prof_steps for c in prof if prof[c]["count"]},
            "kernel_timing_note": "per-kernel CUDA-event durations and the roofline come from one extra profiled pass of the same "
                                  "step with the two-stream overlap off; `value` is measured with the overlap on and profiling off",
            "cpu_baseline": cpu,
            "e2e": {"value": e2e_sec, "unit": "s", "h2d_bytes_per_step": h2d_bytes, "d2h_bytes_per_step": d2h_bytes,
                    "api": "ONE C-ABI call per proof (layer) with pinned HOST witness columns: b200zk_run_column_jobs (mode 2 per "
                           "column, mode 0 coefficient commits, mode 5 / 4 for device-produced polynomials which stay resident); H2D "
                           "double-buffered on the library's copy stream, commitments read back; rank 0 bytes"},
            "gpu_launches": launches, "clocks": clocks, "wall_s_per_step": wall,
            "msm_last_window": {"c": st["window_bits"], "W": st["n_windows"]},
        }
        print(json.dumps(line))
    if dist:
        dist.barrier()
        dist.destroy_process_group()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=2)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--k", type=int, default=0, help="replay ONE layer of the layer-1 shape at this degree (sweeps; 24 = configs[1]); "
                                                     "default 0 = the chunk proof of configs[2]: inner k=20 + layer1 k=24 + layer2 k=25")
    ap.add_argument("--shrink", type=int, default=0, help="subtract from every layer's k (contract tests on small machines)")
    ap.add_argument("--only", default="", help="profiling: restrict the chunk step to these layers, e.g. inner or layer1,layer2")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--skip-e2e", action="store_true", help="profiling runs only (ncu): device-resident arm only")
    ap.add_argument("--dump-outputs", metavar="DIR", default="", help="write the last timed step's outputs to DIR/<name>.npy")
    args = ap.parse_args()
    if args.impl == "reference":
        return run_reference(args)
    return run_b200(args)


if __name__ == "__main__":
    sys.exit(main())
