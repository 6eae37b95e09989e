"""The quotient step (coefficient-form columns -> evaluate_h -> divide by X^n - 1 -> n * J coefficients) on full extended
cosets and part by part, alternately in one process, with per-phase device time and the device bytes each path holds.

usage: quotient_parts_time.py [out.jsonl]     (default profiles/quotient_parts_r03.jsonl; needs a CUDA device)

Sizes: k = 20 with 64 advice and 16 fixed columns; k = 24 and k = 25 with 8 advice and 2 fixed columns (at k = 25 a full coset
is 4 GiB per column); J = 4 throughout, the 16-gate program of tools/quotient_time.py.  Phases: transforms (coeff_to_extended /
coeff_to_extended_parts of every column), graph (the program over the extended domain / over each part), recombination
(the 1/(X^n - 1) column multiply + extended_to_coeff / extended_parts_to_coeff).  Every column is larger than the L2 at these
sizes (32 MiB at k = 20), so the timed passes read HBM.
"""
import importlib
import json
import os
import subprocess
import sys

import numpy as np
import torch

_ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, _ROOT)
sys.path.insert(0, os.path.join(_ROOT, "tools"))
sys.path.insert(0, os.path.join(_ROOT, "tests"))
zk = importlib.import_module("scroll-prover_b200")
from quick_time import rand_fr  # noqa: E402
from quotient_programs import R_MOD, ZETA, omega_of  # noqa: E402
from quotient_time import gate_program  # noqa: E402

SIZES = [(20, 64, 16), (24, 8, 2), (25, 8, 2)]
REPS = 3


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,clocks.sm,clocks.max.sm,power.limit", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()[0]
    name, sm, sm_max, power = [x.strip() for x in q.split(",")]
    return {"gpu": name, "sm_clock": sm, "sm_clock_max": sm_max, "power_limit": power}


class Phases:
    """device time per phase: CUDA events on the current stream around each phase, summed after one synchronise"""

    def __init__(self):
        self.spans = []

    def span(self, name):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        outer = self

        class _S:
            def __enter__(self):
                e0.record()

            def __exit__(self, *a):
                e1.record()
                outer.spans.append((name, e0, e1))

        return _S()

    def totals(self):
        torch.cuda.synchronize()
        out = {}
        for name, e0, e1 in self.spans:
            out[name] = out.get(name, 0.0) + e0.elapsed_time(e1)
        return out


def used_bytes():
    free, total = torch.cuda.mem_get_info()
    return total - free


def run_full(ctx, dom, graph, fixed_c, advice_c, y, t_col):
    k, ek, J, n = dom.k, dom.extended_k, dom.n_parts, dom.n
    P = Phases()
    base = used_bytes()
    with P.span("transforms"):
        fixed = [dom.coeff_to_extended(c) for c in fixed_c]
        advice = [dom.coeff_to_extended(c) for c in advice_c]
    h = torch.zeros((J * n, 4), dtype=torch.int64, device="cuda")
    with P.span("graph"):
        graph.evaluate(h, ek, J, fixed=fixed, advice=advice, y=y)
    with P.span("recombination"):
        ctx.poly_mul(h, t_col, out=h)
        out = dom.extended_to_coeff(h)
    torch.cuda.synchronize()
    held = used_bytes() - base
    res = P.totals()
    del fixed, advice, h, out
    return res, held


def run_parts(ctx, dom, graph, fixed_c, advice_c, y):
    k, ek, J, n = dom.k, dom.extended_k, dom.n_parts, dom.n
    P = Phases()
    base = used_bytes()
    fixed = [torch.empty_like(c) for c in fixed_c]
    advice = [torch.empty_like(c) for c in advice_c]
    parts = torch.zeros((J * n, 4), dtype=torch.int64, device="cuda")
    for r in range(J):
        with P.span("transforms"):
            dom.coeff_to_extended_parts(fixed_c + advice_c, r, fixed + advice)
        with P.span("graph"):
            graph.evaluate_part(parts[r * n:(r + 1) * n], k, ek, r, fixed=fixed, advice=advice, y=y)
    with P.span("recombination"):
        out = dom.extended_parts_to_coeff(parts, True)
    torch.cuda.synchronize()
    held = used_bytes() - base
    res = P.totals()
    del fixed, advice, parts, out
    return res, held


def main():
    path = sys.argv[1] if len(sys.argv) > 1 else os.path.join(_ROOT, "profiles", "quotient_parts_r03.jsonl")
    ctx = zk.Context(0)
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    ctx.set_stream(stream.cuda_stream)
    info = card()
    lines = []
    for k, n_advice, n_fixed in SIZES:
        dom = zk.EvaluationDomain(ctx, 5, k)
        J, n, ek = dom.n_parts, dom.n, dom.extended_k
        advice_c = [rand_fr(n, 100 + i) for i in range(n_advice)]
        fixed_c = [rand_fr(n, 200 + i) for i in range(n_fixed)]
        graph = ctx.graph(gate_program(16, n_advice), [zk.fr_from_int(1)], [0, 1, 2, 3])
        y = zk.fr_from_int(0x1234567)
        w_ext, zn = omega_of(ek), pow(ZETA, n, R_MOD)
        t_inv = [zk.fr_from_int(pow(zn * pow(w_ext, n * t, R_MOD) - 1, -1, R_MOD)) for t in range(J)]
        t_col = torch.from_numpy(np.tile(np.stack(t_inv), (n, 1)).view(np.int64)).cuda()
        cols = n_advice + n_fixed
        shapes = {"full": 32 * n * (cols * J + J), "parts": 32 * n * (cols + J)}  # beyond the resident coefficient columns
        torch.cuda.synchronize()
        # warm-up of both paths (module loads, twiddle tables, allocator), then alternate
        run_full(ctx, dom, graph, fixed_c, advice_c, y, t_col)
        run_parts(ctx, dom, graph, fixed_c, advice_c, y)
        for rep in range(REPS):
            for path_name in ("full", "parts"):
                torch.cuda.empty_cache()
                torch.cuda.synchronize()
                if path_name == "full":
                    ph, held = run_full(ctx, dom, graph, fixed_c, advice_c, y, t_col)
                else:
                    ph, held = run_parts(ctx, dom, graph, fixed_c, advice_c, y)
                rec = {"path": path_name, "k": k, "extended_k": ek, "J": J, "advice": n_advice, "fixed": n_fixed, "rep": rep,
                       "total_ms": sum(ph.values()), **{f"{p}_ms": v for p, v in ph.items()},
                       "device_bytes_from_shapes": shapes[path_name], "device_bytes_mem_get_info": held, **info}
                print(json.dumps(rec), flush=True)
                lines.append(rec)
        graph.release()
        del advice_c, fixed_c, t_col
        torch.cuda.empty_cache()
    with open(path, "w") as f:
        for rec in lines:
            f.write(json.dumps(rec) + "\n")
    ctx.close()


if __name__ == "__main__":
    main()
