"""The quotient-by-parts figures quoted in DESIGN.md are the ones in the committed measurement files."""
import json
import os

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _rows(name):
    return [json.loads(l) for l in open(os.path.join(ROOT, "profiles", name)) if l.startswith("{")]


def _median(vals):
    vals = sorted(vals)
    return vals[len(vals) // 2]


def test_quotient_parts_timings_quoted_in_design():
    design = open(os.path.join(ROOT, "DESIGN.md")).read()
    rows = _rows("quotient_parts_r03.jsonl")
    assert {r["gpu"] for r in rows} == {"NVIDIA B200"} and "1000 W" in design and {r["power_limit"] for r in rows} == {"1000.00 W"}
    for k in (20, 24, 25):
        for path in ("full", "parts"):
            sel = [r for r in rows if r["k"] == k and r["path"] == path]
            assert len(sel) == 3 and all(r["device_bytes_from_shapes"] == r["device_bytes_mem_get_info"] for r in sel)
            for key in ("total_ms", "transforms_ms", "graph_ms", "recombination_ms"):
                assert f"{_median(r[key] for r in sel):.2f}" in design, (k, path, key)


def test_bench_before_and_after_quoted_in_design():
    design = open(os.path.join(ROOT, "DESIGN.md")).read()
    ab = _rows("bench_r03_parts_ab.jsonl")
    assert [a["arm"] for a in ab] == ["parent", "quotient-parts", "parent", "quotient-parts"]
    for a in ab:
        assert f"{a['bench']['value']:.3f}" in design
        assert f"{a['bench']['kernel_ms_per_step_rank0']['ntt_pass']:.1f}" in design
