"""Where the map step's time goes between the two field kernels: per-kernel times and the gap between each pair of
consecutive kernels of one FusedMapper.step at the bench shape (4096 rays x 43 samples), from torch.profiler with CUDA
activities, the 256 MB L2 flush between steps as in bench.py.

    python scripts/prof_glue.py --out DIR [--steps 20] [--warmup 5] [--pdl on|off] [--tag NAME]

Writes DIR/glue_<tag>.json (the card and its power limit, read in the same run, are part of it) and the raw trace
DIR/glue_<tag>.pt.trace.json.  Kernel times are medians over the profiled steps.  With programmatic dependent launch a
kernel's interval can start before its predecessor ends (its CTAs are resident and wait): gaps are then negative and a
kernel's time includes its wait, so the step span (first kernel start to last kernel end) is the number to compare.
"glue_us" is that span minus the two field kernels (field_fwd_tc3, field_bwd_tc2)."""
import argparse
import json
import os
import re
import statistics
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def short_name(name):
    n = re.sub(r"^void ", "", name)
    n = n.split("(")[0]
    if "FillFunctor" in name:
        return "torch_fill"
    if "distribution" in name or "uniform" in name:
        return "torch_uniform"
    return re.sub(r"<.*", "", n)


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=60).stdout.strip()
    except Exception as e:                                       # (the numbers are still valid; the record says why it is missing)
        out = "nvidia-smi unavailable: %s" % e
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--pdl", choices=("on", "off"), default=None, help="default: the library's setting")
    ap.add_argument("--tag", default=None)
    a = ap.parse_args()
    tag = a.tag or ("pdl_" + (a.pdl or "default"))
    os.makedirs(a.out, exist_ok=True)

    import bench
    import helpers as H
    from mipsfusion_b200 import _lib as L
    from mipsfusion_b200.mapper import FusedMapper
    assert torch.cuda.is_available(), "prof_glue.py measures on the GPU"
    if a.pdl:
        L.call("mf_set_pdl", 1 if a.pdl == "on" else 0)
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    cfg, of = bench.build_model()
    model = H.cuda_model(cfg, H.state_of(of))
    rays_o, rays_d, rgb, d, _ = bench.make_inputs(0)
    dv = torch.cat([rays_o, rays_d, rgb, d], -1).contiguous().to(dev)
    ro, rd, tc, td = dv[:, 0:3].contiguous(), dv[:, 3:6].contiguous(), dv[:, 6:9].contiguous(), dv[:, 9].contiguous()
    mapper = FusedMapper(model)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    for _ in range(a.warmup):
        flush.zero_()
        mapper.step(ro, rd, tc, td)
    torch.cuda.synchronize()

    trace = os.path.join(a.out, "glue_%s.pt.trace.json" % tag)
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        for _ in range(a.steps):
            flush.zero_()
            mapper.step(ro, rd, tc, td)
        torch.cuda.synchronize()
    prof.export_chrome_trace(trace)

    ev = json.load(open(trace))["traceEvents"]
    ks = sorted(((float(e["ts"]), float(e["dur"]), short_name(e["name"])) for e in ev if e.get("cat") == "kernel"), key=lambda x: x[0])
    # split into steps at the flush kernels; each step = the kernels after one flush
    steps, cur = [], None
    for k in ks:
        if k[2] == "torch_fill" and k[1] > 20.0:               # the 256 MB flush (other fills are tiny)
            if cur:
                steps.append(cur)
            cur = []
        elif cur is not None:
            cur.append(k)
    if cur:
        steps.append(cur)
    seqs = {tuple(k[2] for k in s) for s in steps}
    assert len(seqs) == 1, "steps launched different kernel sequences: %s" % seqs
    names = list(next(iter(seqs)))
    med = lambda xs: statistics.median(xs)
    kern = [{"kernel": n, "us": round(med([s[i][1] for s in steps]), 2)} for i, n in enumerate(names)]
    gaps = [{"after": names[i], "before": names[i + 1],
             "us": round(med([s[i + 1][0] - (s[i][0] + s[i][1]) for s in steps]), 2)} for i in range(len(names) - 1)]
    spans = [s[-1][0] + s[-1][1] - s[0][0] for s in steps]
    field = [i for i, n in enumerate(names) if n in ("field_fwd_tc3_kernel", "field_bwd_tc2_kernel")]
    glue = [sp - sum(s[i][1] for i in field) for sp, s in zip(spans, steps)]
    res = {"gpu": gpu_info(), "pdl": a.pdl, "steps_profiled": len(steps), "shape": "R=4096 rays x S=43 samples (bench.py)",
           "l2": "256 MB flush between steps", "torch": torch.__version__,
           "step_span_us": round(med(spans), 2), "glue_us": round(med(glue), 2),
           "kernels_sum_us": round(sum(k["us"] for k in kern), 2), "gaps_sum_us": round(sum(g["us"] for g in gaps), 2),
           "kernels": kern, "gaps": gaps}
    path = os.path.join(a.out, "glue_%s.json" % tag)
    with open(path, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({k: v for k, v in res.items() if k not in ("kernels", "gaps")}))


if __name__ == "__main__":
    main()
