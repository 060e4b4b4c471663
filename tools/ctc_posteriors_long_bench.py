"""Forward-backward posteriors of unbanded long-form lattices on the chain-of-warps pass (DESIGN.md 3.9g), timed
next to the long-form alignment of the same plan and to the banded pass (beam_size=1000) of 3.9f.

    python tools/ctc_posteriors_long_bench.py --out profiles/r03_ctc_posteriors_long_bench.json

Workloads: 3.9b's one-hour chapter, T = 180 000, L = 54 000 (S = 108 001), log_softmax of seeded Gaussian logits
(2 randn), unbanded (kab_plan_create_ctc_long); "chapter" at V = 32, blank 0; "chapter_v1025" at V = 1025,
blank 1024, its targets drawn from 271 ids (the compact copy of 3.9c at Vc = 272: the alignment stays on the wide
kernel).  Per
workload, one plan each: the long-form plan (alignment, then the chain pass) and the banded plan at beam_size =
1000 (alignment, then the single-CTA banded pass).  CUDA events around each call, log-probs resident, L2 flushed
(a 512 MB write) before every timed run, the four calls alternated.  torch's float64 ctc_loss is not run: its
log_alpha and log_beta would need 156 GB each.  One JSON line per workload, with the card's name and power limit
read in the same run.
"""
import argparse
import ctypes
import json
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from tools.forced_align_bench import card  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--workloads", default="chapter,chapter_v1025")
    args = ap.parse_args()
    import torch
    from kokoro_align_b200 import _lib, align
    assert torch.cuda.is_available(), "needs a CUDA device"
    dev = torch.device("cuda", 0)
    name, power = card()
    flush = torch.empty(128 << 20, dtype=torch.float32, device=dev)
    s = torch.cuda.current_stream(dev)
    L_ = _lib.lib()
    vp = ctypes.c_void_p
    lines = []
    for kind in args.workloads.split(","):
        V, blank = (32, 0) if kind == "chapter" else (1025, 1024)
        T, Lb = 180000, 54000
        rng = np.random.default_rng(4321)
        ids = np.arange(1, V) if V == 32 else rng.choice(1024, 271, replace=False)
        tg = rng.choice(ids, Lb).astype(np.int32)
        g = torch.Generator(device=dev).manual_seed(99)
        lp = torch.log_softmax(2.0 * torch.randn(T, V, device=dev, generator=g), dim=-1).contiguous()
        t_off, l_off = np.array([0, T], np.int64), np.array([0, Lb], np.int64)
        plans = {"long": align.AlignPlan.ctc(t_off, tg, l_off, V, blank, long_form=True),
                 "band": align.AlignPlan.ctc(t_off, tg, l_off, V, blank, beam_size=1000)}
        bufs = {k: dict(path=torch.empty(T, dtype=torch.int32, device=dev), labs=torch.empty(T, dtype=torch.int32, device=dev),
                        sc=torch.empty(T, dtype=torch.float32, device=dev), final=torch.empty(1, dtype=torch.float32, device=dev),
                        st=torch.empty(1, dtype=torch.int32, device=dev), post=torch.empty(T, dtype=torch.float32, device=dev),
                        ll=torch.empty(1, dtype=torch.float64, device=dev)) for k in plans}

        def run_align(k):
            b = bufs[k]
            plans[k].run_device(lp.data_ptr(), b["path"].data_ptr(), b["labs"].data_ptr(), b["sc"].data_ptr(),
                                b["final"].data_ptr(), b["st"].data_ptr(), s.cuda_stream)

        def run_post(k):
            b = bufs[k]
            _lib.check(L_.kab_plan_ctc_posteriors_device(plans[k]._h, vp(lp.data_ptr()), vp(b["path"].data_ptr()),
                                                         vp(b["st"].data_ptr()), vp(b["ll"].data_ptr()),
                                                         vp(b["post"].data_ptr()), vp(s.cuda_stream)))
        for k in plans:
            run_align(k)
            torch.cuda.synchronize()
            run_post(k)   # (first call: the pass's set-up, outside the timed runs)
            torch.cuda.synchronize()
        calls = [("align_long", lambda: run_align("long")), ("posteriors_long", lambda: run_post("long")),
                 ("align_band1000", lambda: run_align("band")), ("posteriors_band1000", lambda: run_post("band"))]
        times = {k: [] for k, _ in calls}
        for _ in range(args.reps):
            for k, fn in calls:
                flush.fill_(1.0)
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(s)
                fn()
                e1.record(s)
                e1.synchronize()
                times[k].append(e0.elapsed_time(e1))
        assert int(bufs["long"]["st"][0]) == 0 and int(bufs["band"]["st"][0]) == 0
        med = {k: float(np.median(v)) for k, v in times.items()}
        pl, pb = bufs["long"], bufs["band"]
        line = {
            "bench": "ctc_posteriors_long", "workload": kind, "frames": T, "L": Lb, "S": 2 * Lb + 1, "V": V,
            "blank": blank, "n_class": list(plans["long"].info.n_class),
            **{f"{k}_ms_median": v for k, v in med.items()}, **{f"{k}_ms_all": v for k, v in times.items()},
            "posteriors_long_us_per_frame": 1e3 * med["posteriors_long"] / T,
            "posteriors_long_over_align_long": med["posteriors_long"] / med["align_long"],
            "posteriors_long_over_band1000": med["posteriors_long"] / med["posteriors_band1000"],
            "log_z_long": float(pl["ll"][0]), "log_z_band1000": float(pb["ll"][0]),
            "post_median_long": float(pl["post"].median()), "post_median_band1000": float(pb["post"].median()),
            "same_path": bool(torch.equal(pl["path"], pb["path"])),
            "torch_ctc_loss_fp64": "not run: log_alpha and log_beta need 156 GB each",
            "l2_flushed": True, "timing": "CUDA events, log-probs resident, the four calls alternated",
            "gpu": name, "power_limit": power, "torch": torch.__version__,
        }
        for p in plans.values():
            p.close()
        print(json.dumps(line), flush=True)
        lines.append(line)
        del lp, bufs
        torch.cuda.empty_cache()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            for line in lines:
                f.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
