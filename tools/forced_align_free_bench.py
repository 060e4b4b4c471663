"""CTC forced alignment with free ends on the B200: free-ends plans (kab_plan_create_ctc_free) against the plans
that align the whole recording (kab_plan_create_ctc for the utterances, kab_plan_create_ctc_long for the
chapter), on the same log-probs.

    python tools/forced_align_free_bench.py --out profiles/r03_forced_align_free_bench.json

Workloads (V = 32, blank 0):
  "utterances": DESIGN.md 3.9's batch of 4 096 utterances, T ~ U[250, 1500], L = 0.3 T, log_softmax of seeded
                Gaussian logits (warp and band kernels);
  "chapter":    a one-hour chapter, T = 180 000, L = 54 000 (wide kernel), whose transcript is planted in frames
                [3 000, 178 500): a 3 000-frame preamble and a 1 500-frame outro that favour the blank.
The two plans of a workload are built outside the timed window and timed alternately: CUDA events around
plan.run_device, log-probs resident on the device, L2 flushed (a 512 MB write) before every run.  One JSON line
per workload, with the card's name and power limit read in the same run.
"""
import argparse
import json
import os
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from tools.forced_align_bench import card, workload  # noqa: E402


def chapter(dev, seed):
    """(T [1], targets, log-probs on dev): the planted chapter."""
    import torch
    rng = np.random.default_rng(seed)
    T, L, V, a, b = 180000, 54000, 32, 3000, 178500
    tg = rng.integers(1, V, L).astype(np.int32)
    seq = []
    for k in range(L):
        if k and tg[k] == tg[k - 1]:
            seq.append(0)
        seq.append(int(tg[k]))
    n = b - a
    stay = np.bincount((np.arange(n - len(seq)) * len(seq)) // (n - len(seq)), minlength=len(seq))
    tok = np.repeat(np.asarray(seq), 1 + stay)
    g = torch.Generator(device=dev).manual_seed(seed)
    x = torch.randn(T, V, device=dev, generator=g)
    x[:a, 0] += 8.0
    x[b:, 0] += 8.0
    x[torch.arange(a, b, device=dev), torch.from_numpy(tok).to(dev)] += 8.0
    return np.array([T], np.int64), [tg], torch.log_softmax(x, dim=-1).contiguous()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--workloads", default="utterances,chapter")
    args = ap.parse_args()
    import torch
    from kokoro_align_b200 import align
    assert torch.cuda.is_available(), "needs a CUDA device"
    dev = torch.device("cuda", 0)
    name, power = card()
    flush = torch.empty(128 << 20, dtype=torch.float32, device=dev)
    s = torch.cuda.current_stream(dev)
    lines = []
    for kind in args.workloads.split(","):
        V = 32
        if kind == "chapter":
            T, tgs, lp = chapter(dev, 4321)
            base = "long_form"
        else:
            T, tgs = workload("utterances", 1234)
            g = torch.Generator(device=dev).manual_seed(99)
            lp = torch.log_softmax(2.0 * torch.randn(int(T.sum()), V, device=dev, generator=g), dim=-1).contiguous()
            base = "default"
        B = len(T)
        t_off = np.concatenate([[0], np.cumsum(T)]).astype(np.int64)
        l_off = np.concatenate([[0], np.cumsum([len(x) for x in tgs])]).astype(np.int64)
        labels = np.concatenate(tgs)
        n = int(t_off[-1])
        plans, outs, times, plan_ms = {}, {}, {"free_ends": [], base: []}, {}
        for mode in ("free_ends", base):
            t0 = time.perf_counter()
            plans[mode] = align.AlignPlan.ctc(t_off, labels, l_off, V, 0, long_form=mode != "default",
                                              free_ends=mode == "free_ends")
            plan_ms[mode] = (time.perf_counter() - t0) * 1e3
            outs[mode] = (torch.empty(n, dtype=torch.int32, device=dev), torch.empty(n, dtype=torch.int32, device=dev),
                          torch.empty(n, dtype=torch.float32, device=dev), torch.empty(B, dtype=torch.float32, device=dev),
                          torch.empty(B, dtype=torch.int32, device=dev))

        def run(mode):
            o = outs[mode]
            plans[mode].run_device(lp.data_ptr(), *(x.data_ptr() for x in o), s.cuda_stream)
        for mode in plans:   # warm-up: module load, first launches
            run(mode)
        torch.cuda.synchronize()
        for _ in range(args.reps):
            for mode in plans:
                flush.fill_(1.0)
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(s)
                run(mode)
                e1.record(s)
                e1.synchronize()
                times[mode].append(e0.elapsed_time(e1))
        fr, bs = [x.cpu().numpy() for x in outs["free_ends"]], [x.cpu().numpy() for x in outs[base]]
        assert (fr[4] == 0).all() and (bs[4] == 0).all()
        inside = fr[0] >= 0
        fm, bm = float(np.median(times["free_ends"])), float(np.median(times[base]))
        line = {
            "bench": "forced_align_free", "workload": kind, "utterances": B, "frames": n, "V": V, "baseline": base,
            "free_ends_ms_median": fm, "free_ends_ms_all": times["free_ends"],
            f"{base}_ms_median": bm, f"{base}_ms_all": times[base], "free_ends_over_baseline": fm / bm,
            "free_ends_n_class": list(plans["free_ends"].info.n_class), f"{base}_n_class": list(plans[base].info.n_class),
            "free_ends_plan_create_ms": plan_ms["free_ends"], f"{base}_plan_create_ms": plan_ms[base],
            "frames_outside_window": int((~inside).sum()),
            "final_free_ge_baseline": bool((fr[3] >= bs[3]).all()),
        }
        if kind == "chapter":
            w = np.flatnonzero(inside)
            line.update(window=[int(w[0]), int(w[-1])], planted=[3000, 178499])
        line.update(l2_flushed=True, timing="CUDA events around kab_plan_run_device, log-probs resident, the two "
                    "plans alternated", gpu=name, power_limit=power, torch=torch.__version__)
        print(json.dumps(line), flush=True)
        lines.append(line)
        for p in plans.values():
            p.close()
        del outs, lp
        torch.cuda.empty_cache()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            for line in lines:
                f.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
