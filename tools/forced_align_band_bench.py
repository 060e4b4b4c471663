"""Banded CTC forced alignment on the B200: banded plans (kab_plan_create_ctc_band, beam_size) against the
unbanded default and long-form plans wherever those can run.

    python tools/forced_align_band_bench.py --out profiles/r03_forced_align_band_bench.json

Emissions are planted paths: log_softmax of seeded Gaussian logits (V columns) plus a bonus of 6 on the token
of a CTC path that follows the diagonal S*t/T with a bounded sinusoidal drift, so that the unbanded best path
lies inside the band and banded and unbanded outputs can be compared byte for byte.  Each workload records its
largest drift |state - floor(S*t/T)| of the planted path.  L = 0.3 T (50 frames/s), blank 0, V = 32 unless said:
  (d) "batch": 256 utterances, T ~ U[6 000, 15 000] (2-5 minutes), W = 1000 and 2000, against the default plan
      (generic kernel) and the long-form plan;
  (c) "hour": one hour, T = 180 000, L = 54 000, W = 1000, against the long-form plan (wide kernel);
  (f) "three_hours": T = 540 000, L = 162 000, W = 2000; no unbanded plan can run it (beyond the wide kernel's
      resident chain, 84 GB of generic backpointers): time and backptr_bytes only;
  (v) "hour_v1025": (c) at V = 1025, blank 1024 (NeMo), targets drawn from 300 ids, so that the wide kernel takes
      the unbanded long-form plan on the compact copy (Vc <= 336).
Our time: CUDA events around plan.run_device, log-probs resident on the device, L2 flushed (a 512 MB write)
before every run, the plan built outside the timed window.  One JSON line per (workload, beam), with the
card's name and power limit read in the same run.
"""
import argparse
import json
import os
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from tools.forced_align_bench import card  # noqa: E402

WORKLOADS = {   # key: (utterances' T, V, blank, label pool size, beams, unbanded plans to compare with)
    "batch": (None, 32, 0, None, (1000, 2000), ("default", "long_form")),
    "hour": ([180000], 32, 0, None, (1000,), ("long_form",)),
    "three_hours": ([540000], 32, 0, None, (2000,), ()),
    "hour_v1025": ([180000], 1025, 1024, 300, (1000,), ("long_form",)),
}


def planted_states(T, tg, amp, cycles):
    """CTC state path along S*(t+1)/T + amp*sin(2 pi cycles t/T), as closely as the moves allow."""
    S = 2 * len(tg) + 1
    ext = np.zeros(S, np.int64)
    ext[1::2] = tg
    t = np.arange(T)
    goal = np.clip(np.floor(S * (t + 1) / T + amp * np.sin(2 * np.pi * cycles * t / T)).astype(np.int64), 0, S - 1)
    states = np.empty(T, np.int64)
    v = 0
    for i in range(T):
        if goal[i] > v:
            v += 2 if (v + 2 <= goal[i] and v % 2 == 1 and ext[v + 2] != ext[v]) else 1
        states[i] = v
    assert v >= S - 2
    return states, ext


def make_workload(kind, seed, dev):
    import torch
    Ts, V, blank, n_ids, beams, compare = WORKLOADS[kind]
    rng = np.random.default_rng(seed)
    T = rng.integers(6000, 15001, 256) if Ts is None else np.array(Ts)
    L = (0.3 * T).astype(np.int64)
    pool = np.array([x for x in range(V) if x != blank]) if n_ids is None else rng.choice(np.arange(1, 1024), n_ids, replace=False)
    tgs, toks, drift = [], [], 0
    for Tb, Lb in zip(T, L):
        tg = rng.choice(pool, int(Lb)).astype(np.int32)
        # a drift of at most ~150 states, well inside the narrowest band's half width (500), changing slowly
        st, ext = planted_states(int(Tb), tg, amp=150.0, cycles=max(1.0, Tb / 30000))
        drift = max(drift, int(np.abs(st - (2 * Lb + 1) * np.arange(Tb) // Tb).max()))
        tgs.append(tg)
        toks.append(ext[st])
    t_off = np.concatenate([[0], np.cumsum(T)]).astype(np.int64)
    l_off = np.concatenate([[0], np.cumsum(L)]).astype(np.int64)
    n = int(t_off[-1])
    g = torch.Generator(device=dev).manual_seed(seed)
    lp = torch.randn(n, V, device=dev, generator=g)
    tok = torch.from_numpy(np.concatenate(toks)).to(dev)
    lp[torch.arange(n, device=dev), tok] += 6.0
    lp = torch.log_softmax(lp, dim=-1).contiguous()
    return T, t_off, np.concatenate(tgs), l_off, V, blank, beams, compare, lp, drift


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--workloads", default="batch,hour,three_hours,hour_v1025")
    args = ap.parse_args()
    import torch
    from kokoro_align_b200 import align
    assert torch.cuda.is_available(), "needs a CUDA device"
    dev = torch.device("cuda", 0)
    name, power = card()
    flush = torch.empty(128 << 20, dtype=torch.float32, device=dev)
    s = torch.cuda.current_stream(dev)
    lines = []

    def measure(plan, lp, n, B):
        path = torch.empty(n, dtype=torch.int32, device=dev)
        labs = torch.empty_like(path)
        sc = torch.empty(n, dtype=torch.float32, device=dev)
        fs = torch.empty(B, dtype=torch.float32, device=dev)
        st = torch.empty(B, dtype=torch.int32, device=dev)

        def run():
            plan.run_device(lp.data_ptr(), path.data_ptr(), labs.data_ptr(), sc.data_ptr(), fs.data_ptr(), st.data_ptr(),
                            s.cuda_stream)
        run()   # warm-up: module load, first launches
        torch.cuda.synchronize()
        times = []
        for _ in range(args.reps):
            flush.fill_(1.0)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(s)
            run()
            e1.record(s)
            e1.synchronize()
            times.append(e0.elapsed_time(e1))
        out = [x.cpu().numpy() for x in (path, labs, sc, fs, st)]
        return times, out

    for kind in args.workloads.split(","):
        T, t_off, labels, l_off, V, blank, beams, compare, lp, drift = make_workload(kind, 1234, dev)
        n, B = int(t_off[-1]), len(T)
        ref = {}
        for mode in compare:
            plan = align.AlignPlan.ctc(t_off, labels, l_off, V, blank, long_form=(mode == "long_form"))
            times, out = measure(plan, lp, n, B)
            ref[mode] = dict(times=times, out=out, n_class=list(plan.info.n_class), backptr_bytes=int(plan.info.backptr_bytes))
            plan.close()
            torch.cuda.empty_cache()
        for W in beams:
            t0 = time.perf_counter()
            plan = align.AlignPlan.ctc(t_off, labels, l_off, V, blank, beam_size=W)
            plan_ms = (time.perf_counter() - t0) * 1e3
            info = plan.info
            times, out = measure(plan, lp, n, B)
            plan.close()
            torch.cuda.empty_cache()
            line = {
                "bench": "forced_align_band", "workload": kind, "beam_size": W, "utterances": B, "frames": n, "V": V,
                "blank": blank, "max_drift_states": drift, "status_counts": np.bincount(out[4], minlength=4).tolist(),
                "band_n_class": list(info.n_class), "band_ms_median": float(np.median(times)), "band_ms_all": times,
                "band_plan_create_ms": plan_ms, "band_backptr_bytes": int(info.backptr_bytes),
                "band_workspace_bytes": int(info.workspace_bytes), "band_cells_eval": int(info.cells_eval),
                "cells_nominal": int(info.cells_nominal),
            }
            for mode, r in ref.items():
                line.update({f"{mode}_ms_median": float(np.median(r["times"])), f"{mode}_ms_all": r["times"],
                             f"{mode}_n_class": r["n_class"], f"{mode}_backptr_bytes": r["backptr_bytes"],
                             f"speedup_vs_{mode}": float(np.median(r["times"]) / np.median(times)),
                             f"equal_{mode}": all(a.tobytes() == b.tobytes() for a, b in zip(out, r["out"]))})
            line.update(l2_flushed=True, timing="CUDA events around kab_plan_run_device, log-probs resident",
                        gpu=name, power_limit=power, torch=torch.__version__)
            print(json.dumps(line), flush=True)
            lines.append(line)
        del lp
        torch.cuda.empty_cache()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            for line in lines:
                f.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
