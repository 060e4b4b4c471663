"""CTC forced alignment of wide vocabularies on the B200: the compact copy (kab_compact_ctc_kernel feeding
the warp, band and wide kernels, the default for V > 512) against the generic kernel (KAB_CTC_COMPACT=0,
the routing before the compact copy) and torchaudio.

    python tools/forced_align_vocab_bench.py --out profiles/r03_forced_align_vocab_bench.json

Workloads (log-probs = log_softmax of seeded Gaussian logits; token ids by a Zipf-like rank distribution,
p(rank r) ~ 1 / (r + 1), over a seeded permutation of the non-blank ids):
  (a) "utterances_v1025": 4 096 utterances, T ~ U[250, 1 500], L = 0.3 T, V = 1025, blank = 1024
      (tools/forced_align_bench.py's shape with NeMo's vocabulary);
  (b) "nemo_v1025": 4 096 utterances, T ~ U[60, 400] (80 ms frames), L = 0.3 T, V = 1025, blank = 1024;
  (c) "utterances_v5000": 1 024 utterances, T ~ U[100, 500], L = 0.2 T, V = 5000, blank = 0;
  (d) "long_v1025": long_form=True, one 10-minute utterance, T = 7 500, L = 2 500, ids from the 300
      highest ranks (wide kernel against generic).
Our time: CUDA events around plan.run_device over --reps runs, log-probs resident on the device, L2
flushed (a 512 MB write) before every run, plans built outside the timed window.  A separate profiled
run (torch.profiler) gives the kernels' device times, kab_compact_ctc_kernel's among them.  torchaudio:
CPU on --ta-cpu-sample utterances, CUDA's per-item loop on --ta-cuda-sample utterances, both by a host
clock around a device synchronise, extrapolated to the whole workload and labelled so.  Outputs of the two
arms are compared byte for byte, ours against torchaudio CPU on its sample.  One JSON line per workload,
with the card's name and power limit read in the same run.
"""
import argparse
import json
import os
import re
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from tools.forced_align_bench import card  # noqa: E402

MAX_STAGE_V = 512
WARP_STAGES, WARPS_PER_CTA, WARP_MINBLOCKS = 3, 4, 6   # kab_common.cuh / kab_warp.cuh
SMEM_PER_SM = 228 * 1024                               # B200: shared memory per SM (1 KB reserved per CTA)


def workload(kind, seed):
    """-> (V, blank, long_form, T [B], targets [B][L])."""
    rng = np.random.default_rng(seed)
    V, blank, long_form = {"utterances_v1025": (1025, 1024, False), "nemo_v1025": (1025, 1024, False),
                           "utterances_v5000": (5000, 0, False), "long_v1025": (1025, 1024, True)}[kind]
    if kind == "utterances_v1025":
        T, frac = rng.integers(250, 1501, 4096), 0.3
    elif kind == "nemo_v1025":
        T, frac = rng.integers(60, 401, 4096), 0.3
    elif kind == "utterances_v5000":
        T, frac = rng.integers(100, 501, 1024), 0.2
    else:
        T, frac = np.array([7500]), 2500 / 7500
    ids = rng.permutation(np.delete(np.arange(V), blank))     # rank -> token id
    n_rank = 300 if kind == "long_v1025" else V - 1
    p = 1.0 / np.arange(1, n_rank + 1)
    p /= p.sum()
    tgs = []
    for t in T:
        L = max(1, int(round(frac * t)))
        tg = ids[rng.choice(n_rank, L, p=p)].astype(np.int32)
        while L + int((tg[1:] == tg[:-1]).sum()) > t:   # (T >= L + R: redraw the rare over-repeated one)
            tg = ids[rng.choice(n_rank, L, p=p)].astype(np.int32)
        tgs.append(tg)
    return V, blank, long_form, T.astype(np.int64), tgs


def compact_width(tgs):
    """Vc by the plan's rule (kab_api.cu): 4-aligned, >= 8, over the lattices with <= 511 distinct labels."""
    d = [len(np.unique(tg)) for tg in tgs]
    fit = [x for x in d if x + 1 <= MAX_STAGE_V]
    vc = max(8, -(-(max(fit) + 1) // 4) * 4) if fit else 0
    return vc, int(max(d)), int(len(d) - len(fit))


def warp_ctas_per_sm(vc):
    """Resident CTAs of the warp kernel by shared memory, 128 + 4 (3 stage_bytes + 256) (kab_api.cu), and
    its __launch_bounds__ minimum of 6; arithmetic, not a measurement."""
    frames = 16 if vc <= 64 else 8
    stage = -(-(frames * vc * 4 + 24) // 16) * 16
    smem = 128 + WARPS_PER_CTA * (WARP_STAGES * stage + 256)
    return min(WARP_MINBLOCKS, SMEM_PER_SM // (smem + 1024)), smem


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--workloads", default="utterances_v1025,nemo_v1025,utterances_v5000,long_v1025")
    ap.add_argument("--ta-cpu-sample", type=int, default=64)
    ap.add_argument("--ta-cuda-sample", type=int, default=256)
    args = ap.parse_args()
    import torch
    import torchaudio.functional as F
    from torch.profiler import ProfilerActivity, profile
    from kokoro_align_b200 import align
    assert torch.cuda.is_available(), "needs a CUDA device"
    dev = torch.device("cuda", 0)
    name, power = card()
    flush = torch.empty(128 << 20, dtype=torch.float32, device=dev)
    s = torch.cuda.current_stream(dev)
    lines = []
    for kind in args.workloads.split(","):
        V, blank, long_form, T, tgs = workload(kind, 1234)
        B = len(T)
        t_off = np.concatenate([[0], np.cumsum(T)]).astype(np.int64)
        l_off = np.concatenate([[0], np.cumsum([len(x) for x in tgs])]).astype(np.int64)
        labels = np.concatenate(tgs)
        n = int(t_off[-1])
        g = torch.Generator(device=dev).manual_seed(99)
        lp = torch.empty(n, V, dtype=torch.float32, device=dev)
        for r0 in range(0, n, 1 << 18):   # (in chunks: no second full-size temporary)
            r1 = min(n, r0 + (1 << 18))
            lp[r0:r1] = torch.log_softmax(2.0 * torch.randn(r1 - r0, V, device=dev, generator=g), dim=-1)
        res = {}
        for arm in ("compact", "generic"):
            if arm == "generic":
                os.environ["KAB_CTC_COMPACT"] = "0"
            try:
                t0 = time.perf_counter()
                plan = align.AlignPlan.ctc(t_off, labels, l_off, V, blank, long_form=long_form)
                plan_ms = (time.perf_counter() - t0) * 1e3
            finally:
                os.environ.pop("KAB_CTC_COMPACT", None)
            info = plan.info
            out = [torch.empty(n, dtype=torch.int32, device=dev), torch.empty(n, dtype=torch.int32, device=dev),
                   torch.empty(n, dtype=torch.float32, device=dev), torch.empty(B, dtype=torch.float32, device=dev),
                   torch.empty(B, dtype=torch.int32, device=dev)]

            def run():
                plan.run_device(lp.data_ptr(), *(x.data_ptr() for x in out), s.cuda_stream)
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
            # kernel device times, in a run of their own (3 runs, L2 flushed before each)
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                for _ in range(3):
                    flush.fill_(1.0)
                    run()
                torch.cuda.synchronize()
            kern = {}
            for e in prof.key_averages():
                m = re.search(r"kab_\w+(<[^>]*>)?", e.key)
                if m:
                    us = getattr(e, "device_time_total", None)
                    if us is None:
                        us = e.cuda_time_total
                    kern[m.group(0)] = round(kern.get(m.group(0), 0.0) + us / 3 / 1e3, 4)   # ms per run
            res[arm] = dict(times=times, plan_ms=plan_ms, n_class=list(info.n_class), launches=int(info.kernel_launches),
                            kernels_ms=kern, out=[x.cpu().numpy() for x in out])
            plan.close()
            del out
            torch.cuda.empty_cache()
        c, gn = res["compact"], res["generic"]
        assert (c["out"][4] == 0).all() and (gn["out"][4] == 0).all()
        S = 2 * np.array([len(x) for x in tgs]) + 1
        cells = int((T * S).sum())
        vc, dmax, n_over = compact_width(tgs)
        ctas, wsmem = warp_ctas_per_sm(vc)
        cmp_ms = c["kernels_ms"].get("kab_compact_ctc_kernel", float("nan"))
        line = {
            "bench": "forced_align_vocab", "workload": kind, "V": V, "blank": blank, "long_form": long_form,
            "utterances": B, "frames": n, "cells": cells, "Vc": vc, "max_distinct_labels": dmax,
            "lattices_over_511_distinct": n_over,
            "compact_n_class": c["n_class"], "generic_n_class": gn["n_class"],
            "compact_kernel_launches": c["launches"], "generic_kernel_launches": gn["launches"],
            "compact_ms_median": float(np.median(c["times"])), "compact_ms_all": c["times"],
            "generic_ms_median": float(np.median(gn["times"])), "generic_ms_all": gn["times"],
            "speedup_compact_vs_generic": float(np.median(gn["times"]) / np.median(c["times"])),
            "compact_gcells_per_s": cells / float(np.median(c["times"])) / 1e6,
            "compact_plan_create_ms": c["plan_ms"], "generic_plan_create_ms": gn["plan_ms"],
            "compact_kernels_ms": c["kernels_ms"], "generic_kernels_ms": gn["kernels_ms"],
            "compact_kernel_ms": cmp_ms,
            "compact_kernel_bytes": n * V * 4 + n * vc * 4,
            "compact_kernel_tb_per_s": (n * V * 4 + n * vc * 4) / (cmp_ms * 1e-3) / 1e12,
            "compact_kernel_timing": "torch.profiler device time, mean of 3 runs with L2 flushed, separate from the timed runs",
            "warp_ctas_per_sm_by_arithmetic": ctas, "warp_smem_bytes": wsmem,
            "equal_compact_generic": all(a.tobytes() == b.tobytes() for a, b in zip(c["out"], gn["out"])),
        }
        if long_form:
            line["compact_ns_per_frame"] = float(np.median(c["times"])) * 1e6 / n

        def ta(device, items):
            outs = []
            if device.type == "cuda":
                b = items[0]
                F.forced_align(lp[None, int(t_off[b]):int(t_off[b + 1])], torch.from_numpy(tgs[b]).to(device)[None], blank=blank)
                torch.cuda.synchronize()
            xs = [lp[int(t_off[b]):int(t_off[b + 1])].to(device)[None] for b in items]
            ys = [torch.from_numpy(tgs[b]).to(device)[None] for b in items]
            if device.type == "cuda":
                torch.cuda.synchronize()
            t0 = time.perf_counter()
            for x, y in zip(xs, ys):
                outs.append(F.forced_align(x, y, blank=blank))
            if device.type == "cuda":
                torch.cuda.synchronize()
            ms = (time.perf_counter() - t0) * 1e3
            return ms, [(o[0][0].cpu().numpy(), o[1][0].cpu().numpy()) for o in outs]
        rng = np.random.default_rng(5)
        cpu_items = sorted(rng.choice(B, min(B, args.ta_cpu_sample), replace=False).tolist())
        cuda_items = sorted(rng.choice(B, min(B, args.ta_cuda_sample), replace=False).tolist())
        ta_cpu_ms, cpu_out = ta(torch.device("cpu"), cpu_items)
        ta_cuda_ms, cuda_out = ta(dev, cuda_items)
        labs, sc = c["out"][1], c["out"][2]

        def equal(items, outs):
            return all(np.array_equal(labs[t_off[b]:t_off[b + 1]], p) and sc[t_off[b]:t_off[b + 1]].tobytes() == q.tobytes()
                       for b, (p, q) in zip(items, outs))
        fr_cpu = float(T[cpu_items].sum()) / n
        fr_cuda = float(T[cuda_items].sum()) / n
        line.update(
            torchaudio_cpu_sample=len(cpu_items), torchaudio_cpu_sample_ms=ta_cpu_ms,
            torchaudio_cpu_ms_extrapolated=ta_cpu_ms / fr_cpu,
            torchaudio_cuda_sample=len(cuda_items), torchaudio_cuda_sample_ms=ta_cuda_ms,
            torchaudio_cuda_ms_extrapolated=ta_cuda_ms / fr_cuda,
            torchaudio_extrapolation="sample time x (all frames / sample frames); not measured on the whole workload"
                                     if len(cpu_items) < B or len(cuda_items) < B else "whole workload",
            equal_torchaudio_cpu=bool(equal(cpu_items, cpu_out)),
            torchaudio_cuda_same_as_ours=bool(equal(cuda_items, cuda_out)),   # (not a reference: see DESIGN.md 3.9)
            l2_flushed=True, timing="CUDA events around kab_plan_run_device, log-probs resident",
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
