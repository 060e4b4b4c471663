"""Long-form CTC forced alignment on the B200: long-form plans (kab_plan_create_ctc_long, the wide kernel
for S > 3296) against default plans (kab_plan_create_ctc, the generic kernel there) and torchaudio.

    python tools/forced_align_long_bench.py --out profiles/r03_forced_align_long_bench.json

Workloads (V = 32, blank 0, log-probs = log_softmax of seeded Gaussian logits, 50 frames/s, L = 0.3 T):
  (b) "long": one 10-minute utterance, T = 30 000, L = 9 000 (S = 18 001), tools/forced_align_bench.py's
      workload, plus torchaudio's CUDA and CPU forced_align;
  (c) "chapter": a one-hour chapter, T = 180 000, L = 54 000 (S = 108 001, 1.9e10 cells); the default plan
      runs once (about half a minute), torchaudio CPU only with --chapter-torchaudio-cpu; also the chain
      forced_align -> merge_tokens_batch -> word_spans by the host clock;
  (d) "batch": 256 utterances, T ~ U[6 000, 15 000] (2-5 minutes), all of them S > 3296.  The wide kernel
      runs its lattices one after another on the whole GPU, the generic kernel side by side; here the
      generic kernel is faster (230 against 276 ms when measured), and the long-form plan's makespan
      estimate keeps them there.  (b) and (c) are on the other side of that choice.
Our time: CUDA events around plan.run_device, log-probs resident on the device, L2 flushed (a 512 MB write)
before every run, the plan built outside the timed window.  torchaudio is timed once with a host clock
around a device synchronise.  Outputs are compared byte for byte.  One JSON line per workload, with the
card's name and power limit read in the same run.
"""
import argparse
import json
import os
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from tools.forced_align_bench import card, workload  # noqa: E402


def workload_long(kind, seed):
    if kind == "long":
        return workload("long", seed)
    rng = np.random.default_rng(seed)
    T = np.array([180000]) if kind == "chapter" else rng.integers(6000, 15001, 256)
    L = np.maximum(1, (0.3 * T).astype(np.int64))
    tgs = [rng.integers(1, 32, int(n)).astype(np.int32) for n in L]   # blank 0; adjacent repeats allowed
    return T.astype(np.int64), tgs


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--workloads", default="long,chapter,batch")
    ap.add_argument("--chapter-torchaudio-cpu", action="store_true", help="time torchaudio CPU on (c) (minutes)")
    args = ap.parse_args()
    import torch
    import torchaudio.functional as F
    from kokoro_align_b200 import align
    assert torch.cuda.is_available(), "needs a CUDA device"
    dev = torch.device("cuda", 0)
    name, power = card()
    flush = torch.empty(128 << 20, dtype=torch.float32, device=dev)
    s = torch.cuda.current_stream(dev)
    lines = []
    for kind in args.workloads.split(","):
        T, tgs = workload_long(kind, 1234)
        V, B = 32, len(T)
        t_off = np.concatenate([[0], np.cumsum(T)]).astype(np.int64)
        l_off = np.concatenate([[0], np.cumsum([len(x) for x in tgs])]).astype(np.int64)
        labels = np.concatenate(tgs)
        n = int(t_off[-1])
        g = torch.Generator(device=dev).manual_seed(99)
        lp = torch.log_softmax(2.0 * torch.randn(n, V, device=dev, generator=g), dim=-1).contiguous()
        res = {}
        for mode in ("long_form", "default"):
            t0 = time.perf_counter()
            plan = align.AlignPlan.ctc(t_off, labels, l_off, V, 0, long_form=(mode == "long_form"))
            plan_ms = (time.perf_counter() - t0) * 1e3
            info = plan.info
            path = torch.empty(n, dtype=torch.int32, device=dev)
            labs = torch.empty_like(path)
            sc = torch.empty(n, dtype=torch.float32, device=dev)
            fs = torch.empty(B, dtype=torch.float32, device=dev)
            st = torch.empty(B, dtype=torch.int32, device=dev)

            def run():
                plan.run_device(lp.data_ptr(), path.data_ptr(), labs.data_ptr(), sc.data_ptr(), fs.data_ptr(),
                                st.data_ptr(), s.cuda_stream)
            slow = mode == "default" and kind == "chapter"   # ~30 s: one timed run, no warm-up
            if not slow:
                run()   # warm-up: module load, first launches
                torch.cuda.synchronize()
            times = []
            for _ in range(1 if slow else args.reps):
                flush.fill_(1.0)
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(s)
                run()
                e1.record(s)
                e1.synchronize()
                times.append(e0.elapsed_time(e1))
            assert (st.cpu().numpy() == 0).all()
            res[mode] = dict(times=times, plan_ms=plan_ms, n_class=list(info.n_class), backptr_bytes=int(info.backptr_bytes),
                             workspace_bytes=int(info.workspace_bytes),
                             out=[x.cpu().numpy() for x in (path, labs, sc, fs)])
            plan.close()
            del path, labs, sc, fs, st
            torch.cuda.empty_cache()
        ours_labs, ours_sc = res["long_form"]["out"][1], res["long_form"]["out"][2]
        cells = int((T * (2 * np.array([len(x) for x in tgs]) + 1)).sum())
        lf, df = res["long_form"], res["default"]
        line = {
            "bench": "forced_align_long", "workload": kind, "utterances": B, "frames": n, "cells": cells, "V": V,
            "long_form_n_class": lf["n_class"], "default_n_class": df["n_class"],
            "long_form_ms_median": float(np.median(lf["times"])), "long_form_ms_all": lf["times"],
            "default_ms_median": float(np.median(df["times"])), "default_ms_all": df["times"],
            "long_form_plan_create_ms": lf["plan_ms"], "default_plan_create_ms": df["plan_ms"],
            "long_form_backptr_bytes": lf["backptr_bytes"], "default_backptr_bytes": df["backptr_bytes"],
            "long_form_workspace_bytes": lf["workspace_bytes"], "default_workspace_bytes": df["workspace_bytes"],
            "speedup_long_form_vs_default": float(np.median(df["times"]) / np.median(lf["times"])),
            "long_form_gcells_per_s": cells / float(np.median(lf["times"])) / 1e6,
            "equal_long_form_default": all(a.tobytes() == b.tobytes() for a, b in zip(lf["out"], df["out"])),
        }

        def ta(device, items):
            x = lp.to(device)
            outs = []
            if device.type == "cuda":
                F.forced_align(x[None, :int(T[0])], torch.from_numpy(tgs[0]).to(device)[None], blank=0)   # warm-up
                torch.cuda.synchronize()
            t0 = time.perf_counter()
            for b in items:
                outs.append(F.forced_align(x[None, int(t_off[b]):int(t_off[b + 1])], torch.from_numpy(tgs[b]).to(device)[None],
                                           blank=0))
            if device.type == "cuda":
                torch.cuda.synchronize()
            ms = (time.perf_counter() - t0) * 1e3
            return ms, torch.cat([o[0][0] for o in outs]).cpu().numpy(), torch.cat([o[1][0] for o in outs]).cpu().numpy()
        if kind == "long":
            ta_cuda_ms, pc, qc = ta(dev, range(B))
            ta_cpu_ms, pp, qp = ta(torch.device("cpu"), range(B))
            line.update(torchaudio_cuda_ms=ta_cuda_ms, torchaudio_cpu_ms=ta_cpu_ms,
                        speedup_vs_torchaudio_cuda=ta_cuda_ms / line["long_form_ms_median"],
                        speedup_vs_torchaudio_cpu=ta_cpu_ms / line["long_form_ms_median"],
                        equal_torchaudio_cpu=bool(np.array_equal(ours_labs, pp) and ours_sc.tobytes() == qp.tobytes()),
                        equal_torchaudio_cuda=bool(np.array_equal(ours_labs, pc) and ours_sc.tobytes() == qc.tobytes()))
        if kind == "chapter":
            if args.chapter_torchaudio_cpu:
                ta_cpu_ms, pp, qp = ta(torch.device("cpu"), range(B))
                line.update(torchaudio_cpu_ms=ta_cpu_ms,
                            equal_torchaudio_cpu=bool(np.array_equal(ours_labs, pp) and ours_sc.tobytes() == qp.tobytes()))
            # the Python chain from CUDA tensors: forced_align -> merge_tokens_batch -> word_spans (words of 1-9 tokens)
            wrng = np.random.default_rng(7)
            L = len(tgs[0])
            wl = []
            while sum(wl) < L:
                wl.append(int(min(wrng.integers(1, 10), L - sum(wl))))
            x, tg = lp[None], torch.from_numpy(tgs[0]).to(dev)[None]
            chain = []
            for _ in range(3):
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                p, q = align.forced_align(x, tg, blank=0, long_form=True)
                spans = align.merge_tokens_batch(p, q, blank=0)
                words = align.word_spans(spans, [wl])
                torch.cuda.synchronize()
                chain.append((time.perf_counter() - t0) * 1e3)
            line.update(chain_ms_all=chain, chain_ms_median=float(np.median(chain)),
                        chain_spans=int(spans.count[0]), chain_words=int(words.count[0]),
                        equal_chain_paths=bool(np.array_equal(p[0].cpu().numpy(), ours_labs)),
                        chain_timing="host clock, forced_align(long_form=True) + merge_tokens_batch + word_spans "
                                     "from a CUDA tensor to a synchronise (plan creation included)")
        line.update(l2_flushed=True, timing="CUDA events around kab_plan_run_device, log-probs resident",
                    gpu=name, power_limit=power, torch=torch.__version__)
        print(json.dumps(line), flush=True)
        lines.append(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            for line in lines:
                f.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
