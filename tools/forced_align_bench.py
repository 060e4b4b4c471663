"""CTC forced alignment on the B200: the CTC plans (kab_plan_create_ctc) against torchaudio's own
forced_align on CUDA and on CPU (one call per utterance: its batch dimension must be 1).

    python tools/forced_align_bench.py --out profiles/r03_forced_align_bench.json

Workloads (V = 32, log-probs = log_softmax of seeded Gaussian logits, 50 frames/s):
  (a) "utterances": 4 096 utterances, T ~ U[250, 1 500] (5-30 s), L = 0.3 T -- warp and band kernels;
  (b) "long": one 10-minute utterance, T = 30 000, L = 9 000 (S = 18 001) -- the generic kernel.
Our time: CUDA events around plan.run_device over --reps runs, log-probs already on the device, L2
flushed (a 512 MB write) before every run; the plan is built once, outside the timed window.  torchaudio
is timed once per workload with a host clock around a device synchronise.  The outputs of all three are
compared (paths and scores bit for bit).  One JSON line per workload, with the card's name and power
limit read in the same run.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        name, power = [x.strip() for x in out.split(",")[:2]]
        return name, power
    except Exception as e:  # noqa: BLE001
        import torch
        return torch.cuda.get_device_name(0), f"unknown ({e})"


def workload(kind, seed):
    rng = np.random.default_rng(seed)
    if kind == "utterances":
        T = rng.integers(250, 1501, 4096)
    else:
        T = np.array([30000])
    L = np.maximum(1, (0.3 * T).astype(np.int64))
    tgs = [rng.integers(1, 32, int(n)).astype(np.int32) for n in L]   # blank 0; adjacent repeats allowed
    return T.astype(np.int64), tgs


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--workloads", default="utterances,long")
    args = ap.parse_args()
    import torch
    import torchaudio.functional as F
    from kokoro_align_b200 import align
    assert torch.cuda.is_available(), "needs a CUDA device"
    dev = torch.device("cuda", 0)
    name, power = card()
    flush = torch.empty(128 << 20, dtype=torch.float32, device=dev)
    lines = []
    for kind in args.workloads.split(","):
        T, tgs = workload(kind, 1234)
        V, B = 32, len(T)
        t_off = np.concatenate([[0], np.cumsum(T)]).astype(np.int64)
        l_off = np.concatenate([[0], np.cumsum([len(x) for x in tgs])]).astype(np.int64)
        labels = np.concatenate(tgs)
        g = torch.Generator(device=dev).manual_seed(99)
        lp = torch.log_softmax(2.0 * torch.randn(int(t_off[-1]), V, device=dev, generator=g), dim=-1).contiguous()
        t0 = time.perf_counter()
        plan = align.AlignPlan.ctc(t_off, labels, l_off, V, 0)
        plan_ms = (time.perf_counter() - t0) * 1e3
        info = plan.info
        n = int(t_off[-1])
        path = torch.empty(n, dtype=torch.int32, device=dev)
        labs = torch.empty_like(path)
        sc = torch.empty(n, dtype=torch.float32, device=dev)
        fs = torch.empty(B, dtype=torch.float32, device=dev)
        st = torch.empty(B, dtype=torch.int32, device=dev)
        s = torch.cuda.current_stream(dev)

        def run():
            plan.run_device(lp.data_ptr(), path.data_ptr(), labs.data_ptr(), sc.data_ptr(), fs.data_ptr(),
                            st.data_ptr(), s.cuda_stream)
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
        ours_labs, ours_sc = labs.cpu().numpy(), sc.cpu().numpy()
        assert (st.cpu().numpy() == 0).all()
        plan.close()

        # torchaudio, one call per utterance: CUDA, then CPU
        def ta(device):
            x = lp.to(device)
            tg = [torch.from_numpy(t).to(device)[None] for t in tgs]
            outs = []
            if device.type == "cuda":
                F.forced_align(x[None, :int(T[0])], tg[0], blank=0)   # warm-up
                torch.cuda.synchronize()
            t0 = time.perf_counter()
            for b in range(B):
                outs.append(F.forced_align(x[None, int(t_off[b]):int(t_off[b + 1])], tg[b], blank=0))
            if device.type == "cuda":
                torch.cuda.synchronize()
            ms = (time.perf_counter() - t0) * 1e3
            p = torch.cat([o[0][0] for o in outs]).cpu().numpy()
            q = torch.cat([o[1][0] for o in outs]).cpu().numpy()
            return ms, p, q
        ta_cuda_ms, pc, qc = ta(dev)
        ta_cpu_ms, pp, qp = ta(torch.device("cpu"))
        cells = int((T * (2 * np.array([len(x) for x in tgs]) + 1)).sum())
        line = {
            "bench": "forced_align", "workload": kind, "utterances": B, "frames": n, "cells": cells, "V": V,
            "n_class": list(info.n_class), "kernel_launches": info.kernel_launches,
            "ours_ms_median": float(np.median(times)), "ours_ms_min": float(min(times)), "ours_ms_all": times,
            "ours_plan_create_ms": plan_ms,
            "torchaudio_cuda_ms": ta_cuda_ms, "torchaudio_cpu_ms": ta_cpu_ms,
            "speedup_vs_torchaudio_cuda": ta_cuda_ms / float(np.median(times)),
            "speedup_vs_torchaudio_cpu": ta_cpu_ms / float(np.median(times)),
            "equal_torchaudio_cpu": bool(np.array_equal(ours_labs, pp) and ours_sc.tobytes() == qp.tobytes()),
            "equal_torchaudio_cuda": bool(np.array_equal(ours_labs, pc) and ours_sc.tobytes() == qc.tobytes()),
            "l2_flushed": True, "timing": "CUDA events around kab_plan_run_device, log-probs resident",
            "gpu": name, "power_limit": power, "torch": torch.__version__,
        }
        print(json.dumps(line), flush=True)
        lines.append(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            for line in lines:
                f.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
