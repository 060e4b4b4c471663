"""Forward-backward posteriors of CTC alignments on the B200 (kab_plan_ctc_posteriors_device, DESIGN.md 3.9f):
the alignment (kab_plan_run_device) and the posterior pass timed separately on the same plan, against torch's
CUDA ctc_loss forward + backward on the same log-probs where its T x S tensors fit.

    python tools/ctc_posteriors_bench.py --out profiles/r03_ctc_posteriors_bench.json

Workloads (V = 32, blank 0, log_softmax of seeded Gaussian logits):
  "utterances": DESIGN.md 3.9's batch of 4 096 utterances, T ~ U[250, 1500], L = 0.3 T (default plan);
  "long":       3.9b's 10-minute utterance, T = 30 000, L = 9 000, S = 18 001 (long-form plan, unbanded);
  "chapter":    3.9d's one-hour chapter, T = 180 000, L = 54 000, beam_size = 1000 (banded plan).
CUDA events around each call, log-probs resident on the device, L2 flushed (a 512 MB write) before every timed
run, alignment and posterior pass alternated.  Peak memory: torch.cuda.max_memory_allocated over the call,
above what was allocated before it.  One JSON line per workload, with the card's name and power limit read in
the same run.
"""
import argparse
import ctypes
import json
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from tools.forced_align_bench import card, workload  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--workloads", default="utterances,long,chapter")
    args = ap.parse_args()
    import torch
    from kokoro_align_b200 import _lib, align
    assert torch.cuda.is_available(), "needs a CUDA device"
    dev = torch.device("cuda", 0)
    name, power = card()
    flush = torch.empty(128 << 20, dtype=torch.float32, device=dev)
    s = torch.cuda.current_stream(dev)
    L_ = _lib.lib()
    lines = []
    for kind in args.workloads.split(","):
        V, W = 32, None
        if kind == "chapter":
            rng = np.random.default_rng(4321)
            T = np.array([180000], np.int64)
            tgs = [rng.integers(1, V, 54000).astype(np.int32)]
            W = 1000
        else:
            T, tgs = workload(kind, 1234)
        g = torch.Generator(device=dev).manual_seed(99)
        lp = torch.log_softmax(2.0 * torch.randn(int(T.sum()), V, device=dev, generator=g), dim=-1).contiguous()
        B = len(T)
        t_off = np.concatenate([[0], np.cumsum(T)]).astype(np.int64)
        l_off = np.concatenate([[0], np.cumsum([len(x) for x in tgs])]).astype(np.int64)
        labels = np.concatenate(tgs)
        n = int(t_off[-1])
        plan = align.AlignPlan.ctc(t_off, labels, l_off, V, 0, long_form=kind != "utterances", beam_size=W)
        path, labs = torch.empty(n, dtype=torch.int32, device=dev), torch.empty(n, dtype=torch.int32, device=dev)
        sc, final = torch.empty(n, dtype=torch.float32, device=dev), torch.empty(B, dtype=torch.float32, device=dev)
        st = torch.empty(B, dtype=torch.int32, device=dev)
        post, ll = torch.empty(n, dtype=torch.float32, device=dev), torch.empty(B, dtype=torch.float64, device=dev)
        vp = ctypes.c_void_p

        def run_align():
            plan.run_device(lp.data_ptr(), path.data_ptr(), labs.data_ptr(), sc.data_ptr(), final.data_ptr(),
                            st.data_ptr(), s.cuda_stream)

        def run_post():
            _lib.check(L_.kab_plan_ctc_posteriors_device(plan._h, vp(lp.data_ptr()), vp(path.data_ptr()),
                                                         vp(st.data_ptr()), vp(ll.data_ptr()), vp(post.data_ptr()),
                                                         vp(s.cuda_stream)))
        run_align()
        torch.cuda.synchronize()
        run_post()   # (first call: the pass's set-up, outside the timed runs)
        torch.cuda.synchronize()
        times = {"align": [], "posteriors": []}
        for _ in range(args.reps):
            for k, fn in (("align", run_align), ("posteriors", run_post)):
                flush.fill_(1.0)
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(s)
                fn()
                e1.record(s)
                e1.synchronize()
                times[k].append(e0.elapsed_time(e1))
        status = st.cpu().numpy()
        assert (status == 0).all()
        am, pm = float(np.median(times["align"])), float(np.median(times["posteriors"]))
        S = 2 * np.array([len(x) for x in tgs]) + 1
        w = S if W is None else np.minimum(S, W)
        line = {
            "bench": "ctc_posteriors", "workload": kind, "utterances": B, "frames": n, "V": V, "beam_size": W,
            "S_max": int(S.max()), "cells_per_pass": int((T * w).sum()), "n_class": list(plan.info.n_class),
            "align_ms_median": am, "align_ms_all": times["align"],
            "posteriors_ms_median": pm, "posteriors_ms_all": times["posteriors"], "posteriors_over_align": pm / am,
            "posterior_gcells_per_s": 2 * float((T * w).sum()) / (pm * 1e6),
            "ours_workspace_bytes": int(plan.info.workspace_bytes),
            "ours_posterior_extra_bytes": int(16 * n + 4 * len(labels) + 48 * B),
            "ll_finite": bool(torch.isfinite(ll).all()), "post_median": float(post.median()),
        }
        plan.close()
        # torch: ctc_loss forward + backward on the same log-probs, padded [T_max, B, V], where it fits (the chapter's
        # alpha and beta are 180 000 x 108 001 floats, 78 GB each)
        try:
            if kind == "chapter":
                raise torch.cuda.OutOfMemoryError("not run: log_alpha and log_beta need 78 GB each")
            T_max, L_max = int(T.max()), int(max(len(x) for x in tgs))
            x = torch.zeros(T_max, B, V, device=dev)
            for b in range(B):
                x[:int(T[b]), b] = lp[int(t_off[b]):int(t_off[b + 1])]
            tg = torch.zeros(B, L_max, dtype=torch.long, device=dev)
            for b in range(B):
                tg[b, :len(tgs[b])] = torch.from_numpy(tgs[b]).to(dev)
            tl, tll = torch.from_numpy(T).to(dev), torch.tensor([len(x) for x in tgs], device=dev)
            x.requires_grad_(True)
            tt = []
            for r in range(1 + min(args.reps, 3)):
                x.grad = None
                flush.fill_(1.0)
                torch.cuda.synchronize()
                base = torch.cuda.memory_allocated(dev)
                torch.cuda.reset_peak_memory_stats(dev)
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(s)
                loss = torch.nn.functional.ctc_loss(x, tg, tl, tll, blank=0, reduction="none")
                loss.sum().backward()
                e1.record(s)
                e1.synchronize()
                if r:
                    tt.append(e0.elapsed_time(e1))
                peak = torch.cuda.max_memory_allocated(dev) - base
            if W is None:
                d = np.abs(-loss.detach().cpu().double().numpy() - ll.cpu().numpy())
                line.update(ll_max_abs_diff_vs_torch_fp32=float(d.max()))
            line.update(torch_ctc_loss_fwd_bwd_ms_median=float(np.median(tt)), torch_ctc_loss_fwd_bwd_ms_all=tt,
                        torch_peak_bytes=int(peak))
            del x, tg, loss
        except torch.cuda.OutOfMemoryError as e:
            line.update(torch_ctc_loss="out of memory", torch_error=str(e)[:200])
        torch.cuda.empty_cache()
        line.update(l2_flushed=True, timing="CUDA events, log-probs resident, alignment and posterior pass alternated",
                    gpu=name, power_limit=power, torch=torch.__version__)
        print(json.dumps(line), flush=True)
        lines.append(line)
        del lp, path, labs, sc, post
        torch.cuda.empty_cache()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            for line in lines:
                f.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
