#!/usr/bin/env python
"""bench.py -- lattice cells/s of the CTC best-path hot path (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload segments|chapters|gon|books]
                    [--scaling weak|strong]
    python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...
    python bench.py --impl reference ...      # the reference's own ctc_best_path on the host cores
    python bench.py --dump-outputs DIR ...    # also write the last timed step's outputs as DIR/<name>.npy

A "step" is one pass of the hot path over one batch of synthetic lattices.  The default
workload is BASELINE config 2 (10 000 silence-split segments of 1-10 s: T_b ~ U{86..861},
L_b = round(0.14 T_b), V = 39, beam_size 1000, max_move 4; SURVEY.md 8d) -- for these shapes
the window never clips, so evaluated cells == nominal T*S cells.

value  : cells/s with log_probs already resident in HBM (CUDA events on the launch stream).
e2e    : same metric through the host-buffer C-ABI call (pinned host memory, H2D of the
         log-probs and D2H of the three output arrays inside the timed region).
The default run also carries (rank 0, N = 1) the rest of the metric as sub-records: `gon`
(config 1) and `book` (config 3: device, host buffers, files -> files), `e2e_with_plan`
(kab_plan_create inside the timed region, as the reference expands its labels inside
ctc_best_path), `e2e_segment_records` (only align()'s per-segment numbers come back) and
`e2e_device_logits` (the encoder's logits never leave HBM).
Multi-GPU: one process per GPU, no collective on the data path.  --scaling weak (default): every
rank aligns its own batch; --scaling strong: ONE job (a book / 18 books) LPT-sharded over the
ranks.  time = max over ranks; value = cells of all ranks / that time.
"""
import os
os.environ.setdefault("TQDM_DISABLE", "1")   # (before anything imports tqdm: the reference wraps its frame loop in it)
import argparse
import contextlib
import io
import json
import os
import shutil
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from kokoro_align_b200 import parallel, synth  # noqa: E402

METRIC = "lattice cells/sec (TxS)"
UNIT = "cells/s"
REF_DIR = os.path.join(ROOT, "baseline", "_ref")


def band_kernel_name(info):
    """The kernel kab_plan_create chose for the band lattices (kab_plan_info.band_kernel)."""
    from kokoro_align_b200 import _lib
    name = _lib.BAND_KERNELS.get(int(info.band_kernel))
    return f"{name} (cluster of {int(info.band_cluster)})" if name and info.band_cluster > 1 else name


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def workload_shapes(name, seed, n_lattices=None):
    """(T[], L[], description) of a workload."""
    if name == "segments":      # BASELINE config 2
        B = n_lattices or 10000
        T, L = synth.segment_lengths(B, seed)
        return T, L, f"config2: {B} silence-split segments, T~U{{86..861}}, L=round(0.14T), V=39, W=1000, M=4"
    if name == "chapters":      # BASELINE config 3
        C = n_lattices or 36
        T, L = synth.chapter_lengths(C, 2721800, seed)
        return T, L, f"config3: Kokoro book, {C} chapter lattices, sum T=2721800, V=39, W=1000, M=4"
    if name == "books":         # a multi-book job: example.json lists 18 books (run_example.py:247-254 per book)
        nb = n_lattices or 18
        Ts, Ls = zip(*(synth.chapter_lengths(36, 2721800, seed + 31 * k) for k in range(nb)))
        return (np.concatenate(Ts), np.concatenate(Ls),
                f"{nb} config-3 books = {36 * nb} chapter lattices, sum T={2721800 * nb}, V=39, W=1000, M=4")
    if name == "gon":           # BASELINE config 1
        return (np.array([81135]), np.array([11359]),
                "config1: Gon gitsune single lattice T=81135 L=11359 V=39 W=1000 M=4")
    raise SystemExit(f"unknown workload {name}")


def workload_config(name, T, L, desc, world, scaling):
    """The `config` object: a function of the workload alone (computed on the CPU), so that the
    reference arm and the B200 arm print the SAME config."""
    cells = int(sum(parallel.cells_eval(int(t), int(l)) for t, l in zip(T, L)))
    nominal = int((T * (2 * L + 1)).sum())
    n_frames = int(T.sum())
    per = "per_gpu" if scaling == "weak" else "per_job"
    return {"workload": desc, f"lattices_{per}": int(len(T)), f"frames_{per}": n_frames,
            f"cells_eval_{per}": cells, f"cells_nominal_{per}": nominal,
            "l2": f"inputs ({n_frames * 39 * 4 / 1e6:.0f} MB log-probs per step) exceed the 126 MB L2"
                  if n_frames * 39 * 4 > 126e6 else
                  f"inputs ({n_frames * 39 * 4 / 1e6:.0f} MB log-probs) fit in L2: a 256 MB buffer is written between timed iterations",
            "parallelism": (f"{world} independent ranks, no collective on the data path" if scaling == "weak"
                            else f"one job LPT-sharded over {world} ranks, no collective on the data path")}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                 "-i", str(self.index), "-lms", "100"], stdout=subprocess.PIPE, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        self.thread.join(timeout=2)
        sm = [float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for k, n in enumerate(names) if any(len(r) > 3 + k and r[3 + k] == "Active" for r in self.rows)]
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": reasons}


# ------------------------------------------------------------------ the reference's CPU path
_REF = None


def reference_ctc_best_path():
    """kokoro_align.align.ctc_best_path of the UNMODIFIED reference, pip-installed into the
    git-ignored baseline/_ref by __graft_entry__.build() (it travels to the GPU box with the
    snapshot).  Falls back to the numpy port (oracle/ctc_oracle_np.py) when that install is
    absent.  Returns (callable, kind)."""
    global _REF
    if _REF is None:
        fn, kind = None, "port"
        if os.path.exists(os.path.join(REF_DIR, "kokoro_align", "align.py")):
            os.environ.setdefault("TQDM_DISABLE", "1")        # the reference wraps its frame loop in tqdm
            sys.path.insert(0, REF_DIR)
            try:
                from kokoro_align.align import ctc_best_path as ref_fn   # baseline/_ref, not the product
                fn, kind = ref_fn, "reference"
            except Exception as e:   # noqa: BLE001
                print(f"[bench] baseline/_ref not importable ({e}); timing the numpy port", file=sys.stderr)
            finally:
                sys.path.remove(REF_DIR)
        if fn is None:
            from oracle import ctc_oracle_np
            fn = ctc_oracle_np.ctc_best_path
        _REF = (fn, kind)
    return _REF


def _ref_call(lp, labels):
    fn, _ = reference_ctc_best_path()
    with contextlib.redirect_stdout(io.StringIO()), contextlib.redirect_stderr(io.StringIO()):
        return fn(lp, labels)                                 # (align.py:53-54 prints two lines per call, :62 a tqdm bar)


def _pool_job(args):
    lp, labels = args
    _ref_call(lp, labels)
    return parallel.cells_eval(lp.shape[0], labels.shape[0])


def reference_rate_one_core(lp, t_off, labels, l_off, budget_s, picks, check=None):
    """The reference on ONE core over lattices `picks` until budget_s; check(b, path) optional."""
    cells, t0, used = 0, time.perf_counter(), 0
    for b in picks:
        a, e = int(t_off[b]), int(t_off[b + 1])
        la, le = int(l_off[b]), int(l_off[b + 1])
        out = _ref_call(lp[a:e], labels[la:le].astype(np.int8))
        if check is not None:
            check(b, out[0])
        cells += parallel.cells_eval(e - a, le - la)
        used += 1
        if time.perf_counter() - t0 > budget_s:
            break
    dt = time.perf_counter() - t0
    return cells / dt, used, dt


def run_reference(args):
    """--impl reference: the reference's own CPU implementation of the path on all host cores
    (one process per core: ctc_best_path is single-threaded), bounded sample of the same workload
    per step.  Under torchrun only rank 0 works."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import multiprocessing as mp
    world = max(1, args.gpus)
    cores = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    T, L, desc = workload_shapes(args.workload, args.seed, args.lattices)
    config = workload_config(args.workload, T, L, desc, world, args.scaling)
    per_step = max(cores * 32, 64) if args.workload == "segments" else min(len(T), cores)
    n = min(len(T), per_step)
    order = np.random.default_rng(args.seed + 1).permutation(len(T))[:n]
    truncated = ""
    if args.workload != "segments":       # bound long lattices to ~20k frames each
        T, L = T.copy(), L.copy()
        for b in order:
            if T[b] > 20000:
                L[b] = int(round(L[b] * 20000 / T[b])); T[b] = 20000
        truncated = ", each cut to <= 20000 frames (same S/T)"
    jobs = [synth.make_lattice(int(T[b]), int(L[b]), 39, args.seed + 10 + int(b)) for b in order]
    _, kind = reference_ctc_best_path()
    with mp.get_context("fork").Pool(min(cores, n)) as pool:
        for _ in range(args.warmup):
            pool.map(_pool_job, jobs, chunksize=1)
        t0 = time.perf_counter()
        cells = 0
        for _ in range(args.steps):
            cells += sum(pool.map(_pool_job, jobs, chunksize=1))
        dt = time.perf_counter() - t0
    value = cells / dt
    what = ("kokoro_align.align.ctc_best_path (unmodified reference, baseline/_ref)" if kind == "reference"
            else "numpy port of align.py:43-109 (oracle/ctc_oracle_np.py)")
    sample = (f"{n} lattices of the workload per step (sum T={int(T[order].sum())}{truncated}), {what}, "
              f"multiprocessing.Pool({min(cores, n)})")
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3,
        "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None, "dtype": "f32",
        "data": "synthetic", "config": config,
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": min(cores, n), "kind": kind, "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }), flush=True)


# ------------------------------------------------------------------ B200 arm helpers
class L2Flush:
    """Between timed iterations of a workload whose inputs fit in the 126 MB L2: write 256 MB."""

    def __init__(self, dev, needed):
        import torch
        self.buf = torch.empty(256 << 20, dtype=torch.uint8, device=dev) if needed else None

    def __call__(self):
        if self.buf is not None:
            self.buf.fill_(1)


def time_device(plan, d_lp, steps, warmup, flush, barrier=lambda: None):
    """Device-resident steps: CUDA events around every plan.run_torch (the launch stream is torch's
    current stream); returns (per-step ms list, total ms over the K steps incl. gaps, last outputs)."""
    import torch
    outs = None
    for _ in range(warmup):
        outs = plan.run_torch(d_lp)
    torch.cuda.synchronize()
    barrier()
    ev0 = [torch.cuda.Event(enable_timing=True) for _ in range(steps)]
    ev1 = [torch.cuda.Event(enable_timing=True) for _ in range(steps)]
    for k in range(steps):
        flush()
        ev0[k].record()
        outs = plan.run_torch(d_lp)
        ev1[k].record()
    barrier()
    torch.cuda.synchronize()
    step_ms = [ev0[k].elapsed_time(ev1[k]) for k in range(steps)]
    return step_ms, outs


def sub_record(name, seed, steps, dev, peak, files_dir=None):
    """Configs 1 and 3 inside the default run: device-resident ms (CUDA events), e2e ms through
    kab_plan_run_host, cells/s, roofline; for the book also files -> files through best_path_files."""
    import torch
    from kokoro_align_b200 import align
    T, L, desc = workload_shapes(name, seed)
    lp, t_off, labels, l_off = synth.make_batch_fast(T, L, seed=seed + 1)
    rec = {"workload": desc}
    with align.AlignPlan(t_off, labels, l_off, 39, device=dev.index) as plan:
        info = plan.info
        h_lp = torch.from_numpy(lp).pin_memory()
        d_lp = h_lp.to(dev)
        flush = L2Flush(dev, lp.nbytes < 126e6)
        step_ms, outs = time_device(plan, d_lp, steps, 3, flush)
        assert (outs[4].cpu().numpy() == 0).all()
        ms = float(np.mean(step_ms))
        n = int(t_off[-1])
        out_np = (np.empty(n, np.int32), np.empty(n, np.int32), np.empty(n, np.float32),
                  np.empty(plan.B, np.float32), np.empty(plan.B, np.int32))
        for _ in range(2):
            plan.run_host(h_lp.numpy(), out=out_np)
        t0 = time.perf_counter()
        for _ in range(steps):
            plan.run_host(h_lp.numpy(), out=out_np)
        e2e_ms = (time.perf_counter() - t0) / steps * 1e3
        np.testing.assert_array_equal(out_np[0], outs[0].cpu().numpy())
        alg = int(info.algorithmic_bytes)
        rec.update({
            "device_ms": ms, "cells_eval": int(info.cells_eval), "cells_nominal": int(info.cells_nominal),
            "cells_per_s": info.cells_eval / (ms * 1e-3), "ns_per_frame_longest": ms * 1e6 / int(T.max()),
            "e2e_ms": e2e_ms, "e2e_cells_per_s": info.cells_eval / (e2e_ms * 1e-3),
            "kernel": band_kernel_name(info), "gpu_launches_per_step": int(info.kernel_launches),
            "roofline": {"bound": "hbm", "achieved": alg / (ms * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                         "frac": alg / (ms * 1e-3) / 1e9 / peak, "algorithmic_bytes_per_launch": alg,
                         "note": "ONE sequential recurrence per lattice: latency bound (DESIGN.md section 4)"}})
        del d_lp
    if files_dir:   # files -> files: run_example.py:247-254's loop over *.logits.npz / *.voca.txt
        from kokoro_align_b200 import encoder
        tokens = list(encoder.VOCAB[1:])
        rng = np.random.default_rng(seed + 2)
        lf, vf, bf = [], [], []
        for c in range(len(T)):
            lf.append(os.path.join(files_dir, f"c{c:02d}.logits.npz"))
            vf.append(os.path.join(files_dir, f"c{c:02d}.voca.txt"))
            bf.append(os.path.join(files_dir, f"c{c:02d}.best_path.npz"))
            a, b = int(t_off[c]), int(t_off[c + 1])
            np.savez(lf[-1], data=lp[a:b] * np.float32(3.0), indices=np.array([b - a], np.int32))
            ids = labels[int(l_off[c]):int(l_off[c + 1])] - 1
            with open(vf[-1], "w") as f:
                for k in range(0, len(ids), 8):
                    f.write("w|" + " ".join(tokens[i] for i in ids[k:k + 8]) + "\n")
        walls = {}
        for mode in ("host_numpy", "device", "host_numpy", "device"):    # second pass of each: warm
            for f in bf:
                if os.path.exists(f):
                    os.unlink(f)
            t0 = time.perf_counter()
            written = align.best_path_files(lf, vf, bf, verbose=False, device_log_softmax=(mode == "device"))
            walls[mode] = time.perf_counter() - t0
            assert len(written) == len(T)
        rec["files_to_files_s"] = {"log_softmax_numpy_host": walls["host_numpy"], "log_softmax_device": walls["device"],
                                   "what": f"{len(T)} *.logits.npz + *.voca.txt -> *.best_path.npz (align.best_path_files, {os.path.dirname(files_dir)})"}
    return rec


DUMP_BYTES = 64_000_000 - 4096     # --dump-outputs: 64 MB in all, .npy headers included


def dump_outputs(dirname, outs, t_off, budget, suffix=""):
    """--dump-outputs: what AlignPlan.run_torch returned (best_path, best_labels, best_scores per frame;
    final_score, status per lattice) as DIR/<name><suffix>.npy in float32, exact for these integers
    (all below 2^24).  When the batch's outputs exceed `budget` bytes, a fixed seeded sample of whole
    lattices is kept; lattice_index.npy names them, their frames stay in batch order."""
    path, labs, scores, final, status = (x.cpu().numpy() for x in outs)
    T = np.diff(t_off)
    order = np.random.default_rng(0).permutation(len(T))
    keep = np.zeros(len(T), bool)
    keep[order[np.cumsum(12 * T[order] + 12) <= budget]] = True    # 3 float32 per frame, 3 per lattice
    rows = np.repeat(keep, T)
    os.makedirs(dirname, exist_ok=True)
    for name, a in (("best_path", path[rows]), ("best_labels", labs[rows]), ("best_scores", scores[rows]),
                    ("final_score", final[keep]), ("status", status[keep]), ("lattice_index", np.flatnonzero(keep))):
        np.save(os.path.join(dirname, f"{name}{suffix}.npy"), a.astype(np.float32))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="segments", choices=["segments", "chapters", "gon", "books"])
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"])
    ap.add_argument("--lattices", type=int, default=None)
    ap.add_argument("--seed", type=int, default=2000)
    ap.add_argument("--cpu-seconds", type=float, default=15.0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the gon / book / hand-off sub-records")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed step as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup
    if args.impl == "reference":
        return run_reference(args)

    # libraries (NCCL prints its version) write to fd 1: keep the real stdout for the one JSON line
    sys.stdout.flush()
    json_fd = os.dup(1)
    os.dup2(2, 1)

    import torch
    import torch.distributed as dist
    from kokoro_align_b200 import align

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback)"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    cpus = parallel.bind_host_to_gpu(local_rank, world) if world > 1 else None   # NUMA-local pinned buffers
    strong = args.scaling == "strong"
    # ---- this rank's batch.  weak: every rank its own 10k segments / book; strong: the rank's
    # LPT shard (by evaluated cells) of ONE job
    if strong:
        T_all, L_all, desc = workload_shapes(args.workload, args.seed, args.lattices)
        config = workload_config(args.workload, T_all, L_all, desc, world, "strong")
        mine = parallel.shard_batch(T_all, L_all, rank, world)
        T, L = T_all[mine], L_all[mine]
    else:
        T, L, desc = workload_shapes(args.workload, args.seed + 7919 * rank, args.lattices)
        T0, L0, _ = workload_shapes(args.workload, args.seed, args.lattices)
        config = workload_config(args.workload, T0, L0, desc, world, "weak")
    lp, t_off, labels, l_off = synth.make_batch_fast(T, L, seed=args.seed + 1 + 7919 * rank)
    plan = align.AlignPlan(t_off, labels, l_off, 39, device=local_rank)
    info = plan.info
    cells_eval, cells_nominal = int(info.cells_eval), int(info.cells_nominal)
    n_frames = int(t_off[-1])

    # pinned host buffers for the e2e path
    h_lp = torch.from_numpy(lp).pin_memory()
    h_out = (torch.empty(n_frames, dtype=torch.int32).pin_memory(), torch.empty(n_frames, dtype=torch.int32).pin_memory(),
             torch.empty(n_frames, dtype=torch.float32).pin_memory(), torch.empty(plan.B, dtype=torch.float32).pin_memory(),
             torch.empty(plan.B, dtype=torch.int32).pin_memory())
    h_out_np = tuple(t.numpy() for t in h_out)
    d_lp = h_lp.to(dev, non_blocking=True)
    torch.cuda.synchronize()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if world > 1:
            t = torch.tensor([x], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            return float(t.item())
        return x

    def sum_over_ranks(x):
        if world > 1:
            t = torch.tensor([x], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.SUM)
            return float(t.item())
        return float(x)

    # ---- device-resident: value + roofline (CUDA events on the launching stream)
    flush = L2Flush(dev, lp.nbytes < 126e6)
    outs = None
    for _ in range(args.warmup):
        outs = plan.run_torch(d_lp)
    torch.cuda.synchronize()
    status = outs[4].cpu().numpy()
    assert (status == 0).all(), f"non-zero lattice status in bench: {np.unique(status)}"
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    barrier()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2 * args.steps)]
    for k in range(args.steps):
        flush()
        ev[2 * k].record()
        outs = plan.run_torch(d_lp)
        ev[2 * k + 1].record()
    barrier()
    step_ms = [ev[2 * k].elapsed_time(ev[2 * k + 1]) for k in range(args.steps)]
    # K steps back to back (first launch -> last completion); with an L2 flush between the steps
    # (inputs smaller than L2) the flushes are excluded: the sum of the K step times
    total_ms = max_over_ranks(float(np.sum(step_ms)) if flush.buf is not None else ev[0].elapsed_time(ev[2 * args.steps - 1]))
    cells_all = sum_over_ranks(cells_eval)
    nominal_all = sum_over_ranks(cells_nominal)
    value = cells_all * args.steps / (total_ms * 1e-3)
    kernel_ms = float(np.mean(step_ms))

    # ---- e2e: host buffers through the C-ABI (H2D + kernels + D2H per step)
    def timed_host(fn, reps=None):
        reps = reps or args.steps
        for _ in range(2):
            fn()
        barrier()
        t0 = time.perf_counter()
        for _ in range(reps):
            fn()
        barrier()
        return max_over_ranks(time.perf_counter() - t0) / reps

    e2e_s = timed_host(lambda: plan.run_host(h_lp.numpy(), out=h_out_np))
    e2e_value = cells_all / e2e_s
    clocks = sampler.stop() if rank == 0 else None   # sampled over both timed regions
    np.testing.assert_array_equal(h_out_np[0], outs[0].cpu().numpy())

    extras = {}
    if not args.no_extras:
        # ---- the same call on RAW LOGITS, align.py:116-117 on the device (kab_softmax.cuh)
        e2e_logits_s = timed_host(lambda: plan.run_host(h_lp.numpy(), out=h_out_np, logits=True))
        sm_ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
        d_tmp = torch.empty_like(d_lp)
        align.log_softmax_torch(d_lp, out=d_tmp)
        sm_ev[0].record()
        for _ in range(args.steps):
            align.log_softmax_torch(d_lp, out=d_tmp)
        sm_ev[1].record()
        torch.cuda.synchronize()
        softmax_ms = sm_ev[0].elapsed_time(sm_ev[1]) / args.steps
        extras["e2e_raw_logits"] = {"value": cells_all / e2e_logits_s, "unit": UNIT, "ms_per_step": e2e_logits_s * 1e3,
                                    "note": "same call on raw logits, log-softmax (align.py:116-117) on the device",
                                    "log_softmax_kernel_ms": softmax_ms,
                                    "log_softmax_gbs": 8.0 * n_frames * 39 / (softmax_ms * 1e-3) / 1e9}
        plan.run_host(h_lp.numpy(), out=h_out_np)   # restore the log-prob results for the parity spot check

        # ---- kab_plan_create INSIDE the timed region: the reference expands its labels inside
        # ctc_best_path (align.py:46-48); a new batch of transcripts pays classification + label
        # upload + workspace allocation (pooled after the first call)
        def with_plan():
            with align.AlignPlan(t_off, labels, l_off, 39, device=local_rank) as p2:
                p2.run_host(h_lp.numpy(), out=h_out_np)
        wp_s = timed_host(with_plan)
        extras["e2e_with_plan"] = {"value": cells_all / wp_s, "unit": UNIT, "ms_per_step": wp_s * 1e3,
                                   "note": "kab_plan_create + kab_plan_run_host + kab_plan_destroy per step"}

        # ---- only align()'s per-segment records come back (align.py:151-162 on the device)
        seg_idx = [np.array([int(t)], np.int32) for t in T] if args.workload == "segments" else \
                  [np.arange(500, int(t) + 499, 500, dtype=np.int32).clip(max=int(t)) for t in T]
        n_seg = int(sum(len(x) for x in seg_idx))
        seg_idx = align.flat_segments(seg_idx)      # (seg_lat_off, seg_end): built once, as a pipeline would
        rec_s = timed_host(lambda: plan.run_host_segments(h_lp.numpy(), seg_idx))
        extras["e2e_segment_records"] = {"value": cells_all / rec_s, "unit": UNIT, "ms_per_step": rec_s * 1e3,
                                         "segments": n_seg, "h2d_bytes_per_step": n_frames * 39 * 4 + (plan.B + 1 + n_seg) * 8,
                                         "d2h_bytes_per_step": n_seg * 24 + plan.B * 8,
                                         "note": "kab_plan_run_host_segments: boundaries, counts and both np.sum's per segment (numpy's pairwise order) instead of 12 B per frame"}

        # ---- the encoder's logits never leave HBM (train.py:215-229 -> align.py:113-117 without the
        # PCIe round trip): raw logits resident -> log-softmax in place -> alignment -> segment records
        d_logits = torch.empty_like(d_lp)

        def device_step():
            d_logits.copy_(d_lp)      # (stand-in for the encoder writing its output; outside the events)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            o = plan.run_torch(d_logits, logits=True)
            r = plan.segment_stats_torch(o[0], o[1], o[2], o[4], seg_idx)[0]
            host = r.cpu()            # 24 B per segment: the step's result read back
            e1.record()
            torch.cuda.synchronize()
            return e0.elapsed_time(e1), host
        for _ in range(2):
            device_step()
        dl_ms = float(np.mean([device_step()[0] for _ in range(args.steps)]))
        extras["e2e_device_logits"] = {"value": sum_over_ranks(cells_eval) / (max_over_ranks(dl_ms) * 1e-3), "unit": UNIT,
                                       "ms_per_step": dl_ms, "h2d_bytes_per_step": (plan.B + 1 + n_seg) * 8,
                                       "d2h_bytes_per_step": n_seg * 24,
                                       "note": "logits already in HBM (encoder output): kab_log_softmax_device in place + kab_plan_run_device + kab_plan_segment_stats_device, records read back"}
        del d_logits, d_tmp

    # ---- CPU baseline (rank 0, N = 1: bounded sample of the same workload, the reference on 1 core)
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        picks = np.random.default_rng(args.seed + 1).permutation(plan.B)
        _, kind = reference_ctc_best_path()
        lim = 20000 if args.workload != "segments" else None
        if lim is None:
            def check(b, ref_path):    # the reference's answer for the bench's own inputs == the GPU's
                np.testing.assert_array_equal(h_out_np[0][int(t_off[b]):int(t_off[b + 1])], ref_path)
            rate, used, dt = reference_rate_one_core(lp, t_off, labels, l_off, args.cpu_seconds, picks, check)
            sample = f"{used} randomly chosen lattices of the workload, {dt:.1f} s; every one of them compared with the GPU result (identical paths)"
        else:                          # long lattices: the first 20 000 frames of one chapter (same S/T)
            b = int(picks[0])
            a = int(t_off[b]); tl = min(lim, int(T[b])); ll = int(round(int(L[b]) * tl / int(T[b])))
            t0 = time.perf_counter()
            _ref_call(lp[a:a + tl], labels[int(l_off[b]):int(l_off[b]) + ll].astype(np.int8))
            dt = time.perf_counter() - t0
            rate, sample = parallel.cells_eval(tl, ll) / dt, f"first {tl} frames of one lattice of the workload, {dt:.1f} s"
        what = "kokoro_align.align.ctc_best_path (unmodified reference, baseline/_ref)" if kind == "reference" \
            else "numpy port of align.py:43-109 (oracle/ctc_oracle_np.py)"
        cpu = {"value": rate, "unit": UNIT, "cores": 1, "kind": kind, "sample": f"{sample}; {what}"}
        # parity spot check of the bench inputs against the C oracle
        from oracle import ctc_oracle
        for b in picks[:16]:
            a, e = int(t_off[b]), int(t_off[b + 1])
            rp = ctc_oracle.ctc_best_path(lp[a:e], labels[int(l_off[b]):int(l_off[b + 1])])[0]
            np.testing.assert_array_equal(h_out_np[0][a:e], rp)

    # ---- the rest of the metric (configs 1 and 3) as sub-records of the default run
    subs = {}
    peak, peak_src = load_peaks()
    if rank == 0 and world == 1 and args.workload == "segments" and not args.no_extras:
        plan.close()
        del d_lp, h_lp
        align.trim_pool()
        subs["gon"] = sub_record("gon", 1000, args.steps, dev, peak)
        # the book's files go to a fresh directory, in /dev/shm when writable (no disk I/O in the wall time)
        book_dir = tempfile.mkdtemp(prefix="kab_bench_book_", dir="/dev/shm" if os.access("/dev/shm", os.W_OK) else None)
        try:
            subs["book"] = sub_record("chapters", args.seed, args.steps, dev, peak, files_dir=book_dir)
        finally:
            shutil.rmtree(book_dir, ignore_errors=True)

    if args.dump_outputs:
        dump_outputs(args.dump_outputs, outs, t_off, DUMP_BYTES // world, f"_rank{rank}" if world > 1 else "")

    if rank == 0:
        achieved = int(info.algorithmic_bytes) / (kernel_ms * 1e-3) / 1e9
        prof = os.path.join(ROOT, "profiles", "ncu_traffic.json")
        traffic = None
        if os.path.exists(prof):
            with open(prof) as f:
                traffic = json.load(f).get(args.workload)
        plan_info = ({"kernel_classes": {"warp": int(info.n_class[0]), "band": int(info.n_class[1]),
                                          "generic": int(info.n_class[2]), "wide": int(info.n_class[3])},
                       "cells_nominal_per_s": nominal_all * args.steps / (total_ms * 1e-3),
                       "backpointer_bytes_per_gpu": int(info.backptr_bytes),
                       "host_binding": (f"rank 0 bound to {len(cpus)} cores (NVML affinity, split between the ranks that share it)" if cpus else "none")})
        out = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": total_ms / args.steps, "higher_is_better": True,
            "scaling": args.scaling, "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": config, "plan": plan_info,
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": n_frames * 39 * 4,
                    "d2h_bytes_per_step": n_frames * 12 + plan.B * 8, "ms_per_step": e2e_s * 1e3},
            "gpu_launches": int(info.kernel_launches) * args.steps,
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": achieved / peak, "traffic": traffic, "peak_source": peak_src,
                         "kernel": "kab_warp_kernel" if info.n_class[0] >= info.n_class[1] else band_kernel_name(info),
                         "algorithmic_bytes_per_launch": int(info.algorithmic_bytes), "kernel_ms": kernel_ms},
            "cpu_baseline": cpu, "clocks": clocks,
        }
        out.update(extras)
        out.update(subs)
        os.write(json_fd, (json.dumps(out) + "\n").encode())
    if not subs:
        plan.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
