#!/usr/bin/env python
"""Benchmark of the matching hot path: image-pairs/sec @640x480, indoor_ds dual-softmax (BASELINE.json).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--no-extra] [--dump-outputs DIR]

One "step" = one `matcher(batch)` call on a batch of 8 synthetic 640x480 grayscale pairs per GPU
(BASELINE.json configs[1]; weak scaling: every rank processes its own 8 pairs, then ONE NCCL all-gather of the
match lists).  Random-init weights (torch.manual_seed(0)), uniform-random images; thr = 0.0 so the fine level
actually runs (with random weights conf.max < the cfg default 0.2 and the fine path would be dead code,
SURVEY.md finding 3) -- recorded in `config`; the thr = 0.2 line is in `extra_workloads`.

Prints ONE JSON line (rank 0).  Keys follow the driver's contract:
  value      pairs/s, inputs resident in HBM, CUDA-event timed, max over ranks, L2 flushed between steps
  e2e        pairs/s through the public API with pinned-host inputs (H2D + D2H inside the timed region)
  roofline   the score-matrix kernel (EpiScoreLse pass of gemm_split_kernel): algorithmic 2*N*L*S*C flops per
             launch / its CUDA-event duration, against the measured bf16 peak of MEASURED_PEAKS.json
  cpu_baseline  the oracle port (PyTorch-CPU backbone + numpy restatement of the reference) on the host cores
  rank_ms    per-rank ms/step (min / median / max) and the CUDA-event time of the match all-gather alone
  gather_check  (N > 1) every rank verified that its slice of the gathered list equals its local result
  extra_workloads  the other BASELINE.json configs, same timing rules (N = 1: configs[2] shard, configs[3] sweep,
             configs[4] Sinkhorn, thr 0.2; N > 1: configs[2] = 4 pairs 832x832 per GPU + the all-gather)
`--impl reference` times that CPU port as the whole arm (rank 0 only).
`--dump-outputs DIR` writes the match lists of the last timed step (rank 0; the gathered lists when N > 1) as
DIR/<key>.npy, so that two builds can be compared output for output on the same seeded inputs.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

H, W_IMG = 480, 640
BATCH_PER_GPU = 8
METRIC = "image-pairs/sec @640x480 indoor_ds dual-softmax"
DTYPE = ("f32-equivalent: every product (backbone convolutions, transformer, score matrix) = 3x fp16 tcgen05 MMA "
         "(hi*hi + hi*lo + lo*hi) with fp32 accumulate; CUDA-core kernels fp32")


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--thr", type=float, default=0.0)
    ap.add_argument("--batch", type=int, default=BATCH_PER_GPU)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip the extra_workloads block")
    ap.add_argument("--backbone", default="b200", choices=["b200", "torch"],
                    help="b200: implicit-GEMM convolutions on tcgen05 (default); torch: PyTorch/cuDNN fp32 backbone")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the outputs of the last timed step as DIR/<key>.npy (float32 / float64)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the b200 arm")
    return args


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"hbm_gbs": d["hbm_gbs"], "bf16_tflops": d["bf16_tflops"],
                "bf16_tflops_sustained": d.get("bf16_tflops_sustained", d["bf16_tflops"]), "source": "measured"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback"}


def dump_outputs(out, dirname, max_bytes=64 << 20):
    """Every tensor of `out` -> <dirname>/<key>.npy: floating point stays float32 / float64, integer ids become float64
    (exact below 2^53), masks float32.  Above `max_bytes` in all, every array keeps the same seeded sample of rows."""
    import numpy as np
    import torch
    arrs = {}
    for k, v in out.items():
        if torch.is_tensor(v):
            a = v.detach().cpu().numpy()
            arrs[k] = a.astype(np.float64 if a.dtype == np.float64 or np.issubdtype(a.dtype, np.integer) else np.float32)
    total = sum(a.nbytes for a in arrs.values())
    if total > max_bytes:
        for k, a in arrs.items():
            n = a.shape[0]
            arrs[k] = a[np.sort(np.random.default_rng(0).choice(n, int(n * max_bytes / total), replace=False))]
    os.makedirs(dirname, exist_ok=True)
    for k, a in arrs.items():
        np.save(os.path.join(dirname, k + ".npy"), a)


# ------------------------------------------------------------------------------------------------ CPU arm
def cpu_pairs_per_sec(thr, steps, warmup, pairs_per_step=1):
    """PyTorch-CPU backbone + numpy oracle hot path on all host cores; each step = `pairs_per_step` pairs."""
    import numpy as np  # noqa: F401
    import torch
    import loftr_b200
    from oracle import loftr_oracle as O
    # all host cores up to 32 threads: beyond that the ~1-10 ms numpy / BLAS calls of this workload only
    # oversubscribe (measured on the 128-core GPU host: 12.1 s/pair with 128 threads)
    cores = min(os.cpu_count() or 1, 32)
    torch.set_num_threads(cores)
    try:
        from threadpoolctl import threadpool_limits
        threadpool_limits(limits=cores)
    except Exception:
        pass
    torch.manual_seed(0)
    cfg = loftr_b200.get_cfg("indoor_ds", thr=thr)
    model = loftr_b200.LoFTR(cfg).eval()
    state = {k: v.detach().numpy() for k, v in model.state_dict().items()}
    g = torch.Generator().manual_seed(0)
    img0 = torch.rand(pairs_per_step, 1, H, W_IMG, generator=g)
    img1 = torch.rand(pairs_per_step, 1, H, W_IMG, generator=g)
    times, m = [], 0
    for it in range(warmup + steps):
        t0 = time.perf_counter()
        with torch.no_grad():
            fc, ff = model.backbone(torch.cat([img0, img1], 0))
        (c0, c1), (f0, f1) = fc.split(pairs_per_step), ff.split(pairs_per_step)
        out = O.hot_path(c0.numpy(), c1.numpy(), f0.numpy(), f1.numpy(), state, cfg, (H, W_IMG), (H, W_IMG))
        dt = time.perf_counter() - t0
        m = len(out["b_ids"])
        if it >= warmup:
            times.append(dt)
    return pairs_per_step * len(times) / sum(times), cores, m, sum(times) / len(times)


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    steps, warmup = args.steps, max(0, args.warmup)
    v, cores, m, s_per_step = cpu_pairs_per_sec(args.thr, steps, warmup)
    sample = f"{steps} timed steps of 1 pair 640x480 (of the batch of {args.batch}), M={m} matches/pair"
    line = {
        "impl": "reference", "metric": METRIC, "value": v, "unit": "pairs/s", "n_gpus": args.gpus,
        "steps": steps, "warmup": warmup, "ms_per_step": s_per_step * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"batch={args.batch} 640x480 pairs, indoor_ds dual-softmax, thr={args.thr}",
                   "global_batch": args.batch * args.gpus, "thr": args.thr, "weights": "random-init seed 0"},
        "cpu_baseline": {"value": v, "unit": "pairs/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": v, "unit": "pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------ clocks
class ClockSampler:
    """`nvidia-smi -lms 25` in the background for the whole run (its start-up alone can take longer than a short timed
    region); `with sampler:` marks the timed region and summary() keeps the rows whose nvidia-smi timestamp falls
    inside it (same wall clock as datetime.now())."""
    Q = ("timestamp,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows, self.proc, self.index = [], None, index
        self.t0 = self.t1 = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "25", "-i", str(self.index)], stdout=subprocess.PIPE, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
            import atexit
            atexit.register(self.stop)       # every rank: never leave the sampling loop behind
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def __enter__(self):
        import datetime
        self.t0 = datetime.datetime.now()
        return self

    def __exit__(self, *a):
        import datetime
        self.t1 = datetime.datetime.now()

    def stop(self):
        if self.proc:
            time.sleep(0.1)   # let the rows of the last milliseconds arrive
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()
            self.proc = None

    @staticmethod
    def _ts(text):
        import datetime
        return datetime.datetime.strptime(text, "%Y/%m/%d %H:%M:%S.%f")

    def summary(self):
        self.stop()
        inside, near = [], []
        for r in self.rows:
            try:
                ts = self._ts(r[0])
            except Exception:
                continue
            if self.t0 is not None and self.t0 <= ts <= self.t1:
                inside.append(r)
            elif self.t0 is not None and abs((ts - self.t1).total_seconds()) < 0.25:
                near.append(r)
        use, where = (inside, "timed region") if inside else (near, "within 0.25 s of the timed region")
        sm, mx, reasons = [], 0, set()
        for r in use:
            try:
                sm.append(float(r[1]))
                mx = max(mx, float(r[2]))
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[4:8]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": mx or None, "samples": len(sm),
                "sampled": where, "reasons": sorted(reasons)}


# ------------------------------------------------------------------------------------------------ B200 arm
def run_b200(args):
    import torch
    import torch.distributed as dist
    import loftr_b200
    from loftr_b200 import _lib, parallel

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the B200 arm has no CPU fallback (use --impl reference for the CPU port)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    clk = ClockSampler(local)                        # sampling from now on; the timed region is marked with `with clk:`
    torch.backends.cudnn.allow_tf32 = False          # only matters for --backbone torch (fp32 parity mode)
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.benchmark = True

    B = args.batch
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)   # > 126 MB L2
    lib = _lib.load()
    stream = torch.cuda.current_stream()
    pk = peaks()
    t_start = time.perf_counter()

    def note(msg):
        print(f"[bench rank {rank} +{time.perf_counter() - t_start:6.1f}s] {msg}", file=sys.stderr, flush=True)

    def timed(fn, n):
        """per-step CUDA-event times (ms), L2 flushed (untimed) before every step"""
        evs = []
        for _ in range(n):
            flush.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            fn()
            e1.record(stream)
            evs.append((e0, e1))
        torch.cuda.synchronize()
        return [a.elapsed_time(b) for a, b in evs]

    def barrier():
        if world > 1 and dist.is_initialized():
            dist.barrier()
        torch.cuda.synchronize()

    def over_ranks(x, op="max"):
        if world == 1 or not dist.is_initialized():
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX if op == "max" else dist.ReduceOp.MIN)
        return float(t.item())

    def all_ranks(x):
        if world == 1 or not dist.is_initialized():
            return [x]
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        out = torch.empty(world, dtype=torch.float64, device=dev)
        dist.all_gather_into_tensor(out, t)
        return out.tolist()

    gatherer = [None]   # library-side NCCL communicator (created after the torch process group)

    class Workload:
        """One (cfg, batch, image size) configuration: model, device + pinned-host inputs, step functions."""

        def __init__(self, cfg_name, thr, batch, h, w, seed=1000):
            torch.manual_seed(0)
            self.cfg = loftr_b200.get_cfg(cfg_name, thr=thr)
            self.model = loftr_b200.LoFTR(self.cfg, backbone_impl=args.backbone).eval().to(dev)
            g = torch.Generator().manual_seed(seed + rank)
            self.h_img0 = torch.rand(batch, 1, h, w, generator=g).pin_memory()
            self.h_img1 = torch.rand(batch, 1, h, w, generator=g).pin_memory()
            self.d_img0, self.d_img1 = self.h_img0.to(dev), self.h_img1.to(dev)
            self.batch, self.h, self.w = batch, h, w
            self.L = (h // 8) * (w // 8)
            self.cap = batch * self.L
            self.lo_pair, _ = parallel.shard_range(batch * world, rank, world)
            self.out_host = {}

        def local_step(self, i0=None, i1=None):
            data = {"image0": self.d_img0 if i0 is None else i0, "image1": self.d_img1 if i1 is None else i1}
            self.model(data)
            return data

        def gather(self, data):
            return parallel.all_gather_matches(data, self.lo_pair, self.cap, gatherer=gatherer[0])

        def step(self):
            data = self.local_step()
            if world > 1 and dist.is_initialized():
                return data, self.gather(data)
            return data, None

        def e2e_step(self):
            i0 = self.h_img0.to(dev, non_blocking=True)
            i1 = self.h_img1.to(dev, non_blocking=True)
            d = self.local_step(i0, i1)
            if world > 1 and dist.is_initialized():
                d = self.gather(d)
            for k in ("mkpts0_f", "mkpts1_f", "mconf", "m_bids"):
                self.out_host[k] = d[k].cpu()

        def score_frac(self, nprof=3):
            """CUDA-event time of the score LSE kernel(s) inside `nprof` steps -> (avg_ms, launches/step, frac)."""
            _lib.timing_enable(True)
            for _ in range(nprof):
                flush.zero_()
                self.local_step()
            torch.cuda.synchronize()
            rec = _lib.timing_collect()
            _lib.timing_enable(False)
            ms, cnt = rec.get("score_lse", (0.0, 0))
            if not cnt:
                return None, rec, nprof
            flops = 2.0 * self.batch * self.L * self.L * self.cfg["coarse"]["d_model"]
            avg = ms / cnt
            return {"avg_launch_ms": avg, "launches_per_step": cnt / nprof, "flops_per_launch": flops,
                    "achieved_tflops": flops / (avg * 1e-3) * 1e-12,
                    "frac": flops / (avg * 1e-3) * 1e-12 / pk["bf16_tflops_sustained"]}, rec, nprof

    K, Wm = args.steps, max(3, args.warmup)
    main = Workload("indoor_ds", args.thr, B, H, W_IMG)
    hc, wc = H // 8, W_IMG // 8

    # algorithmic FLOPs of the backbone for one step, counted on a meta-device copy (no kernels are launched)
    import copy
    from torch.utils.flop_counter import FlopCounterMode
    with FlopCounterMode(display=False) as fcm:
        copy.deepcopy(main.model.backbone).to("meta")(torch.empty(2 * B, 1, H, W_IMG, device="meta"))
    backbone_flops = float(fcm.get_total_flops())

    # Phase A -- everything that loads CUDA kernels runs BEFORE the NCCL communicator exists.  With the
    # communicator created first, the first launch of every not-yet-loaded kernel module stalls for tens of
    # seconds on this image (measured with tools/mgpu_diag.py) -- slow module loading, not a deadlock.
    extra_defs = []
    if not args.no_extra:
        if world == 1:
            extra_defs = [
                ("configs[2] shard: 4 pairs 832x832 per GPU, outdoor_ds (of batch=32 over 8 GPUs)", "outdoor_ds", 0.0, 4, 832, 832),
                ("configs[4]: batch=8 640x480, indoor_ot Sinkhorn", "indoor_ot", 0.0, 8, H, W_IMG),
                ("configs[1] at the cfg default thr=0.2 (no confidence reaches it with random weights: M=0, fine level idle)",
                 "indoor_ds", 0.2, B, H, W_IMG),
            ] + [(f"configs[3] sweep: batch=1 {w_}x{h_}", "indoor_ds", 0.0, 1, h_, w_)
                 for h_, w_ in ((240, 320), (480, 640), (720, 960), (960, 1280))]
        else:
            extra_defs = [(f"configs[2]: batch={4 * world} 832x832 pairs, outdoor_ds, 4 per GPU over {world} GPUs + NCCL "
                           "all-gather of the match lists", "outdoor_ds", 0.0, 4, 832, 832)]
    extras = [(label, Workload(cfg_name, thr, b_, h_, w_, seed=2000 + i))
              for i, (label, cfg_name, thr, b_, h_, w_) in enumerate(extra_defs)]

    last = None
    for wl in [main] + [w for _, w in extras]:
        for _ in range(Wm if wl is main else 2):
            last_wl = wl.local_step()
            parallel.unpack_matches(parallel.pack_matches(last_wl, wl.lo_pair, 16384).unsqueeze(0))
        if wl is main:
            last = last_wl
    m_per_step = int(last["mconf"].shape[0])
    timed(main.e2e_step, 1)
    torch.tensor([1.0], dtype=torch.float64, device=dev).max().item()
    note("single-process warm-up done")
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        # NCCL prints its version banner to stdout while the communicator is created; stdout must carry exactly one
        # JSON line, so fd 1 points at stderr during initialisation and the collective warm-up.
        sys.stdout.flush()
        saved_stdout = os.dup(1)
        os.dup2(2, 1)
        dist.init_process_group("nccl", device_id=dev)
        gatherer[0] = parallel.MatchGatherer(dev)
        note("process group + library communicator up")
        for wl in [w for _, w in extras] + [main]:   # collective warm-up (NCCL channels, all-gather kernel)
            for _ in range(2):
                wl.step()
        # the GPUs idled (and dropped their clocks) while the communicators were being created: repeat the W warm-up
        # steps of the headline workload right before the timed region (measured at N = 2: 28.4 ms/step for the first
        # ten steps after the idle gap vs 24.8 ms afterwards, 1665 MHz vs 1965 MHz)
        # (r2w: eight steps were not always enough -- 28.05 ms/step timed right after them vs 22.5 ms a second later;
        # the count is fixed, not time-based, so that every rank issues the same number of collectives)
        for _ in range(max(Wm, 60)):
            main.step()
        torch.cuda.synchronize()
        over_ranks(0.0)
        barrier()
        sys.stdout.flush()
        os.dup2(saved_stdout, 1)
        os.close(saved_stdout)
    note("collective warm-up done")

    # ---- multi-GPU correctness: rank r's slice of the gathered list must equal its local result
    gather_check = None
    if world > 1:
        data, gathered = main.step()
        counts = gathered["counts"]
        lo = sum(counts[:rank])
        ok = counts[rank] == int(data["mconf"].shape[0])
        if ok:
            sl = slice(lo, lo + counts[rank])
            ok = (torch.equal(gathered["mkpts0_f"][sl], data["mkpts0_f"]) and
                  torch.equal(gathered["mkpts1_f"][sl], data["mkpts1_f"]) and
                  torch.equal(gathered["mconf"][sl], data["mconf"]) and
                  torch.equal(gathered["m_bids"][sl], data["m_bids"] + main.lo_pair))
        bids = gathered["m_bids"]
        ok = ok and bool((bids[1:] >= bids[:-1]).all().item()) and int(gathered["mconf"].shape[0]) == sum(counts)
        gather_check = over_ranks(1.0 if ok else 0.0, "min") == 1.0
        if not gather_check:
            raise SystemExit(f"bench.py rank {rank}: gathered match list does not reproduce the local result")

    # ---- device-resident throughput
    barrier()
    launches0 = lib.lb_launch_count()
    last_step = None

    def timed_step():
        nonlocal last_step
        last_step = main.step()

    with clk:
        ms_steps = timed(timed_step, K)
        barrier()
    launches = lib.lb_launch_count() - launches0
    my_ms = sum(ms_steps) / K
    rank_ms_list = all_ranks(my_ms)
    ms_step = max(rank_ms_list)
    value = B * world / (ms_step * 1e-3)
    note(f"device-resident timing done: {ms_step:.2f} ms/step")

    # collective alone (pack + NCCL all-gather + unpack on the result of one local step), CUDA events
    coll_ms = None
    if world > 1:
        data = main.local_step()
        barrier()
        cs = timed(lambda: main.gather(data), K)
        coll_ms = max(all_ranks(sum(cs) / K))

    # ---- end to end through the public API: pinned host images in, host match lists out
    for _ in range(2):
        main.e2e_step()
    barrier()
    t0 = time.perf_counter()
    ms_e2e_steps = timed(main.e2e_step, K)
    barrier()
    wall_e2e = (time.perf_counter() - t0) * 1e3
    ms_e2e = over_ranks(sum(ms_e2e_steps) / K)
    h2d = 2 * B * H * W_IMG * 4
    d2h = sum(v.numel() * v.element_size() for v in main.out_host.values())
    e2e = {"value": B * world / (ms_e2e * 1e-3), "unit": "pairs/s", "h2d_bytes_per_step": h2d,
           "d2h_bytes_per_step": d2h, "ms_per_step": ms_e2e, "wall_ms_per_step_incl_l2_flush": wall_e2e / K}
    note("e2e timing done")

    # ---- the other BASELINE.json configs (same timing rules; every rank runs them so collectives stay matched)
    extra_out = []
    for label, wl in extras:
        barrier()
        ms = timed(lambda: wl.step(), max(3, K // 2))
        ms_w = over_ranks(sum(ms) / len(ms))
        m_w = int(wl.local_step()["mconf"].shape[0])
        torch.cuda.synchronize()
        barrier()
        ms_e = timed(wl.e2e_step, max(3, K // 2))
        ms_e_w = over_ranks(sum(ms_e) / len(ms_e))
        rec = {"workload": label, "cfg": wl.cfg["match_coarse"]["match_type"], "thr": wl.cfg["match_coarse"]["thr"],
               "pairs_per_gpu": wl.batch, "image": f"{wl.w}x{wl.h}", "L": wl.L, "ms_per_step": ms_w,
               "pairs_per_s": wl.batch * world / (ms_w * 1e-3), "ms_per_pair": ms_w / wl.batch,
               "e2e_pairs_per_s": wl.batch * world / (ms_e_w * 1e-3), "matches_per_step_rank0": m_w}
        if rank == 0 or world == 1:
            sf, _, _ = wl.score_frac()
            if sf:
                rec["score_lse"] = sf
        barrier()
        extra_out.append(rec)
        note(f"extra workload done: {label}: {ms_w:.2f} ms/step")

    # ---- per-kernel CUDA-event timing of the tensor-core kernels (rank 0), separate pass
    roof, kernels = None, {}
    if rank == 0:
        sf, rec, nprof = main.score_frac()
        for tag, (ms, cnt) in rec.items():
            if cnt:
                kernels[tag] = {"launches_per_step": cnt / nprof, "avg_ms": ms / cnt, "total_ms_per_step": ms / nprof}
        if sf:
            traffic, traffic_src = None, None
            tp = os.path.join(ROOT, "profiles", "r2_score_lse_traffic.json")
            if os.path.exists(tp):
                tj = json.load(open(tp))
                traffic, traffic_src = tj.get("dram_bytes_per_launch"), tj.get("source")
            roof = {"kernel": "gemm_split_kernel<256, EpiScoreLse<rows,cols>> (score matrix + dual-softmax statistics)",
                    "bound": "tensor", "achieved": sf["achieved_tflops"], "peak": pk["bf16_tflops_sustained"],
                    "unit": "TFLOP/s", "frac": sf["frac"], "traffic": traffic, "traffic_source": traffic_src,
                    "peak_source": pk["source"] + " (bf16_tflops_sustained)",
                    "flops_per_launch": sf["flops_per_launch"], "avg_launch_ms": sf["avg_launch_ms"],
                    "issued_flops_factor": 3, "note": "three fp16 MMAs per product (hi*hi+hi*lo+lo*hi) for fp32-level accuracy; "
                    "frac counts algorithmic flops once"}
        if "backbone_conv" in kernels:
            tot_ms = kernels["backbone_conv"]["total_ms_per_step"]
            ach = backbone_flops / (tot_ms * 1e-3) * 1e-12
            kernels["backbone_conv"].update({"algorithmic_flops_per_step": backbone_flops, "achieved_tflops": ach,
                                             "frac_of_measured_bf16_sustained": ach / pk["bf16_tflops_sustained"]})
        tf_tags = [t for t in kernels if t.startswith("tf_") or t in ("proj_act", "merge_ln", "mlp1_relu", "mlp2_ln_res")]
        if tf_tags:
            # coarse + fine transformer GEMM launches; algorithmic coarse-transformer FLOPs: 103.2 GFLOP per pair at
            # 640x480 (SURVEY.md §8(a1)) scaled by L
            kernels["transformer_gemms_total_ms_per_step"] = sum(kernels[t]["total_ms_per_step"] for t in tf_tags)

    # ---- CPU baseline (rank 0, single GPU run only)
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        v, cores, m_cpu, s = cpu_pairs_per_sec(args.thr, steps=3, warmup=1)
        cpu = {"value": v, "unit": "pairs/s", "cores": cores, "kind": "port",
               "sample": f"3 timed forwards of 1 pair 640x480 after 1 warm-up ({s:.2f} s each, M={m_cpu}); "
                         "PyTorch-CPU backbone + numpy oracle of the reference hot path"}

    if rank == 0 and args.dump_outputs:
        local_out, gathered_out = last_step
        dump_outputs(gathered_out if gathered_out is not None else
                     {k: v for k, v in local_out.items() if k not in ("image0", "image1")}, args.dump_outputs)

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": "pairs/s", "n_gpus": world, "steps": K, "warmup": Wm,
            "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": DTYPE if args.backbone == "b200" else DTYPE + " (backbone: PyTorch/cuDNN fp32)",
            "data": "synthetic",
            "config": {"workload": f"batch={B} 640x480 pairs per GPU, indoor_ds dual-softmax, thr={args.thr}",
                       "global_batch": B * world, "thr": args.thr, "weights": "random-init seed 0",
                       "matches_per_step_rank0": m_per_step, "l2": "256 MiB flush buffer written before every timed step",
                       "backbone": ("ResNetFPN_8_2 as implicit-GEMM convolutions on tcgen05 (3x fp16 split, fp32 accumulate)"
                                    if args.backbone == "b200" else "PyTorch/cuDNN fp32 (TF32 off)"),
                       "parallelism": f"pairs sharded over {world} GPU(s), one NCCL all-gather of match lists"},
            "clocks": clk.summary(),
            "e2e": e2e, "gpu_launches": int(launches),
            "gpu_launches_per_step": launches / K,
            "rank_ms": {"per_rank_ms_per_step": rank_ms_list, "min": min(rank_ms_list),
                        "median": statistics.median(rank_ms_list), "max": max(rank_ms_list),
                        "all_gather_ms": coll_ms,
                        "note": "all_gather_ms = pack kernel + ncclAllGather + unpack kernel, CUDA events, max over ranks"},
            "gather_check": gather_check,
            "roofline": roof, "kernels": kernels, "cpu_baseline": cpu,
            "extra_workloads": extra_out,
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        gatherer[0].close()
        dist.destroy_process_group()


def main():
    args = parse()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
