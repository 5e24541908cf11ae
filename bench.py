#!/usr/bin/env python
"""Benchmark of the FACT hot path on B200: autoregressive motion frames/sec (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--batch B] [--mode precise|bf16] [--impl ours|reference]
                    [--dump-outputs DIR]

A "step" is one autoregressive frame for the whole batch: one full FACT forward (motion encoder, audio encoder,
12-layer cross-modal stack, head on row 0) over [B,120,225] motion + [B,240,35] audio, plus the shift-by-one
(reference: mint/core/fact_model.py:103-132).  Workload = the north_star target configuration: batch 128 clips per
GPU, fact_v5_deeper_t10_cm12, random-init weights, synthetic N(0,1) inputs.  Multi-GPU = independent clips per rank
(weak scaling, no data-path collective; only the timing barrier / max-reduce use NCCL).

Prints ONE JSON line (rank 0).  `value` = frames/s with inputs resident in HBM; `e2e` = the same through the public
`FACTModel.infer_auto_regressive` with pinned HOST inputs and a host copy of the result inside the timed region;
`roofline` = the dominant kernel (tcgen05 GEMM) timed live with CUDA events; `cpu_baseline` = the torch-CPU fp32
port of the reference math (TensorFlow is not installable in this image) on a bounded sample.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "autoregressive motion frames/sec"
WORKLOAD = "fact_v5_deeper_t10_cm12 autoregressive generate"
FLOP_PER_FRAME = 80.97e9  # SURVEY.md 8(d): one full forward per generated frame per clip
DUMP_BYTES = 64 << 20     # cap of --dump-outputs


def positive_int(text):
    v = int(text)
    if v < 1:
        raise argparse.ArgumentTypeError(f"must be at least 1, got {v}")
    return v


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=positive_int, default=12,
                    help="timed steps: AR frames per clip in the generation legs and the batch sweep, optimizer steps "
                         "in the training leg (the single-clip and CPU legs have their own options)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--batch", type=int, default=128, help="clips per GPU")
    ap.add_argument("--mode", default="precise", choices=["precise", "bf16"])
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-extras", action="store_true", help="skip roofline / cpu_baseline / fast-mode legs")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg only")
    ap.add_argument("--cpu-frames", dest="cpu_frames", type=int, default=120,
                    help="upper bound on the AR frames per clip of the cpu_baseline sample (the sample is sized to "
                         "~12 s of CPU work at the calibrated rate)")
    ap.add_argument("--train-batch", dest="train_batch", type=int, default=128,
                    help="clips per GPU of the training leg (BASELINE.json configs[2]/[3])")
    ap.add_argument("--no-train", action="store_true", help="skip the data-parallel training leg")
    ap.add_argument("--dp-overlap", dest="dp_overlap", default="auto",
                    choices=["auto", "fused", "fused_tail", "adam", "backward", "none"],
                    help="how the training leg hides its gradient all-reduce (mint_b200/trainer.py)")
    ap.add_argument("--no-sweep", action="store_true", help="skip the batch 1->512 sweep leg (configs[4])")
    ap.add_argument("--sweep", default="1,2,4,8,16,32,64,128,256,512", help="clips per GPU of the sweep leg")
    ap.add_argument("--b1-frames", dest="b1_frames", type=int, default=1200,
                    help="frames of the single-clip leg (configs[1]: 1200 = 20 s at 60 fps)")
    ap.add_argument("--kernels-only", action="store_true", help="developer aid: time the hot kernels alone and exit")
    ap.add_argument("--flag", action="append", default=[], help="developer aid: fact_set_flag name=value")
    ap.add_argument("--dump-outputs", dest="dump_outputs", metavar="DIR",
                    help="after the timed steps, write the frame the last timed step generated for each of rank 0's "
                         "clips to DIR/last_frame.npy (float32, [batch, 225]) for output-for-output comparison of two "
                         "builds; inputs and weights are seeded, so the same arguments give the same inputs")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl != "ours" or args.kernels_only):
        ap.error("--dump-outputs writes the outputs of the timed generation of --impl ours")
    return args


def dump_outputs(out_dir, name, t):
    """Save `t` ([rows, ...]) as out_dir/<name>.npy in float32; above DUMP_BYTES a fixed, seeded sample of its rows
    (sorted row order), so that two runs with the same arguments store the same rows."""
    import numpy as np
    a = t.detach().float().cpu().numpy()
    if a.nbytes > DUMP_BYTES:
        keep = DUMP_BYTES // (a.nbytes // a.shape[0])
        a = a[np.sort(np.random.default_rng(0).choice(a.shape[0], keep, replace=False))]
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, name + ".npy"), a)


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return {"hbm_gbs": d["hbm_gbs"], "bf16_tflops": d["bf16_tflops"],
                "bf16_tflops_sustained": d.get("bf16_tflops_sustained", d["bf16_tflops"]), "source": "measured"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback"}


class ClockSampler:
    """nvidia-smi clocks + throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100", "-i",
                 str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._pump, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append((time.perf_counter(), line.strip()))

    def stop(self, t0, t1):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unsampled"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ts, line in self.lines:
            parts = [p.strip() for p in line.split(",")]
            if len(parts) < 7:
                continue
            try:
                mx = float(parts[1])
                if t0 - 0.05 <= ts <= t1 + 0.1:
                    sm.append(float(parts[0]))
                    for nm, v in zip(names, parts[3:7]):
                        if v.lower().startswith("active"):
                            reasons.add(nm)
            except ValueError:
                continue
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


# --------------------------------------------------------------------------------------------- reference arm (CPU)
def _cpu_worker(idx, threads, steps, warmup, q, batch=1):
    """One CPU replica: AR generation of `batch` clips with the torch-CPU fp32 port (clips are independent, like on the
    GPU)."""
    import torch
    from oracle import fact_oracle as O, fact_oracle_torch as OT
    torch.set_num_threads(threads)
    dims = O.FACT_V5
    w = OT.to_torch(O.init_weights(dims, seed=0))
    inp = O.synthetic_inputs(dims, batch, audio_len=dims.audio_seq + warmup + steps - 1, seed=idx)
    tin = {k: torch.from_numpy(v).float() for k, v in inp.items()}
    motion = tin["motion_input"]
    q.put(("ready", idx))
    t_total = 0.0
    with torch.no_grad():
        for i in range(warmup + steps):
            t0 = time.perf_counter()
            window = tin["audio_input"][:, i:i + dims.audio_seq]
            first = OT.call(w, dims, {"motion_input": motion, "audio_input": window})[:, :1]
            motion = torch.cat([motion[:, 1:], first], dim=1)
            if i >= warmup:
                t_total += time.perf_counter() - t0
    q.put(("done", idx, t_total))


def cpu_frames_per_sec(steps, warmup, procs=1, threads=None, target_seconds=None):
    """Torch-CPU fp32 restatement of the reference math on the host cores, AR generation.

    Measured on the GPU box (Xeon 8562Y+, 128 hardware threads): one process is fastest at 16 intra-op threads (67 ms
    per forward = 15 frames/s); 32 / 64 / 128 threads are slower, and 8 side-by-side replicas x 16 threads drop to
    6.9 frames/s IN TOTAL (memory-bound weight streaming, 0.5 GB per forward per replica).  So the baseline is ONE
    replica, with the thread count AND the clips per forward calibrated on single forwards (a bigger batch gives the
    CPU GEMMs more rows to spread over the cores): that is the most this port gets out of the box.
    Returns (clip-frames/s, seconds, threads_total, description)."""
    import torch
    from oracle import fact_oracle as O, fact_oracle_torch as OT
    ncpu = os.cpu_count() or 1
    batch = 1
    if threads is None:
        dims = O.FACT_V5
        w = OT.to_torch(O.init_weights(dims, seed=0))
        best = (0.0, min(16, ncpu), 1)                         # (clip-frames/s, threads, batch)
        cands = {(c, 1) for c in (8, 16, 32, 64) if c <= ncpu}
        cands |= {(c, b) for c, b in ((32, 4), (64, 8), (ncpu, 16), (ncpu, 8)) if c <= ncpu}
        for cand, b in sorted(cands):
            one = {k: torch.from_numpy(v).float() for k, v in O.synthetic_inputs(dims, b, seed=1).items()}
            torch.set_num_threads(cand)
            with torch.no_grad():
                OT.call(w, dims, one)
                t0 = time.perf_counter()
                OT.call(w, dims, one)
                dt = time.perf_counter() - t0
            if b / dt > best[0]:
                best = (b / dt, cand, b)
        threads, batch = best[1], best[2]
        del w
        if target_seconds:  # bounded sample: as many AR frames per clip as fit the time budget at the calibrated rate
            steps = max(4, min(steps, int(round(target_seconds * best[0] / batch))))
    if procs == 1:
        import queue
        q = queue.Queue()
        _cpu_worker(0, threads, steps, warmup, q, batch)
        times = [m[2] for m in list(q.queue) if m[0] == "done"]
    else:
        import torch.multiprocessing as mp
        ctx = mp.get_context("spawn")
        q = ctx.Queue()
        ps = [ctx.Process(target=_cpu_worker, args=(i, threads, steps, warmup, q, batch)) for i in range(procs)]
        for p in ps:
            p.start()
        times = []
        for _ in range(2 * procs):
            msg = q.get(timeout=900)
            if msg[0] == "done":
                times.append(msg[2])
        for p in ps:
            p.join(60)
    slowest = max(times)
    desc = (f"{procs} replica(s) x {threads} threads x {batch} clip(s) per forward (thread count and batch calibrated on "
            f"this host; side-by-side replicas measured slower), {steps} AR frames per clip after {warmup} warm-up")
    return procs * batch * steps / slowest, slowest, procs * threads, desc


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    fps, total, threads, desc = cpu_frames_per_sec(args.steps, args.warmup)
    sample = (f"{desc} (bounded sample of the batch-{args.batch} workload), torch {__import__('torch').__version__} "
              f"fp32")
    line = {
        "impl": "reference", "metric": METRIC, "value": fps, "unit": "frames/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * total / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD, "batch_per_gpu": args.batch,
                   "note": "reference's TF-CPU path cannot run (TensorFlow absent); torch-CPU port of the same math, "
                           "independent clips over all host cores"},
        "cpu_baseline": {"value": fps, "unit": "frames/s", "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": fps, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# --------------------------------------------------------------------------------------------- kernel microbench
def time_kernel(fn, stream, iters=8, warm=3):
    import torch
    for _ in range(warm):
        fn()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    stream.synchronize()
    e0.record(stream)
    for _ in range(iters):
        fn()
    e1.record(stream)
    stream.synchronize()
    return e0.elapsed_time(e1) / iters * 1e-3  # seconds per launch


def kernel_rooflines(model, batch, mode, peaks, stream):
    """Time each hot kernel alone at the bench shapes (CUDA events on the launching stream; operands >> L2)."""
    import torch
    from mint_b200 import lib as L
    lib = L.load()
    d, ff, H = model.dims.cross_hidden, model.dims.cross_ff, model.dims.cross_heads
    n_seq = model.dims.cross_seq
    M = batch * n_seq
    dev = model.device
    precise = mode == "precise"
    bf = torch.bfloat16
    st = stream.cuda_stream

    def rnd(*shape):
        return (torch.randn(*shape, device=dev) * 0.05).to(bf)

    a_d = (rnd(M, d), rnd(M, d))
    a_ff = (rnd(M, ff), rnd(M, ff))
    x = torch.randn(M, d, device=dev)
    bias_ff, bias_d = torch.zeros(ff, device=dev), torch.zeros(d, device=dev)
    out_qkv = (torch.empty(M, 3 * d, dtype=bf, device=dev), torch.empty(M, 3 * d, dtype=bf, device=dev))
    out_ff = (torch.empty(M, ff, dtype=bf, device=dev), torch.empty(M, ff, dtype=bf, device=dev))
    out_d = (torch.empty(M, d, dtype=bf, device=dev), torch.empty(M, d, dtype=bf, device=dev))
    w = {"qkv": (rnd(3 * d, d), rnd(3 * d, d)), "o": (rnd(d, d), rnd(d, d)), "ff1": (rnd(ff, d), rnd(ff, d)),
         "ff2": (rnd(d, ff), rnd(d, ff))}
    lo = (lambda t: t[1].data_ptr()) if precise else (lambda t: None)

    def gemm(a, wt, m, n, k, epi):
        def run():
            L.check(lib.fact_gemm(a[0].data_ptr(), lo(a), k, wt[0].data_ptr(), lo(wt), k, m, n, k, C.byref(epi), st))
        return run

    e_qkv = L.GemmEpilogue(kind=L.EPI_SPLIT, out_hi=out_qkv[0].data_ptr(), out_lo=lo(out_qkv), ldo=3 * d, scale=0.05,
                           scale_cols=d)
    e_o = L.GemmEpilogue(kind=L.EPI_BIAS_RESID_F32, out_f32=x.data_ptr(), ldo=d, bias=bias_d.data_ptr(),
                         resid=x.data_ptr(), ldr=d)
    e_ff1 = L.GemmEpilogue(kind=L.EPI_BIAS_GELU_SPLIT, out_hi=out_ff[0].data_ptr(), out_lo=lo(out_ff), ldo=ff,
                           bias=bias_ff.data_ptr())
    e_ff2 = L.GemmEpilogue(kind=L.EPI_BIAS_RESID_F32, out_f32=x.data_ptr(), ldo=d, bias=bias_d.data_ptr(),
                           resid=x.data_ptr(), ldr=d)
    s_el = 4 if precise else 2   # bytes per activation element in split storage (hi+lo or hi)
    res = {}
    specs = [("gemm_qkv", gemm(a_d, w["qkv"], M, 3 * d, d, e_qkv), 2.0 * M * 3 * d * d),
             ("gemm_out", gemm(a_d, w["o"], M, d, d, e_o), 2.0 * M * d * d),
             ("gemm_ff1", gemm(a_d, w["ff1"], M, ff, d, e_ff1), 2.0 * M * ff * d),
             ("gemm_ff2", gemm(a_ff, w["ff2"], M, d, ff, e_ff2), 2.0 * M * d * ff)]
    # the residual GEMMs as the model calls them: LayerNorm of the finished rows inside the launch (LayerNorm warps)
    gam, bet = torch.ones(d, device=dev), torch.zeros(d, device=dev)
    ln_sync = torch.zeros(2 * (M // 32 + 2), dtype=torch.int32, device=dev)
    e_o_ln = L.GemmEpilogue(kind=L.EPI_BIAS_RESID_F32, out_f32=x.data_ptr(), ldo=d, bias=bias_d.data_ptr(),
                            resid=x.data_ptr(), ldr=d, ln_gamma=gam.data_ptr(), ln_beta=bet.data_ptr(),
                            ln_hi=out_d[0].data_ptr(), ln_lo=lo(out_d), ln_sync=ln_sync.data_ptr())
    specs += [("gemm_out_ln", gemm(a_d, w["o"], M, d, d, e_o_ln), 2.0 * M * d * d),
              ("gemm_ff2_ln", gemm(a_ff, w["ff2"], M, d, ff, e_o_ln), 2.0 * M * d * ff)]
    mult = 3.0 if precise else 1.0
    for name, fn, flops in specs:
        t = time_kernel(fn, stream)
        res[name] = {"s": t, "algo_tflops": flops / t / 1e12, "executed_tflops": mult * flops / t / 1e12}

    def sdpa():
        L.check(lib.fact_sdpa(out_qkv[0].data_ptr(), lo(out_qkv), out_d[0].data_ptr(), lo(out_d), batch, n_seq, H,
                              d // H, st))
    t = time_kernel(sdpa, stream)
    sdpa_bytes = 4.0 * M * d * s_el          # read q,k,v + write o (SURVEY.md 8d "SDPA core only")
    res["sdpa"] = {"s": t, "gbs": sdpa_bytes / t / 1e9, "algo_tflops": 3200.0 * n_seq * n_seq * batch / t / 1e12}

    def ln():
        L.check(lib.fact_layernorm_split(x.data_ptr(), bias_d.data_ptr(), bias_d.data_ptr(), out_d[0].data_ptr(),
                                         lo(out_d), M, d, st))
    t = time_kernel(ln, stream)
    res["layernorm_split"] = {"s": t, "gbs": (M * d * 4.0 + M * d * s_el) / t / 1e9}
    # fused attention block as the metric defines it (SURVEY.md 8d): x in + y out + weights, nothing else
    # LN + QKV + core + out-proj; the LayerNorm rides inside a residual GEMM launch when that is the faster pairing
    t_out_ln = min(res["gemm_out_ln"]["s"], res["layernorm_split"]["s"] + res["gemm_out"]["s"])
    t_blk = res["gemm_qkv"]["s"] + res["sdpa"]["s"] + t_out_ln
    blk_bytes = 1600.0 * batch * n_seq * 4 + 2562400.0 * s_el
    blk_flops = mult * (2.0 * M * 3 * d * d + 2.0 * M * d * d + 3200.0 * n_seq * n_seq * batch)
    blk_bytes_s2 = 1600.0 * batch * n_seq * 2 + 2562400.0 * 2
    res["attn_block"] = {"s": t_blk, "gbs": blk_bytes / t_blk / 1e9, "frac_hbm": blk_bytes / t_blk / 1e9 / peaks["hbm_gbs"],
                         "s_el": 4, "frac_hbm_s2": blk_bytes_s2 / t_blk / 1e9 / peaks["hbm_gbs"],
                         "executed_tflops": blk_flops / t_blk / 1e12}
    return res



# --------------------------------------------------------------------------------------------- training leg
TRAIN_FLOP_PER_CLIP = 3 * FLOP_PER_FRAME   # forward + backward (2x forward) of one clip, SURVEY.md 8(a) a14


def time_wgrad(model, batch, stream):
    """gemm_wgrad2_kernel alone at the FFN shape of a B-clip step: dW1[800, 3072] += ln2[M, 800]^T . dz[M, 3072]."""
    import torch
    from mint_b200 import lib as L
    lib = L.load()
    d, ff = model.dims.cross_hidden, model.dims.cross_ff
    M = batch * model.dims.cross_seq
    dev = model.device
    x = (torch.randn(M, d, device=dev) * 0.05).to(torch.bfloat16)
    dy = (torch.randn(M, ff, device=dev) * 0.05).to(torch.bfloat16)
    dw = torch.zeros(d, ff, device=dev)
    st = stream.cuda_stream

    def run():
        L.check(lib.fact_wgrad_gemm(x.data_ptr(), d, dy.data_ptr(), ff, dw.data_ptr(), ff, M, d, ff, st),
                "fact_wgrad_gemm")
    t = time_kernel(run, stream)
    return t, 2.0 * M * d * ff


def gpu_topology(world):
    """Link type between GPU0 and its peers as nvidia-smi reports it (NV18 = 18 NVLink-5 links through NVSwitch; PIX /
    PHB / SYS = PCIe): explains an all-reduce bandwidth that is far from the NVLink figure."""
    try:
        out = subprocess.run(["nvidia-smi", "topo", "-m"], capture_output=True, text=True, timeout=20).stdout
        rows = [ln.split() for ln in out.splitlines() if ln.startswith("GPU0")]
        return rows[0][1:1 + max(world, 1)] if rows else None
    except Exception:
        return None


def run_train_leg(args, cfg, dev, world, rank, local, peaks, stream, barrier, max_over_ranks):
    """BASELINE.json configs[2] (N=1) / configs[3] (N>1): one sync data-parallel training step per "step" --
    fact_train_step (forward with saved activations, L2 motion loss, full backward), ONE logical all-reduce of the
    flat fp32 gradient bucket (three slices, the first two overlapped with the backward), Keras Adam.
    Reference: mint/ctl/single_task_trainer.py:138-199, trainer.py:125-135."""
    import torch
    import torch.distributed as dist
    from mint_b200 import lib as L, model_builder, optim
    from mint_b200.trainer import SingleTaskTrainer

    B, K, Wm = args.train_batch, args.steps, max(args.warmup, 3)
    model = model_builder.build(cfg["model"], is_training=True, device=dev, mode="bf16", seed=0)
    d = model.dims
    opt = optim.Adam(model, learning_rate=optim.learning_rate_from_config(cfg["train_config"]))
    g = torch.Generator(device="cpu").manual_seed(1000 + rank)
    host = {"motion_input": (0.5 * torch.randn(B, d.motion.seq_len, d.motion.feature_dim, generator=g)).pin_memory(),
            "audio_input": torch.randn(B, d.audio.seq_len, d.audio.feature_dim, generator=g).pin_memory(),
            "target": (0.5 * torch.randn(B, 20, d.out_dim, generator=g)).pin_memory()}
    out = {"config": {"workload": "fact_v5_deeper_t10_cm12 training step", "batch_per_gpu": B,
                      "global_batch": B * world, "products": "bf16 (fp32 accumulate, fp32 master weights / Adam state)",
                      "loss": "L2 motion loss on the first 20 frames", "optimizer": "Keras Adam",
                      "parallelism": f"dp{world}: one logical all-reduce of the flat fp32 gradient bucket per step, "
                                     "see allreduce_overlap: 'fused' = no all-reduce, ONE kernel sums the replicas' "
                                     "gradients over NVLink peer memory, applies Adam to this rank's shard and stores "
                                     "the new weights into every replica, launched per slice of the bucket under the "
                                     "backward ('fused_tail': once, after it); 'adam' / 'backward' / 'none' = NCCL "
                                     "all-reduce in slices hidden behind the optimizer pass / the backward / not at all"
                                     if world > 1 else "single GPU"}}
    with torch.cuda.stream(stream):
        batch_d = {k: v.to(dev, non_blocking=True) for k, v in host.items()}
        dp = SingleTaskTrainer([], "target", model, optimizer=opt, overlap=args.dp_overlap)
        local_only = SingleTaskTrainer([], "target", model, optimizer=opt, allreduce=False)
        losses = [dp.train_step(batch_d) for _ in range(Wm)]
        first_loss = float(losses[0])
        barrier()

        def timed(fn, steps):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            barrier()
            t0 = time.perf_counter()
            e0.record(stream)
            for _ in range(steps):
                last = fn()
            e1.record(stream)
            barrier()
            return max_over_ranks(e0.elapsed_time(e1)) / steps, t0, time.perf_counter(), last

        sampler = ClockSampler(local)
        if rank == 0:
            sampler.start()
            time.sleep(0.3)
        launches0 = L.load().fact_launch_count()
        ms, t0, t1, last = timed(lambda: dp.train_step(batch_d), K)
        launches = L.load().fact_launch_count() - launches0
        clocks = sampler.stop(t0, t1) if rank == 0 else None
        ar_ms = exposed = ms_local = ms_sync = None
        modes = None
        if world > 1:
            # Decomposition, all in this process on the same clocks: free-running replicas (no cross-replica op),
            # replicas that only MEET once per step (4-byte all-reduce: pure synchronisation skew -- power-capped GPUs
            # do not run at one clock), and every way of moving the gradients this box supports.
            synced = SingleTaskTrainer([], "target", model, optimizer=opt, allreduce=False, sync_only=True)
            ms_local, _, _, _ = timed(lambda: local_only.train_step(batch_d), K)
            # clocks drift while the GPU warms up under its power cap, so every mode is bracketed by two runs of the
            # meet-only step and compared with their mean
            modes = {}
            sync_runs = [timed(lambda: synced.train_step(batch_d), K)[0]]
            for mode in (["fused", "fused_tail"] if dp.arena is not None else []) + ["none", "adam", "backward"]:
                tr = dp if mode == dp.overlap else SingleTaskTrainer([], "target", model, optimizer=opt, overlap=mode,
                                                                      arena=dp.arena if mode.startswith("fused") else None)
                for _ in range(2):
                    tr.train_step(batch_d)
                m_ms, _, _, _ = timed(lambda: tr.train_step(batch_d), K)
                sync_runs.append(timed(lambda: synced.train_step(batch_d), K)[0])
                ref = 0.5 * (sync_runs[-2] + sync_runs[-1])
                modes[mode] = {"ms_per_step": m_ms, "meet_only_ms_per_step": ref, "exposed_ms": m_ms - ref}
            ms_sync = sum(sync_runs) / len(sync_runs)
            ms = modes[dp.overlap]["ms_per_step"]
            exposed = modes[dp.overlap]["exposed_ms"]
            grads = model.flat_gradients

            def ar():
                dist.all_reduce(grads)
            ar_ms, _, _, _ = timed(ar, 5)
        # end to end: pinned host batch -> device inside the step, loss read back to pinned host memory every step
        loss_host = torch.empty(K, dtype=torch.float32).pin_memory()
        step_i = [0]

        def e2e_step():
            bd = {k: v.to(dev, non_blocking=True) for k, v in host.items()}
            loss = dp.train_step(bd)
            loss_host[step_i[0] % K].copy_(loss, non_blocking=True)
            step_i[0] += 1
            return loss
        e2e_step()
        barrier()
        tw0 = time.perf_counter()
        for _ in range(K):
            e2e_step()
        torch.cuda.synchronize(dev)
        e2e_ms = max_over_ranks((time.perf_counter() - tw0) * 1e3) / K
        barrier()
        assert torch.isfinite(loss_host).all(), "non-finite training loss"
        wg = None
        if rank == 0:
            try:
                t_w, fl = time_wgrad(model, B, stream)
                wg = {"bound": "tensor", "kernel": f"gemm_wgrad2_kernel (dW1: tokens={B * d.cross_seq}, 800x3072, "
                                                   "tcgen05 cta_group::2, MN-major operands)",
                      "achieved": fl / t_w / 1e12, "peak": peaks["bf16_tflops"], "unit": "TFLOP/s",
                      "frac": fl / t_w / 1e12 / peaks["bf16_tflops"], "us_per_launch": t_w * 1e6,
                      "peak_source": peaks["source"] + " (burst: kernel timed alone)"}
            except Exception as exc:
                wg = {"error": repr(exc)[:300]}
    h2d = sum(v.numel() for v in host.values()) * 4
    out.update({
        "ms_per_step": ms, "samples_per_s": world * B * 1e3 / ms, "steps": K, "warmup": Wm,
        "algorithmic_tflops_per_gpu": TRAIN_FLOP_PER_CLIP * B / (ms * 1e-3) / 1e12,
        "frac_of_sustained_tensor_peak": TRAIN_FLOP_PER_CLIP * B / (ms * 1e-3) / 1e12 / peaks["bf16_tflops_sustained"],
        "allreduce_ms": ar_ms, "exposed_allreduce_ms": exposed, "ms_per_step_without_allreduce": ms_sync,
        "ms_per_step_free_running": ms_local,
        "sync_skew_ms": (ms_sync - ms_local) if ms_sync is not None else None,
        "modes": modes,
        "exposed_note": ("exposed_allreduce_ms = data-parallel step - step in which the replicas only meet (4-byte "
                         "all-reduce); sync_skew_ms = that step - free-running replicas (max over ranks of the mean): "
                         "the price of lock step under per-GPU power caps, paid by any synchronous scheme") if world > 1
        else None,
        "grad_bucket_mb": model.flat_gradients.numel() * 4 / 1e6,
        "allreduce_overlap": dp.overlap if world > 1 else None,
        "allreduce_calibration_ms": dp.calibration_ms,
        "fused_step": ({"kernel": "dp_adam_kernel (gradient sum + Adam + weight broadcast over peer memory)",
                        "multicast": dp.arena.mc_ptr is not None, "arena_mb": dp.arena.nbytes / 1e6,
                        "slices_mb": [round(c * 4 / 1e6, 1) for _, c, _ in dp._plan] if dp._plan else None}
                       if dp.arena is not None else {"unavailable": dp.fused_error}) if world > 1 else None,
        "allreduce_slices_mb": ([round(c * 4 / 1e6, 1) for _, c, _ in dp._plan] if dp._plan else
                                [round(c * 4 / 1e6, 1) for _, c in dp.even_slices()])
        if world > 1 and not dp.overlap.startswith("fused") else None,
        "allreduce_busbw_gbs": (model.flat_gradients.numel() * 4 * 2 * (world - 1) / world / (ar_ms * 1e-3) / 1e9
                                if ar_ms else None),
        "gpu_topology": gpu_topology(world) if rank == 0 else None,
        "e2e": {"ms_per_step": e2e_ms, "samples_per_s": world * B * 1e3 / e2e_ms, "h2d_bytes_per_step": h2d,
                "d2h_bytes_per_step": 4},
        "gpu_launches_per_step": int(launches) // K, "loss_first": first_loss, "loss_last": float(last),
        "peak_mem_gb": torch.cuda.max_memory_allocated(dev) / 1e9, "roofline": wg, "clocks": clocks,
        "scaling": "weak"})
    del dp, local_only, opt, model
    torch.cuda.empty_cache()
    return out


def run_sweep_leg(args, model, dev, world, rank, stream, barrier, max_over_ranks, peaks):
    """BASELINE.json configs[4]: AR frames/s at B clips per GPU, B = 1 .. 512, every rank generating its own clips
    (weak scaling, no data-path collective); the attention core's HBM fraction per point on rank 0."""
    import torch
    from mint_b200 import lib as L
    lib = L.load()
    dims = model.dims
    H, d, ns = dims.cross_heads, dims.cross_hidden, dims.cross_seq
    precise = model.mode == "precise"
    pts = []
    for B in [int(v) for v in args.sweep.split(",") if v]:
        k = args.steps
        w = 3
        T = dims.audio.seq_len + w + k - 1
        motion = 0.5 * torch.randn(B, dims.motion.seq_len, dims.motion.feature_dim, device=dev)
        motion[..., :6] = 0
        audio = torch.randn(B, T, dims.audio.feature_dim, device=dev)
        hist = model.new_history(motion, w + k)
        model.generate_into(hist, audio, 0, w)
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        model.generate_into(hist, audio, w, k)
        e1.record(stream)
        barrier()
        ms = max_over_ranks(e0.elapsed_time(e1)) / k
        pt = {"batch_per_gpu": B, "frames_per_s": world * B * 1e3 / ms, "ms_per_step": ms, "frames_timed": k}
        if rank == 0:
            M = B * ns
            qkv = [(torch.randn(M, 3 * d, device=dev) * 0.05).to(torch.bfloat16) for _ in range(2 if precise else 1)]
            ao = [torch.empty(M, d, dtype=torch.bfloat16, device=dev) for _ in range(2 if precise else 1)]

            def sdpa():
                L.check(lib.fact_sdpa(qkv[0].data_ptr(), qkv[-1].data_ptr() if precise else None, ao[0].data_ptr(),
                                      ao[-1].data_ptr() if precise else None, B, ns, H, d // H, stream.cuda_stream))
            t = time_kernel(sdpa, stream, iters=4, warm=2)
            byts = 4.0 * M * d * (4 if precise else 2)
            pt["sdpa_core_gbs"] = byts / t / 1e9
            pt["sdpa_core_frac_hbm"] = byts / t / 1e9 / peaks["hbm_gbs"]
            del qkv, ao
        pts.append(pt)
        del hist, audio, motion
    return pts

# --------------------------------------------------------------------------------------------- our arm
def run_ours(args):
    import torch
    import torch.distributed as dist
    from mint_b200 import config_util, model_builder

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py --impl ours needs a GPU (no CPU fallback)"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    peaks = load_peaks()
    if args.flag:
        from mint_b200 import lib as _L
        for kv in args.flag:
            name, val = kv.split("=")
            _L.check(_L.load().fact_set_flag(name.encode(), int(val)), "fact_set_flag")

    cfg = config_util.get_configs_from_pipeline_file(config_util.DEFAULT_CONFIG)
    model = model_builder.build(cfg["model"], is_training=False, device=dev, mode=args.mode, seed=rank)
    dims = model.dims
    B, K, Wm = args.batch, args.steps, max(args.warmup, 3)
    gen = torch.Generator(device="cpu").manual_seed(100 + rank)
    T = dims.audio.seq_len + Wm + K - 1
    motion_h = (0.5 * torch.randn(B, dims.motion.seq_len, dims.motion.feature_dim, generator=gen)).pin_memory()
    motion_h[..., :6] = 0
    audio_h = torch.randn(B, T, dims.audio.feature_dim, generator=gen).pin_memory()

    stream = torch.cuda.Stream(dev)
    if args.kernels_only:
        with torch.cuda.stream(stream):
            kr = kernel_rooflines(model, args.batch, args.mode, peaks, stream)
        for k, v in kr.items():
            print(k, {kk: round(vv, 6) for kk, vv in v.items()})
        with torch.cuda.stream(stream):
            t_w, fl = time_wgrad(model, args.batch, stream)
        print("wgrad_ff", {"s": round(t_w, 6), "tflops": round(fl / t_w / 1e12, 1)})
        return

    def barrier():
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def max_over_ranks(v):
        if world == 1:
            return v
        t = torch.tensor([v], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---- device-resident leg: W warm-up frames, then exactly K timed frames on the same captured graph
    with torch.cuda.stream(stream):
        motion_d = motion_h.to(dev, non_blocking=True)
        audio_d = audio_h.to(dev, non_blocking=True)
        hist = model.new_history(motion_d, Wm + K)
        model.generate_into(hist, audio_d, 0, Wm)
        barrier()
        sampler = ClockSampler(local)
        if rank == 0:
            sampler.start()
            time.sleep(0.3)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        from mint_b200 import lib as _lib
        launches0 = _lib.load().fact_launch_count()
        t_wall0 = time.perf_counter()
        e0.record(stream)
        model.generate_into(hist, audio_d, Wm, K)
        e1.record(stream)
        launches = _lib.load().fact_launch_count() - launches0
        barrier()
        t_wall1 = time.perf_counter()
        ms = max_over_ranks(e0.elapsed_time(e1))
        clocks = sampler.stop(t_wall0, t_wall1) if rank == 0 else None
        assert torch.isfinite(hist).all(), "non-finite frames generated"
        if args.dump_outputs and rank == 0:
            dump_outputs(args.dump_outputs, "last_frame", hist[:, -1])

        # ---- end-to-end leg: public API, pinned host inputs -> host result, copies inside the timed region
        audio_e2e = audio_h[:, :dims.audio.seq_len + K - 1].contiguous().pin_memory()
        inputs = {"motion_input": motion_h, "audio_input": audio_e2e}
        out_host = torch.empty(B, K, dims.out_dim).pin_memory()
        model.infer_auto_regressive(inputs, steps=K)   # untimed: graph capture for this history shape
        barrier()
        t0 = time.perf_counter()
        frames = model.infer_auto_regressive(inputs, steps=K)
        out_host.copy_(frames, non_blocking=True)
        torch.cuda.synchronize(dev)
        e2e_s = max_over_ranks(time.perf_counter() - t0)
        barrier()
        h2d = (motion_h.numel() + audio_e2e.numel()) * 4 / K
        d2h = out_host.numel() * 4 / K

        extras = {}
        if rank == 0 and not args.no_extras and world == 1:
          try:
            # BASELINE.json configs[1]: ONE clip, 1200 frames (20 s at 60 fps), T = 1439 audio frames, same model / mode.
            # Device-resident leg (frames appended to a resident history) and the public-API leg
            # (FACTModel.infer_auto_regressive: pinned host inputs -> host frames, copies inside the timed region).
            n1 = max(8, args.b1_frames)
            g1 = torch.Generator(device="cpu").manual_seed(7)
            m1_h = motion_h[:1].clone().pin_memory()
            a1_h = torch.randn(1, dims.audio.seq_len + n1 - 1, dims.audio.feature_dim, generator=g1).pin_memory()
            m1, a1w = m1_h.to(dev), a1_h.to(dev)
            h1 = model.new_history(m1, n1 + Wm)
            a1pad = torch.cat([a1w, torch.randn(1, Wm, dims.audio.feature_dim, device=dev)], dim=1)
            model.generate_into(h1, a1pad, 0, Wm)
            stream.synchronize()
            f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            f0.record(stream)
            model.generate_into(h1, a1pad, Wm, n1)
            f1.record(stream)
            stream.synchronize()
            ms1 = f0.elapsed_time(f1) / n1
            model.infer_auto_regressive({"motion_input": m1_h, "audio_input": a1_h}, steps=8)   # untimed warm-up
            stream.synchronize()
            out1 = torch.empty(1, n1, dims.out_dim).pin_memory()
            tb = time.perf_counter()
            fr1 = model.infer_auto_regressive({"motion_input": m1_h, "audio_input": a1_h}, steps=n1)
            out1.copy_(fr1, non_blocking=True)
            torch.cuda.synchronize(dev)
            e2e1 = time.perf_counter() - tb
            assert tuple(fr1.shape) == (1, n1, dims.out_dim) and torch.isfinite(out1).all()
            extras["batch1"] = {"value": 1e3 / ms1, "unit": "frames/s", "ms_per_frame": ms1, "frames": n1,
                                "audio_len": int(a1_h.shape[1]),
                                "e2e": {"value": n1 / e2e1, "unit": "frames/s", "seconds_per_clip": e2e1,
                                        "h2d_bytes": (m1_h.numel() + a1_h.numel()) * 4, "d2h_bytes": out1.numel() * 4},
                                "note": "configs[1]: single clip, 1200 frames; latency-bound small-M launch chain"}
            del h1, a1pad
          except Exception as exc:  # an extra must never cost the headline line
            extras["batch1"] = {"error": repr(exc)[:300]}
        if rank == 0 and not args.no_extras:
          try:
            kr = kernel_rooflines(model, B, args.mode, peaks, stream)
            extras["kernels"] = {k: {kk: (round(vv, 6) if isinstance(vv, float) else vv) for kk, vv in v.items()}
                                 for k, v in kr.items()}
            # per-frame launch counts of each GEMM at the cross-modal shape (encoder shapes are smaller)
            dom = max(("gemm_qkv", "gemm_out", "gemm_ff1", "gemm_ff2"), key=lambda k: kr[k]["s"])
            traffic = None
            tpath = os.path.join(ROOT, "profiles", "r2_dram_traffic.json")
            if not os.path.exists(tpath):
                tpath = os.path.join(ROOT, "profiles", "r1_dram_traffic.json")
            if args.mode == "precise" and B == 128 and os.path.exists(tpath):
                with open(tpath) as f:
                    traffic = json.load(f).get(dom)
            extras["roofline"] = {
                "bound": "tensor", "kernel": f"gemm_tc2_kernel ({dom}, M={B * dims.cross_seq}, tcgen05 cta_group::2)",
                "achieved": kr[dom]["executed_tflops"], "peak": peaks["bf16_tflops"], "unit": "TFLOP/s",
                "frac": kr[dom]["executed_tflops"] / peaks["bf16_tflops"], "traffic": traffic,
                "traffic_source": (os.path.relpath(tpath, ROOT) + " (ncu --set full dram__bytes_read+write per launch, "
                                   "committed; not re-measured in this run)") if traffic is not None else None,
                "frac_of_sustained_peak": kr[dom]["executed_tflops"] / peaks["bf16_tflops_sustained"],
                "peak_source": peaks["source"] + " (burst: kernel timed alone)",
                "algorithmic_tflops": kr[dom]["algo_tflops"],
                "note": ("executed = bf16 tensor FLOPs issued (3 MMAs per product in precise mode); "
                         "algorithmic = 2*M*N*K of the fp32-grade product") if args.mode == "precise" else "bf16",
            }
            extras["attn_roofline"] = {
                "bound": "hbm", "kernel": "attention block = gemm_tc2_kernel (QKV), sdpa_tc_kernel, gemm_tc2_kernel (out-proj + bias + residual, LayerNorm of the finished rows by the kernel's own LayerNorm warps)",
                "achieved": kr["attn_block"]["gbs"], "peak": peaks["hbm_gbs"], "unit": "GB/s",
                "frac": kr["attn_block"]["frac_hbm"],
                "sdpa_core_gbs": kr["sdpa"]["gbs"], "sdpa_core_frac": kr["sdpa"]["gbs"] / peaks["hbm_gbs"],
                "bytes_per_element": kr["attn_block"]["s_el"],
                "frac_at_2_bytes_per_element": kr["attn_block"]["frac_hbm_s2"],
                "tensor_tflops_executed": kr["attn_block"]["executed_tflops"],
                "tensor_frac": kr["attn_block"]["executed_tflops"] / peaks["bf16_tflops"],
                "note": ("BASELINE's metric for the attention block: bytes = 1600*B*N*s + 2562400*s (SURVEY.md 8d: x in, y "
                         "out, weights once), s = bytes_per_element (4 = fp32 residual stream / bf16 hi+lo operands; the "
                         "survey's bf16 figure s = 2 is given beside it). The block executes 289 GFLOP algorithmic "
                         "(x3 products in precise mode) per launch, i.e. it is tensor-bound by >9x: tensor_frac is the "
                         "number that says how good the block is, the HBM fraction cannot approach 0.7 by construction"),
            }
          except Exception as exc:
            extras["roofline"] = {"error": repr(exc)[:300]}
        sweep = None
        if not args.no_extras and not args.no_sweep:
            try:
                sweep = run_sweep_leg(args, model, dev, world, rank, stream, barrier, max_over_ranks, peaks)
            except Exception as exc:
                if world > 1:
                    raise                     # ranks must stay in lock step
                sweep = {"error": repr(exc)[:300]}
    fps = world * B * K / (ms * 1e-3)
    e2e_fps = world * B * K / e2e_s
    train = None
    if not args.no_extras and not args.no_train:
        try:
            train = run_train_leg(args, cfg, dev, world, rank, local, peaks, stream, barrier, max_over_ranks)
        except Exception as exc:
            if world > 1:
                raise
            train = {"error": repr(exc)[:300]}

    line = None
    if rank == 0:
        line = {
            "metric": METRIC, "value": fps, "unit": "frames/s", "n_gpus": world, "steps": K, "warmup": Wm,
            "warmup_requested": args.warmup,     # fewer than 3 requested warm-up steps are raised to 3
            "ms_per_step": ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "bf16x3 (fp32-grade split products, fp32 accumulate)" if args.mode == "precise" else "bf16",
            "data": "synthetic",
            "config": {"workload": WORKLOAD, "batch_per_gpu": B, "global_batch": world * B,
                       "motion_seq": dims.motion.seq_len, "audio_seq": dims.audio.seq_len, "mode": args.mode,
                       "parallelism": f"replicas{world} (independent clips per GPU, no data-path collective)",
                       "l2": "per-frame working set (>1 GB activations + 0.5 GB weights) exceeds the 126 MB L2",
                       "flop_per_frame": FLOP_PER_FRAME},
            "achieved_algorithmic_tflops_per_gpu": fps / world * FLOP_PER_FRAME / 1e12,
            "clocks": clocks,
            "e2e": {"value": e2e_fps, "unit": "frames/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h},
            "gpu_launches": int(launches),
        }
        line.update(extras)
        if sweep is not None:
            line["batch_sweep"] = {"unit": "frames/s (all GPUs)", "n_gpus": world, "mode": args.mode, "points": sweep,
                                   "note": "configs[4]: B clips per GPU, device-resident, 3 warm-up frames then "
                                           "frames_timed frames on the captured graph; max over ranks"}
        if train is not None:
            line["train"] = train
        if world == 1 and not args.no_extras and not args.no_cpu:
            try:
                cpu_fps, cpu_total, threads, desc = cpu_frames_per_sec(args.cpu_frames, 2, target_seconds=12.0)
                line["cpu_baseline"] = {
                    "value": cpu_fps, "unit": "frames/s", "cores": threads, "kind": "port",
                    "sample": f"{desc}; torch-CPU fp32 restatement (TensorFlow absent), {cpu_total:.1f} s"}
            except Exception as exc:
                line["cpu_baseline"] = {"error": repr(exc)[:300]}
    # throughput-mode leg (single bf16 products), reported beside the parity-grade headline
    if args.mode == "precise" and not args.no_extras and world == 1:
      try:
        del model, hist
        torch.cuda.empty_cache()
        m2 = model_builder.build(cfg["model"], is_training=False, device=dev, mode="bf16", seed=rank)
        with torch.cuda.stream(stream):
            h2 = m2.new_history(motion_d, Wm + K)
            m2.generate_into(h2, audio_d, 0, Wm)
            barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            m2.generate_into(h2, audio_d, Wm, K)
            e1.record(stream)
            barrier()
            ms2 = e0.elapsed_time(e1)
        if rank == 0:
            line["fast_bf16"] = {"value": B * K / (ms2 * 1e-3), "unit": "frames/s", "ms_per_step": ms2 / K,
                                 "note": "single bf16 products: ~4e-2 per-joint L2 vs fp64 on random-init weights; "
                                         "outside the 1e-3 parity bar, reported for throughput only"}
      except Exception as exc:
        if rank == 0:
            line["fast_bf16"] = {"error": repr(exc)[:300]}
    if rank == 0:
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    args = parse()
    # stdout carries the ONE JSON line and nothing else: libraries that print to fd 1 (NCCL's version banner ...) go to
    # stderr for the duration of the run
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    sys.stdout = os.fdopen(real_stdout, "w", buffering=1)
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)
    sys.stdout.flush()


if __name__ == "__main__":
    main()
