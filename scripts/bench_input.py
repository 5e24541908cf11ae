#!/usr/bin/env python
"""Training input on one GPU: host-side TFRecord decoding (inputs.create_input) against the device-resident dataset
(device_inputs.create_device_input), on seeded synthetic TFRecords of realistic lengths.  Prints one JSON line:

  decode_ms_per_record        parse_example as it was (np.asarray over protobuf's float lists) and as it is
  create_input_ms_per_batch   steady state (shuffle buffer full), per batch size
  gather_us_per_call          fact_gather_windows alone, CUDA events over many launches, per batch size
  train_steps_per_s           full FACT v5 bf16 training steps fed by synthetic device tensors, by create_input and by
                              create_device_input; the three feeds alternate in rounds after a warm-up of each, and
                              the median, min and max over the rounds are reported, per batch size
  gpu, power_limit_w          read in the same run

    python scripts/bench_input.py [--records 200] [--batches 32,128] [--steps 10] [--rounds 3] [--out FILE]

Everything it writes (the TFRecords) goes to a temporary directory.
"""
import argparse
import glob
import json
import os
import subprocess
import sys
import tempfile
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402
import torch  # noqa: E402

from mint_b200 import config_util, device_inputs, inputs, model_builder, optim  # noqa: E402
from mint_b200 import lib as L  # noqa: E402
from mint_b200.trainer import SingleTaskTrainer  # noqa: E402


def write_records(root, n, lo, hi, seed, files=4):
    """n records of T ~ U[lo, hi] frames (motion [T, 219], audio [T, 35]) over `files` files; returns the glob."""
    rng = np.random.default_rng(seed)
    writers = [inputs.TFRecordWriter(os.path.join(root, f"b_tfrecord-train-{i:05d}")) for i in range(files)]
    for i in range(n):
        t = int(rng.integers(lo, hi + 1))
        ex = inputs.to_tfexample((0.5 * rng.standard_normal((t, 219))).astype(np.float32),
                                 rng.standard_normal((t, 35)).astype(np.float32), f"gBR_sBM_c{i:04d}", f"mBR{i}")
        writers[i % files].write(ex.SerializeToString())
    for w in writers:
        w.close()
    return os.path.join(root, "b_tfrecord-train-*")


def list_decode(record: bytes) -> dict:
    """parse_example before the packed-bytes decoding: np.asarray over protobuf's repeated-float containers."""
    f = inputs.Example.FromString(record).features.feature
    out = {}
    for modality in ("motion", "audio"):
        shape = tuple(int(v) for v in f[f"{modality}_sequence_shape"].int64_list.value)
        out[f"{modality}_sequence"] = np.asarray(f[f"{modality}_sequence"].float_list.value, np.float32).reshape(shape)
        out[f"{modality}_sequence_shape"] = np.asarray(shape, np.int32)
        out[f"{modality}_name"] = bytes(f[f"{modality}_name"].bytes_list.value[0])
    return out


def gpu_identity(dev):
    name = torch.cuda.get_device_name(dev)
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader,nounits", "-i",
                              str(dev.index or 0)], capture_output=True, text=True, timeout=20).stdout.strip()
        power = float(out.splitlines()[0])
    except (OSError, ValueError, IndexError, subprocess.SubprocessError):
        power = None
    return name, power


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--records", type=int, default=200)
    ap.add_argument("--min-frames", type=int, default=600)
    ap.add_argument("--max-frames", type=int, default=3000)
    ap.add_argument("--decode-records", type=int, default=12)
    ap.add_argument("--host-batches", type=int, default=3)
    ap.add_argument("--gather-iters", type=int, default=500)
    ap.add_argument("--batches", default="32,128")
    ap.add_argument("--steps", type=int, default=10, help="timed training steps per feed and round")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--out", default="", help="also write the JSON line to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_input.py measures on a GPU and found none")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    batches = [int(b) for b in args.batches.split(",")]
    res = {"metric": "training input: host decoding vs device-resident dataset",
           "config": "fact_v5_deeper_t10_cm12, bf16 products, L2 loss, Keras Adam", "records": args.records,
           "frames": [args.min_frames, args.max_frames]}
    res["gpu"], res["power_limit_w"] = gpu_identity(dev)
    res["host_cpus"] = os.cpu_count()
    with tempfile.TemporaryDirectory() as root:
        files = write_records(root, args.records, args.min_frames, args.max_frames, args.seed)
        recs = []
        for path in sorted(glob.glob(files)):
            for r in inputs.read_tfrecords(path):
                recs.append(r)
                if len(recs) == args.decode_records:
                    break
            if len(recs) == args.decode_records:
                break
        for fn in (list_decode, inputs.parse_example):                  # warm both, check they agree
            a, b = list_decode(recs[0]), fn(recs[0])
            assert all(np.array_equal(a[k], b[k]) for k in a)
        timing = {}
        for label, fn in (("old", list_decode), ("new", inputs.parse_example)):
            t0 = time.perf_counter()
            for r in recs:
                fn(r)
            timing[label] = (time.perf_counter() - t0) * 1e3 / len(recs)
        res["decode_ms_per_record"] = timing
        res["record_mb_mean"] = sum(map(len, recs)) / len(recs) / 1e6

        cfgs = {B: config_util.get_configs_from_pipeline_file(
            config_util.DEFAULT_CONFIG, 'train_dataset { data_files: "%s" } train_config { batch_size: %d }'
            % (files, B)) for B in batches}
        res["create_input_ms_per_batch"] = {}
        for B in batches:
            it = inputs.create_input(cfgs[B]["train_config"], cfgs[B]["train_dataset"], is_training=True, seed=0)
            for _ in range(2):                                               # fills the shuffle buffer
                next(it)
            t0 = time.perf_counter()
            for _ in range(args.host_batches):
                next(it)
            res["create_input_ms_per_batch"][str(B)] = (time.perf_counter() - t0) * 1e3 / args.host_batches

        # ---------------------------------------------------------------------------------------- device side
        lib = L.load()
        model = model_builder.build(cfgs[batches[0]]["model"], True, device=dev, mode="bf16", seed=0)
        opt = optim.Adam(model, learning_rate=1e-4)
        d = model.dims
        keys = ("motion_input", "audio_input", "target")
        res["gather_us_per_call"], res["train_steps_per_s"], res["construct_s"] = {}, {}, {}
        res["device_batch_equals_host"] = {}
        for B in batches:
            c = cfgs[B]
            t0 = time.perf_counter()
            dev_feed = device_inputs.create_device_input(c["train_config"], c["train_dataset"], dev, seed=0)
            res["construct_s"][str(B)] = time.perf_counter() - t0
            # the device producer's first batch against create_input's (same seed)
            want = next(inputs.create_input(c["train_config"], c["train_dataset"], is_training=True, seed=0))
            got = next(dev_feed)
            res["device_batch_equals_host"][str(B)] = all(
                torch.equal(got[k].cpu(), torch.from_numpy(want[k])) for k in keys)
            host_feed = inputs.create_input(c["train_config"], c["train_dataset"], is_training=True, seed=0)
            g = torch.Generator(device="cpu").manual_seed(B)
            synth = {"motion_input": (0.5 * torch.randn(B, d.motion.seq_len, d.motion.feature_dim, generator=g)).to(dev),
                     "audio_input": torch.randn(B, d.audio.seq_len, d.audio.feature_dim, generator=g).to(dev),
                     "target": (0.5 * torch.randn(B, 20, d.out_dim, generator=g)).to(dev)}

            # fact_gather_windows alone, into preallocated outputs
            p = dev_feed.plan
            rows = torch.from_numpy(p.rows(1)[0]).to(dev)
            outs = [torch.empty(B, p.motion_len, 225, device=dev), torch.empty(B, p.target_len, 225, device=dev),
                    torch.empty(B, p.audio_len, 35, device=dev)]
            st = torch.cuda.current_stream(dev).cuda_stream

            def gather():
                L.check(lib.fact_gather_windows(dev_feed.motion.data_ptr(), 225, dev_feed.audio.data_ptr(), 35,
                                                rows[0].data_ptr(), rows[1].data_ptr(), B, p.motion_len,
                                                p.target_shift, p.target_len, p.audio_len,
                                                *(o.data_ptr() for o in outs), st), "fact_gather_windows")
            for _ in range(20):
                gather()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(args.gather_iters):
                gather()
            e1.record()
            torch.cuda.synchronize(dev)
            res["gather_us_per_call"][str(B)] = e0.elapsed_time(e1) * 1e3 / args.gather_iters
            res.setdefault("gather_mb_per_call", {})[str(B)] = sum(o.numel() for o in outs) * 4 * 2 / 1e6  # read+write

            feeds = {"synthetic": lambda: synth,
                     "create_input": lambda: {k: v for k, v in next(host_feed).items() if k in keys},
                     "create_device_input": lambda: {k: v for k, v in next(dev_feed).items() if k in keys}}
            trainer = SingleTaskTrainer([], "target", model, optimizer=opt)
            rates = {k: [] for k in feeds}
            with torch.cuda.stream(torch.cuda.Stream(dev)):                   # as trainer.py runs the loop
                for name, feed in feeds.items():
                    for _ in range(args.warmup):
                        trainer.train_step(feed())
                torch.cuda.synchronize(dev)
                for _ in range(args.rounds):
                    for name, feed in feeds.items():
                        torch.cuda.synchronize(dev)
                        t0 = time.perf_counter()
                        for _ in range(args.steps):
                            loss = trainer.train_step(feed())
                        torch.cuda.synchronize(dev)
                        rates[name].append(args.steps / (time.perf_counter() - t0))
                        assert np.isfinite(float(loss))
            res["train_steps_per_s"][str(B)] = {
                k: {"median": float(np.median(v)), "min": min(v), "max": max(v)} for k, v in rates.items()}
            del dev_feed, host_feed
            torch.cuda.empty_cache()
    res["peak_mem_gb"] = torch.cuda.max_memory_allocated(dev) / 1e9
    line = json.dumps(res)
    print(line, flush=True)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
