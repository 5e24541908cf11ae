#!/usr/bin/env python
"""Train FACT on B200 -- flag-compatible counterpart of the reference's trainer.py (trainer.py:27-46, 138-178).

    python trainer.py --config_path configs/fact_v5_deeper_t10_cm12.config --model_dir /tmp/fact --steps 100
    python -m torch.distributed.run --nproc-per-node 8 --master-addr 127.0.0.1 trainer.py ...   (sync data parallel)

Data: the TFRecords named by train_dataset.data_files of the config (the reference's own format, read without
TensorFlow by mint_b200/inputs.py, decoded once into GPU memory by mint_b200/device_inputs.py) when that glob matches
files; else --data_npz arrays {motion_input, audio_input,
target}; else the synthetic generator of SURVEY.md 8d.
"""
import argparse
import json
import os

import numpy as np
import torch
import torch.distributed as dist

import glob

from mint_b200 import config_util, device_inputs, model_builder, optim
from mint_b200.trainer import SingleTaskTrainer


def synthetic_batches(dims, batch_size, seed):
    g = torch.Generator(device="cpu").manual_seed(seed)
    while True:
        motion = 0.5 * torch.randn(batch_size, dims.motion.seq_len, dims.motion.feature_dim, generator=g)
        motion[..., :6] = 0
        target = 0.5 * torch.randn(batch_size, 20, dims.out_dim, generator=g)
        target[..., :6] = 0
        yield {"motion_input": motion, "audio_input": torch.randn(batch_size, dims.audio.seq_len,
                                                                   dims.audio.feature_dim, generator=g),
               "target": target}


def npz_batches(path, batch_size, seed):
    data = np.load(path)
    n = data["motion_input"].shape[0]
    rng = np.random.default_rng(seed)
    while True:
        idx = rng.integers(0, n, batch_size)
        yield {k: torch.from_numpy(data[k][idx]).float() for k in ("motion_input", "audio_input", "target")}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--config_path", default=config_util.DEFAULT_CONFIG)
    ap.add_argument("--model_dir", default="/tmp/fact_b200")
    ap.add_argument("--steps", type=int, default=2400000)
    ap.add_argument("--grad_clip_norm", type=float, default=0.0)
    ap.add_argument("--steps_per_loop", type=int, default=10)          # trainer.py:166
    ap.add_argument("--checkpoint_interval", type=int, default=1000)   # trainer.py:170
    ap.add_argument("--max_to_keep", type=int, default=5)
    ap.add_argument("--init_tf_checkpoint", default="", help="TensorFlow checkpoint prefix to start from (weights only)")
    ap.add_argument("--export_tf_checkpoint", action="store_true",
                    help="also write every checkpoint in TensorFlow's format (ckpt-N.index / .data), readable by the "
                         "reference's tf.train.Checkpoint(model=...)")
    ap.add_argument("--data_npz", default="")
    ap.add_argument("--products", default="bf16", choices=["bf16"],
                    help="GEMM operand precision of the training step.  Only the bf16 product path exists (BASELINE.json "
                         "configs[2]: 'training step bf16'): bf16 operands, fp32 accumulation, fp32 residual stream / "
                         "statistics / gradients / master weights / Adam state.  The reference trains in fp32 "
                         "throughout, so loss curves agree to bf16 rounding of the GEMM operands, not bit for bit")
    args = ap.parse_args()
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    cfg = config_util.get_configs_from_pipeline_file(args.config_path)
    model = model_builder.build(cfg["model"], True, device=dev, mode="bf16", seed=0)   # same init on every replica
    opt = optim.Adam(model, learning_rate=optim.learning_rate_from_config(cfg["train_config"]))
    bs = cfg["train_config"].batch_size                                     # per replica, as in the reference
    if glob.glob(cfg["train_dataset"].data_files):           # trainer.py:140-146: inputs.create_input per replica
        # the same batches as inputs.create_input(..., seed=rank), decoded once and gathered on the device
        data = ({k: v for k, v in b.items() if k in ("motion_input", "audio_input", "target")}
                for b in device_inputs.create_device_input(cfg["train_config"], cfg["train_dataset"], dev, seed=rank))
    elif args.data_npz:
        data = npz_batches(args.data_npz, bs, rank)
    else:
        data = synthetic_batches(model.dims, bs, rank)
    trainer = SingleTaskTrainer(data, "target", model, optimizer=opt, grad_clip_norm=args.grad_clip_norm)
    os.makedirs(args.model_dir, exist_ok=True)
    ckpts = sorted(f for f in os.listdir(args.model_dir) if f.startswith("ckpt-") and f.endswith(".pt"))
    if args.init_tf_checkpoint and not ckpts:
        from mint_b200 import tf_checkpoint
        model.set_weights(tf_checkpoint.load_fact_weights(args.init_tf_checkpoint, model.dims))
    if ckpts:                                                               # Controller restores the latest (orbit)
        sd = torch.load(os.path.join(args.model_dir, ckpts[-1]), map_location=dev)
        if list(sd.get("names", model.variable_names())) != model.variable_names() or \
                sd["flat_parameters"].numel() != model.flat_parameters.numel():
            raise ValueError(f"{ckpts[-1]} was written for a different variable layout than this config builds")
        model.flat_parameters.copy_(sd["flat_parameters"])
        model.repack()
        opt.load_state_dict(sd["optimizer"])
    with torch.cuda.stream(torch.cuda.Stream(dev)):
        while opt.iterations < args.steps:
            n = min(args.steps_per_loop, args.steps - opt.iterations)
            logs = trainer.train(n)
            saving = opt.iterations % args.checkpoint_interval == 0 or opt.iterations == args.steps
            opt_state = opt.state_dict() if saving else None      # collective when the moments are sharded ("fused")
            if rank == 0:
                print(json.dumps({"step": opt.iterations, **logs}), flush=True)
                if saving:
                    path = os.path.join(args.model_dir, "ckpt-%09d.pt" % opt.iterations)
                    torch.save({"flat_parameters": model.flat_parameters, "optimizer": opt_state,
                                "names": model.variable_names()}, path)
                    if args.export_tf_checkpoint:
                        from mint_b200 import tf_checkpoint
                        tf_checkpoint.save_fact_weights(os.path.join(args.model_dir, "ckpt-%d" % opt.iterations),
                                                        {n: v.cpu().numpy() for n, v in model.get_weights().items()},
                                                        model.dims, step=opt.iterations)
                        tf_prefixes = sorted((f[:-len(".index")] for f in os.listdir(args.model_dir)
                                              if f.startswith("ckpt-") and f.endswith(".index")),
                                             key=lambda n: int(n.split("-")[1]))
                        for stale in tf_prefixes[:-args.max_to_keep]:            # CheckpointManager(max_to_keep=5)
                            for f in os.listdir(args.model_dir):
                                if f == stale + ".index" or f.startswith(stale + ".data-"):
                                    os.remove(os.path.join(args.model_dir, f))
                        tf_checkpoint.write_checkpoint_state(args.model_dir, tf_prefixes[-args.max_to_keep:])
                    old = sorted(f for f in os.listdir(args.model_dir)
                                 if f.startswith("ckpt-") and f.endswith(".pt"))[:-args.max_to_keep]
                    for f in old:
                        os.remove(os.path.join(args.model_dir, f))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
