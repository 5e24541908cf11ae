#!/usr/bin/env python
"""Golden of the training stream of mint_b200/inputs.py:create_input: sha256 digests of its first batches for a few
seeds, batch sizes and file layouts of seeded synthetic TFRecords.

The digests were generated before create_input's selection logic was factored out into inputs.training_order /
inputs.window_start, so tests/test_device_inputs.py can show that the refactor (and the faster parse_example) left
the stream untouched: same records, same order, same window starts, same bytes.

    python tests/golden/make_input_stream_golden.py
"""
import hashlib
import json
import os
import sys
import tempfile

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
from mint_b200 import config_util, inputs  # noqa: E402

HERE = os.path.dirname(os.path.abspath(__file__))
OUT = os.path.join(HERE, "input_stream_digests.json")

# name -> (records per file, frame range, batch size, seeds, batches digested).  Every layout is digested over at
# least three epochs of the shuffle buffer (fewer and more than its 100 records).
LAYOUTS = {
    "one_file_7": ([7], (240, 300), 3, [0, 1], 8),
    "three_files_130": ([40, 50, 40], (240, 280), 32, [0, 5], 13),
    "two_files_uneven": ([5, 1], (240, 260), 1, [3], 20),
}


def write_layout(root, counts, frames, seed=0):
    """Seeded synthetic TFRecords in the reference's feature layout: file f holds counts[f] records of
    T ~ U[frames] motion frames ([T, 219]) and as many audio frames ([T, 35]).  Returns the file glob."""
    rng = np.random.default_rng(seed)
    for fi, n in enumerate(counts):
        with inputs.TFRecordWriter(os.path.join(root, f"s_tfrecord-train-{fi:05d}")) as w:
            for i in range(n):
                t = int(rng.integers(frames[0], frames[1] + 1))
                m = rng.standard_normal((t, 219)).astype(np.float32)
                a = rng.standard_normal((t, 35)).astype(np.float32)
                w.write(inputs.to_tfexample(m, a, f"gBR_sBM_c{fi:02d}_{i:03d}", f"mBR{fi}_{i}").SerializeToString())
    return os.path.join(root, "s_tfrecord-train-*")


def configs(data_files, batch_size):
    return config_util.get_configs_from_pipeline_file(
        config_util.DEFAULT_CONFIG,
        'train_dataset { data_files: "%s" } train_config { batch_size: %d }' % (data_files, batch_size))


def digest(batch: dict) -> str:
    """sha256 over every key of a batch in order: name, dtype, shape and bytes of arrays; the bytes of name lists."""
    h = hashlib.sha256()
    for k, v in batch.items():
        h.update(k.encode())
        if isinstance(v, np.ndarray):
            h.update(f"{v.dtype.str}{v.shape}".encode())
            h.update(np.ascontiguousarray(v).tobytes())
        else:
            for s in v:
                h.update(len(s).to_bytes(8, "little") + s)
    return h.hexdigest()


def stream_digests(name, seed):
    counts, frames, batch_size, _, n = LAYOUTS[name]
    with tempfile.TemporaryDirectory() as root:
        cfg = configs(write_layout(root, counts, frames), batch_size)
        it = inputs.create_input(cfg["train_config"], cfg["train_dataset"], is_training=True, seed=seed)
        return [digest(next(it)) for _ in range(n)]


def main():
    out = {name: {str(seed): stream_digests(name, seed) for seed in spec[3]} for name, spec in LAYOUTS.items()}
    with open(OUT, "w") as f:
        json.dump(out, f, indent=1)
    print({name: {s: len(d) for s, d in v.items()} for name, v in out.items()})


if __name__ == "__main__":
    main()
