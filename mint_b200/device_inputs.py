"""Device-resident training input: the TFRecords are decoded once into arenas in GPU memory, and every step's windows
are gathered there by fact_gather_windows.

create_device_input yields exactly what inputs.create_input yields for the same seed -- the same clips, windows, names
and bytes -- as device tensors.  Both producers run one selection policy (inputs.training_order over the files,
inputs.window_start after each item): create_input passes parsed examples through it, this module passes sequence
indices and turns each (sequence, start) into arena rows.  What changes is the cost: create_input parses a whole record
every time the shuffle buffer hands it out, to use 240 of its frames; here a step costs a few microseconds of copying
on the device plus, once per block of steps, the host-side draws and one upload of the row table.

WindowPlan is the host half (decode, checks, row tables) and needs no GPU; DeviceInput owns the device arenas.
"""
from __future__ import annotations

import glob

import numpy as np
import torch

from . import inputs

MOTION_PAD = 6          # fact_preprocessing pads motion with six leading zeros (3-dim translation -> 9-dim slot)


class WindowPlan:
    """The decoded training set and the training order as arena rows.

    motion: fp32 [rows, 219 + 6], every sequence padded as fact_preprocessing pads it; audio: fp32 [rows', 35];
    sequence s occupies motion[motion_offset[s]:][:motion_frames[s]] and audio[audio_offset[s]:][:audio_frames[s]].
    Sequences are numbered in sorted(glob) file order, records in file order."""

    def __init__(self, train_eval_config, dataset_config, seed: int | None = None):
        self.batch_size = int(train_eval_config.batch_size)
        files = sorted(glob.glob(dataset_config.data_files))
        if not files:
            raise FileNotFoundError(f"no TFRecord files match {dataset_config.data_files!r}")
        steps = [s.WhichOneof("preprocessor") for s in dataset_config.data_augmentation_options]
        if steps.count("fact_preprocessor") != 1:
            raise ValueError(f"device-resident input implements one fact_preprocessor step, the config has {steps}")
        self.params = params = inputs.get_modality_to_param_dict(dataset_config)
        mp, ap = params["motion"], params["audio"]
        self.window = inputs.training_window(params)
        self.motion_len, self.audio_len = mp["input_length"], ap["input_length"]
        self.target_shift, self.target_len = mp["target_shift"], mp["target_length"]

        motions, audios, self.motion_name, self.audio_name, first = [], [], [], [], [0]
        for path in files:
            for i, rec in enumerate(inputs.read_tfrecords(path)):
                ex = inputs.parse_example(rec)
                m, a = ex["motion_sequence"], ex["audio_sequence"]
                where = f"{path} record {i}"
                if m.ndim != 2 or a.ndim != 2:
                    raise ValueError(f"{where}: motion {m.shape} and audio {a.shape} must be [frames, features]")
                if m.shape[0] < self.window:
                    raise ValueError(f"{where}: sequence of {m.shape[0]} frames is shorter than the "
                                     f"{self.window}-frame window")
                # the latest start is T - window: its audio window must be whole, or the batch would be ragged
                if a.shape[0] < m.shape[0] - self.window + self.audio_len:
                    raise ValueError(f"{where}: audio track of {a.shape[0]} frames is too short for the windows of "
                                     f"a {m.shape[0]}-frame sequence (needs {m.shape[0] - self.window + self.audio_len})")
                if motions and (m.shape[1] != motions[0].shape[1] or a.shape[1] != audios[0].shape[1]):
                    raise ValueError(f"{where}: feature widths {m.shape[1]}/{a.shape[1]} differ from the first "
                                     f"record's {motions[0].shape[1]}/{audios[0].shape[1]}")
                motions.append(m)
                audios.append(a)
                self.motion_name.append(ex["motion_name"])
                self.audio_name.append(ex["audio_name"])
            first.append(len(motions))
        if not motions:
            raise ValueError(f"the files matching {dataset_config.data_files!r} hold no records")
        self.file_first = first
        self.motion_frames = np.array([m.shape[0] for m in motions], np.int64)
        self.audio_frames = np.array([a.shape[0] for a in audios], np.int64)
        self.motion_offset = np.concatenate([[0], np.cumsum(self.motion_frames)[:-1]]).astype(np.int64)
        self.audio_offset = np.concatenate([[0], np.cumsum(self.audio_frames)[:-1]]).astype(np.int64)
        self.motion = np.zeros((int(self.motion_frames.sum()), motions[0].shape[1] + MOTION_PAD), np.float32)
        for off, m in zip(self.motion_offset, motions):
            self.motion[off:off + m.shape[0], MOTION_PAD:] = m
        self.audio = np.concatenate(audios).astype(np.float32, copy=False)
        # create_input's "*_sequence_shape" entries: the unpadded shape of each record, int32
        self.motion_shape = np.array([m.shape for m in motions], np.int32)
        self.audio_shape = np.array([a.shape for a in audios], np.int32)
        self.rng = np.random.default_rng(seed)
        self._order = inputs.training_order(len(files), lambda fi: range(first[fi], first[fi + 1]), self.rng)

    def rows(self, steps: int) -> np.ndarray:
        """int64 [steps, 3, batch]: per step the motion rows, audio rows and sequence indices of its clips, drawn as
        create_input draws them (the window start right after each item leaves the shuffle buffer)."""
        out = np.empty((steps, 3, self.batch_size), np.int64)
        for s in range(steps):
            for b in range(self.batch_size):
                seq = next(self._order)
                start = inputs.window_start(int(self.motion_frames[seq]), self.params, self.rng)
                out[s, 0, b] = self.motion_offset[seq] + start
                out[s, 1, b] = self.audio_offset[seq] + start
                out[s, 2, b] = seq
        return out


class DeviceInput:
    """Iterator of training batches gathered on `device` (see create_device_input)."""

    def __init__(self, plan: WindowPlan, device, steps_per_block: int = 64):
        from . import lib
        self._lib = lib
        self._fn = lib.load().fact_gather_windows
        self.plan = plan
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise ValueError(f"device-resident input needs a CUDA device, got {self.device}")
        self.steps_per_block = max(1, int(steps_per_block))
        with torch.cuda.device(self.device):         # pageable -> device copies: complete when .to() returns
            self.motion = torch.from_numpy(plan.motion).to(self.device)
            self.audio = torch.from_numpy(plan.audio).to(self.device)
            self.motion_shape = torch.from_numpy(plan.motion_shape).to(self.device)
            self.audio_shape = torch.from_numpy(plan.audio_shape).to(self.device)
        self._host = None                             # this block's row table: host copy (names) and device copy
        self._table = None
        self._table_stream = None
        self._step = 0

    def __iter__(self):
        return self

    def _refill(self, stream) -> None:
        self._host = self.plan.rows(self.steps_per_block)
        pinned = torch.from_numpy(self._host).pin_memory()
        # the caching host allocator keeps the pinned block until this copy has run; the device table is a fresh
        # allocation on `stream`, so neither buffer is reused while a gather may still read it
        with torch.cuda.stream(stream):
            self._table = pinned.to(self.device, non_blocking=True)
        self._table_stream = stream
        self._step = 0

    def __next__(self) -> dict:
        p = self.plan
        stream = torch.cuda.current_stream(self.device)
        if self._table is None or self._step == self.steps_per_block:
            self._refill(stream)
        elif stream != self._table_stream:            # iteration moved to another stream mid-block
            stream.wait_stream(self._table_stream)
            self._table.record_stream(stream)
            self._table_stream = stream
        rows, host = self._table[self._step], self._host[self._step]
        self._step += 1
        batch, dev = p.batch_size, self.device
        motion_out = torch.empty((batch, p.motion_len, self.motion.shape[1]), dtype=torch.float32, device=dev)
        target_out = torch.empty((batch, p.target_len, self.motion.shape[1]), dtype=torch.float32, device=dev)
        audio_out = torch.empty((batch, p.audio_len, self.audio.shape[1]), dtype=torch.float32, device=dev)
        with torch.cuda.device(dev):
            self._lib.check(self._fn(self.motion.data_ptr(), self.motion.shape[1], self.audio.data_ptr(),
                                     self.audio.shape[1], rows[0].data_ptr(), rows[1].data_ptr(), batch, p.motion_len,
                                     p.target_shift, p.target_len, p.audio_len, motion_out.data_ptr(),
                                     target_out.data_ptr(), audio_out.data_ptr(), stream.cuda_stream),
                            "fact_gather_windows")
            seq = rows[2]
            motion_shape = self.motion_shape.index_select(0, seq)
            audio_shape = self.audio_shape.index_select(0, seq)
        # create_input's keys, in its order
        return {"motion_sequence_shape": motion_shape, "motion_name": [p.motion_name[s] for s in host[2]],
                "audio_sequence_shape": audio_shape, "audio_name": [p.audio_name[s] for s in host[2]],
                "motion_input": motion_out, "target": target_out, "audio_input": audio_out}


def create_device_input(train_eval_config, dataset_config, device, seed: int | None = None,
                        steps_per_block: int = 64) -> DeviceInput:
    """Training batches of inputs.create_input(train_eval_config, dataset_config, is_training=True, seed=seed),
    bit for bit, as tensors on `device`.  Decodes every file once at construction and raises ValueError there for a
    record create_input could not batch (a sequence shorter than the window, an audio track too short for a window it
    allows).  Each next() launches one gather on the current stream into freshly allocated outputs; the host draws
    the windows of steps_per_block steps at a time and uploads their row table with one non-blocking copy."""
    return DeviceInput(WindowPlan(train_eval_config, dataset_config, seed), device, steps_per_block)
