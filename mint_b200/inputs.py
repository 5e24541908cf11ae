"""Input pipeline for the reference's on-disk format, without TensorFlow (SURVEY.md 8f N1).

Reads / writes the TFRecord files produced by the reference's tools/preprocessing.py:54-69 (`tf.train.Example` with
`{motion,audio}_sequence` float lists, `*_sequence_shape` int64 lists, `*_name` bytes) and applies the reference's
`fact_preprocessing` windowing (mint/utils/inputs_util.py:59-107): motion padded 219 -> 225 with six leading zeros;
training: random `start`, motion_input = seq[start:start+120], target = seq[start+120:start+140], audio_input =
audio[start:start+240]; eval: start = 0 and the FULL audio track.  `create_input` mirrors mint/core/inputs.py:20-123
(shuffle buffer 100 + repeat + drop_remainder in training; one ordered pass in eval) and yields dicts of NumPy arrays.
Its training order (training_order) and window starts (window_start) are shared with mint_b200/device_inputs.py, which
yields the same batches from a dataset decoded once into GPU memory.

TFRecord framing: u64 length | u32 masked-crc32c(length) | payload | u32 masked-crc32c(payload).
"""
from __future__ import annotations

import glob
import struct

import numpy as np
from google.protobuf import descriptor_pb2 as _dpb
from google.protobuf import descriptor_pool as _pool_mod
from google.protobuf import message_factory as _mf

# ------------------------------------------------------------------------------------------- crc32c (Castagnoli)
_POLY = 0x82F63B78
_TABLE = []
for _i in range(256):
    _c = _i
    for _ in range(8):
        _c = (_c >> 1) ^ (_POLY if _c & 1 else 0)
    _TABLE.append(_c)
_TABLE_NP = np.array(_TABLE, dtype=np.uint32)


def crc32c(data: bytes) -> int:
    crc = 0xFFFFFFFF
    tab = _TABLE
    for b in data:
        crc = tab[(crc ^ b) & 0xFF] ^ (crc >> 8)
    return crc ^ 0xFFFFFFFF


def masked_crc(data: bytes) -> int:
    c = crc32c(data)
    return (((c >> 15) | (c << 17)) + 0xA282EAD8) & 0xFFFFFFFF


# ------------------------------------------------------------------------------------------- tf.train.Example schema
def _build_example_classes():
    F = _dpb.FieldDescriptorProto
    fd = _dpb.FileDescriptorProto()
    fd.name = "mint_b200/tf_example_schema.proto"
    fd.package = "tensorflow"
    fd.syntax = "proto3"

    def msg(name):
        m = fd.message_type.add()
        m.name = name
        return m

    def field(m, name, num, ftype, label=F.LABEL_OPTIONAL, type_name=None, oneof=None, packed=None):
        f = m.field.add()
        f.name, f.number, f.type, f.label = name, num, ftype, label
        if type_name:
            f.type_name = type_name
        if oneof is not None:
            f.oneof_index = oneof
        if packed is not None:
            f.options.packed = packed
        return f

    field(msg("BytesList"), "value", 1, F.TYPE_BYTES, F.LABEL_REPEATED)
    field(msg("FloatList"), "value", 1, F.TYPE_FLOAT, F.LABEL_REPEATED, packed=True)
    field(msg("Int64List"), "value", 1, F.TYPE_INT64, F.LABEL_REPEATED, packed=True)
    feat = msg("Feature")
    feat.oneof_decl.add().name = "kind"
    field(feat, "bytes_list", 1, F.TYPE_MESSAGE, type_name=".tensorflow.BytesList", oneof=0)
    field(feat, "float_list", 2, F.TYPE_MESSAGE, type_name=".tensorflow.FloatList", oneof=0)
    field(feat, "int64_list", 3, F.TYPE_MESSAGE, type_name=".tensorflow.Int64List", oneof=0)
    feats = msg("Features")
    entry = feats.nested_type.add()
    entry.name = "FeatureEntry"
    entry.options.map_entry = True
    field(entry, "key", 1, F.TYPE_STRING)
    field(entry, "value", 2, F.TYPE_MESSAGE, type_name=".tensorflow.Feature")
    field(feats, "feature", 1, F.TYPE_MESSAGE, F.LABEL_REPEATED, type_name=".tensorflow.Features.FeatureEntry")
    field(msg("Example"), "features", 1, F.TYPE_MESSAGE, type_name=".tensorflow.Features")
    pool = _pool_mod.DescriptorPool()
    pool.Add(fd)
    return _mf.GetMessageClass(pool.FindMessageTypeByName("tensorflow.Example"))


Example = _build_example_classes()


def to_tfexample(motion_sequence, audio_sequence, motion_name: str, audio_name: str):
    """Same feature set as the reference writer (tools/preprocessing.py:54-69)."""
    ex = Example()
    f = ex.features.feature
    m = np.asarray(motion_sequence, np.float32)
    a = np.asarray(audio_sequence, np.float32)
    f["motion_name"].bytes_list.value.append(motion_name.encode("utf-8"))
    f["motion_sequence"].float_list.value.extend(m.ravel().tolist())
    f["motion_sequence_shape"].int64_list.value.extend(m.shape)
    f["audio_name"].bytes_list.value.append(audio_name.encode("utf-8"))
    f["audio_sequence"].float_list.value.extend(a.ravel().tolist())
    f["audio_sequence_shape"].int64_list.value.extend(a.shape)
    return ex


def float_list_array(float_list) -> np.ndarray:
    """A FloatList's values as a writable float32 array.  The field is declared packed, so its serialisation is one
    tag byte, the varint byte count and the little-endian floats -- whatever encoding the record used -- and one
    np.frombuffer over it replaces np.asarray's element-by-element walk of protobuf's repeated-float container
    (the bulk of the decoding time of a long sequence)."""
    raw = float_list.SerializeToString()
    if not raw:
        return np.zeros(0, np.float32)
    if raw[0] != 0x0A:                                          # field 1, length-delimited
        raise ValueError(f"FloatList serialised with unexpected tag {raw[0]:#x}")
    n, shift, pos = 0, 0, 1
    while True:
        b = raw[pos]
        pos += 1
        n |= (b & 0x7F) << shift
        shift += 7
        if b < 0x80:
            break
    if pos + n != len(raw) or n % 4:
        raise ValueError(f"FloatList of {len(raw)} bytes has a packed field of {n} bytes at offset {pos}")
    return np.frombuffer(raw, "<f4", n // 4, pos).astype(np.float32)     # astype copies: writable, own memory


def parse_example(record: bytes) -> dict:
    """-> {motion_sequence [T,219], audio_sequence [T',35], motion_name, audio_name} (mint/core/inputs.py:78-94)."""
    ex = Example.FromString(record)
    f = ex.features.feature
    out = {}
    for modality in ("motion", "audio"):
        shape = tuple(int(v) for v in f[f"{modality}_sequence_shape"].int64_list.value)
        out[f"{modality}_sequence"] = float_list_array(f[f"{modality}_sequence"].float_list).reshape(shape)
        out[f"{modality}_sequence_shape"] = np.asarray(shape, np.int32)
        out[f"{modality}_name"] = bytes(f[f"{modality}_name"].bytes_list.value[0])
    return out


# ------------------------------------------------------------------------------------------- TFRecord files
class TFRecordWriter:
    def __init__(self, path: str):
        self._f = open(path, "wb")

    def write(self, payload: bytes) -> None:
        header = struct.pack("<Q", len(payload))
        self._f.write(header)
        self._f.write(struct.pack("<I", masked_crc(header)))
        self._f.write(payload)
        self._f.write(struct.pack("<I", masked_crc(payload)))

    def close(self) -> None:
        self._f.close()

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()


def read_tfrecords(path: str, verify_payload_crc: bool = False):
    """Yields the raw payload of every record; the length CRC is always checked."""
    with open(path, "rb") as f:
        while True:
            header = f.read(8)
            if not header:
                return
            if len(header) != 8:
                raise IOError(f"{path}: truncated record header")
            (length,) = struct.unpack("<Q", header)
            (lcrc,) = struct.unpack("<I", f.read(4))
            if lcrc != masked_crc(header):
                raise IOError(f"{path}: corrupted record length")
            payload = f.read(length)
            tail = f.read(4)
            if len(payload) != length or len(tail) != 4:
                raise IOError(f"{path}: truncated record")
            if verify_payload_crc and struct.unpack("<I", tail)[0] != masked_crc(payload):
                raise IOError(f"{path}: corrupted record payload")
            yield payload


# ------------------------------------------------------------------------------------------- preprocessing
def get_modality_to_param_dict(dataset_config) -> dict:
    """mint/utils/inputs_util.py:18-45."""
    out = {}
    for modality in dataset_config.modality:
        kind = modality.WhichOneof("modality")
        if kind != "general_modality":
            raise ValueError("Unknown modality type:", kind)
        m = modality.general_modality
        out[m.feature_name] = {
            "feature_dim": m.dimension,
            "input_length": int(dataset_config.input_length_sec * m.sample_rate),
            "target_length": int(dataset_config.target_length_sec * m.sample_rate),
            "target_shift": int(dataset_config.target_shift_sec * m.sample_rate),
            "sample_rate": m.sample_rate,
            "resize": m.resize,
            "crop_size": m.crop_size,
        }
    return out


def training_window(modality_to_params: dict) -> int:
    """Frames a training window spans: motion input, target and audio input all start at the same frame."""
    mp, ap = modality_to_params["motion"], modality_to_params["audio"]
    return max(mp["input_length"], mp["target_shift"] + mp["target_length"], ap["input_length"])


def window_start(num_frames: int, modality_to_params: dict, rng) -> int:
    """The random first frame of a training window over a sequence of num_frames frames (inputs_util.py:82-86):
    one rng.integers(0, T - window + 1) draw."""
    window = training_window(modality_to_params)
    hi = num_frames - window + 1
    if hi <= 0:
        raise ValueError(f"sequence of {num_frames} frames is shorter than the {window}-frame window")
    return int(rng.integers(0, hi))


def fact_preprocessing(example: dict, modality_to_params: dict, is_training: bool, rng=None) -> dict:
    """mint/utils/inputs_util.py:59-107 on NumPy arrays."""
    ex = dict(example)
    mp, ap = modality_to_params["motion"], modality_to_params["audio"]
    seq = np.pad(ex.pop("motion_sequence"), [[0, 0], [6, 0]])            # 3-dim translation -> 9-dim slot
    audio = ex.pop("audio_sequence")
    if is_training:
        start = window_start(seq.shape[0], modality_to_params, rng or np.random.default_rng())
    else:
        start = 0
    ex["motion_input"] = seq[start:start + mp["input_length"]]
    if is_training:
        ex["target"] = seq[start + mp["target_shift"]:start + mp["target_shift"] + mp["target_length"]]
        ex["audio_input"] = audio[start:start + ap["input_length"]]
    else:
        ex["audio_input"] = audio
    return ex


SHUFFLE_BUFFER = 100        # .shuffle(100) of mint/core/inputs.py
SHUFFLE_DRAIN = 50          # what is left of the buffer when the last file of an epoch has been read


def training_order(num_files: int, file_items, rng):
    """The order in which training draws items (mint/core/inputs.py: interleave + .shuffle(100) + .repeat()): per epoch
    a permutation of the files, each file's items in file order through a shuffle buffer of 100 that yields a random
    item once full, and at the end of an epoch a drain down to 50 items.  file_items(f) gives the items of file f
    (parsed examples for create_input, sequence indices for create_device_input); the items are opaque here.

    The caller may draw from `rng` between two items (the window start of fact_preprocessing is drawn right after
    each item leaves the buffer); the generator only calls rng when the next item is asked for, so such draws
    interleave with its own exactly as they do in create_input.  Ends only if the files hold no items."""
    buf = []
    while True:                                                 # .repeat()
        order = rng.permutation(num_files)                      # interleave(deterministic=False): any file order
        for fi in order:
            for item in file_items(fi):
                buf.append(item)
                if len(buf) >= SHUFFLE_BUFFER:
                    yield buf.pop(int(rng.integers(0, len(buf))))
        if not buf:
            return
        while len(buf) > SHUFFLE_DRAIN:
            yield buf.pop(int(rng.integers(0, len(buf))))


def create_input(train_eval_config, dataset_config, num_cpu_threads: int = 2, is_training: bool = True,
                 use_tpu: bool = False, seed: int | None = None):
    """Generator of batches (dict of NumPy arrays) -- mint/core/inputs.py:20-123."""
    batch_size = train_eval_config.batch_size
    files = sorted(glob.glob(dataset_config.data_files))
    if not files:
        raise FileNotFoundError(f"no TFRecord files match {dataset_config.data_files!r}")
    params = get_modality_to_param_dict(dataset_config)
    steps = [s.WhichOneof("preprocessor") for s in dataset_config.data_augmentation_options]
    rng = np.random.default_rng(seed)

    def examples():
        if is_training:
            yield from training_order(len(files), lambda fi: map(parse_example, read_tfrecords(files[fi])), rng)
        else:
            for path in files:
                for rec in read_tfrecords(path):
                    yield parse_example(rec)

    def processed():
        for ex in examples():
            for step in steps:
                if step == "fact_preprocessor":
                    ex = fact_preprocessing(ex, params, is_training, rng)
            yield ex

    def batches():
        batch = []
        for ex in processed():
            batch.append(ex)
            if len(batch) == batch_size:
                yield _collate(batch)
                batch = []
        if batch and not (is_training or use_tpu):              # drop_remainder only in training / on TPU
            yield _collate(batch)

    return batches()


def _collate(batch: list) -> dict:
    out = {}
    for k in batch[0]:
        vals = [b[k] for b in batch]
        if isinstance(vals[0], np.ndarray):
            if any(v.shape != vals[0].shape for v in vals):
                raise ValueError(f"cannot batch ragged {k}: shapes {[v.shape for v in vals]} (eval uses batch 1)")
            out[k] = np.stack(vals)
        else:
            out[k] = vals
    return out
