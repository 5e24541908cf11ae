"""Host side of the device-resident training input (CPU only): the faster float-list decoding of parse_example, the
unchanged create_input stream, and the shared selection policy of mint_b200/device_inputs.py against create_input."""
import hashlib
import json
import os
import struct

import numpy as np
import pytest

from mint_b200 import device_inputs, inputs
from tests.golden import make_input_stream_golden as G

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def _list_decode(record: bytes) -> dict:
    """parse_example as it was: np.asarray over protobuf's repeated-float containers."""
    f = inputs.Example.FromString(record).features.feature
    out = {}
    for modality in ("motion", "audio"):
        shape = tuple(int(v) for v in f[f"{modality}_sequence_shape"].int64_list.value)
        out[f"{modality}_sequence"] = np.asarray(f[f"{modality}_sequence"].float_list.value, np.float32).reshape(shape)
        out[f"{modality}_sequence_shape"] = np.asarray(shape, np.int32)
        out[f"{modality}_name"] = bytes(f[f"{modality}_name"].bytes_list.value[0])
    return out


def _assert_same_example(got: dict, want: dict):
    assert list(got) == list(want)
    for k, v in want.items():
        if isinstance(v, np.ndarray):
            assert got[k].dtype == v.dtype and got[k].shape == v.shape, k
            assert got[k].tobytes() == v.tobytes(), k               # bitwise, NaN payloads and signed zeros included
            assert got[k].flags.writeable, k
        else:
            assert got[k] == v, k


@pytest.mark.parametrize("t_motion,t_audio", [(0, 0), (1, 0), (0, 3), (1, 1), (37, 74), (600, 600)])
def test_parse_example_equals_the_protobuf_list_decoding(t_motion, t_audio):
    rng = np.random.default_rng(t_motion * 1000 + t_audio)
    m = rng.standard_normal((t_motion, 219)).astype(np.float32)
    a = rng.standard_normal((t_audio, 35)).astype(np.float32)
    if m.size:
        m.ravel()[:6] = [np.nan, -0.0, np.inf, -np.inf, 1e-45, -3.4e38]   # special values survive bit for bit
    rec = inputs.to_tfexample(m, a, "gBR_sBM_c01", "mBR0").SerializeToString()
    got = inputs.parse_example(rec)
    _assert_same_example(got, _list_decode(rec))
    assert got["motion_sequence"].tobytes() == m.tobytes() and got["audio_sequence"].tobytes() == a.tobytes()


def _varint(v: int) -> bytes:
    out = bytearray()
    while True:
        b = v & 0x7F
        v >>= 7
        out.append(b | (0x80 if v else 0))
        if not v:
            return bytes(out)


def _ld(field: int, payload: bytes) -> bytes:
    return _varint(field << 3 | 2) + _varint(len(payload)) + payload


def test_parse_example_reads_unpacked_float_lists():
    """A tf.train.Example framed by hand with every float as its own field-1 fixed32 entry (the unpacked encoding a
    writer may legally use): same arrays as the list decoding."""
    rng = np.random.default_rng(0)
    m = rng.standard_normal((3, 219)).astype(np.float32)
    a = rng.standard_normal((5, 35)).astype(np.float32)

    def floats(x):
        return _ld(2, b"".join(b"\x0d" + struct.pack("<f", v) for v in x.ravel()))           # Feature.float_list

    def ints(shape):
        return _ld(3, _ld(1, b"".join(_varint(v) for v in shape)))                          # Feature.int64_list

    def name(s):
        return _ld(1, _ld(1, s))                                                            # Feature.bytes_list

    feats = {"motion_sequence": floats(m), "motion_sequence_shape": ints(m.shape), "motion_name": name(b"m0"),
             "audio_sequence": floats(a), "audio_sequence_shape": ints(a.shape), "audio_name": name(b"a0")}
    rec = _ld(1, b"".join(_ld(1, _ld(1, k.encode()) + _ld(2, v)) for k, v in feats.items()))
    assert b"\x0d" + struct.pack("<f", m.ravel()[1]) in rec                                   # really unpacked
    got = inputs.parse_example(rec)
    _assert_same_example(got, _list_decode(rec))
    assert np.array_equal(got["motion_sequence"], m) and np.array_equal(got["audio_sequence"], a)


def test_float_lists_of_the_tensorflow_written_sample_hash_to_the_manifest():
    """Every float list of the TensorFlow-written records, through float_list_array, hashes to the manifest's sha256
    of its little-endian fp32 values (tests/golden/make_tfrecord_golden.py:feature_summary)."""
    with open(os.path.join(GOLDEN, "tfrecord_manifest.json")) as f:
        man = json.load(f)
    sample = man["sample"]
    recs = list(inputs.read_tfrecords(os.path.join(GOLDEN, sample["path"]), verify_payload_crc=True))
    seen = 0
    for payload, i in zip(recs, sample["records"]):
        want = man["files"][sample["file"]]["records"][i]["features"]
        for key, feat in inputs.Example.FromString(payload).features.feature.items():
            if feat.WhichOneof("kind") != "float_list":
                continue
            arr = inputs.float_list_array(feat.float_list)
            assert arr.dtype == np.float32 and [want[key][0], want[key][1]] == ["float_list", arr.size], key
            assert hashlib.sha256(arr.astype("<f4").tobytes()).hexdigest() == want[key][2], key
            seen += 1
    assert seen >= 8


@pytest.mark.parametrize("layout", sorted(G.LAYOUTS))
def test_create_input_stream_is_unchanged(tmp_path, layout):
    """Digests of create_input's first batches, generated before its selection logic was factored out."""
    with open(G.OUT) as f:
        want = json.load(f)[layout]
    counts, frames, batch_size, seeds, n = G.LAYOUTS[layout]
    cfg = G.configs(G.write_layout(str(tmp_path), counts, frames), batch_size)
    for seed in seeds:
        it = inputs.create_input(cfg["train_config"], cfg["train_dataset"], is_training=True, seed=seed)
        assert [G.digest(next(it)) for _ in range(n)] == want[str(seed)], seed


@pytest.fixture(scope="module")
def layouts(tmp_path_factory):
    """one file of 7 records (fewer than the shuffle buffer) and three files of 130 (more)."""
    out = {}
    for name, counts in (("one", [7]), ("several", [40, 50, 40])):
        root = tmp_path_factory.mktemp(name)
        out[name] = (G.write_layout(str(root), counts, (240, 300), seed=len(counts)), sum(counts))
    return out


def numpy_gather(plan: device_inputs.WindowPlan, rows: np.ndarray) -> dict:
    """What fact_gather_windows computes, with NumPy slicing over the plan's arenas, in create_input's key order."""
    m0, a0, seq = rows
    return {"motion_sequence_shape": plan.motion_shape[seq], "motion_name": [plan.motion_name[s] for s in seq],
            "audio_sequence_shape": plan.audio_shape[seq], "audio_name": [plan.audio_name[s] for s in seq],
            "motion_input": np.stack([plan.motion[r:r + plan.motion_len] for r in m0]),
            "target": np.stack([plan.motion[r + plan.target_shift:r + plan.target_shift + plan.target_len]
                                for r in m0]),
            "audio_input": np.stack([plan.audio[r:r + plan.audio_len] for r in a0])}


@pytest.mark.parametrize("name,batch_size,seed", [("one", 1, 0), ("one", 3, 7), ("one", 32, 1),
                                                   ("several", 1, 2), ("several", 3, 0), ("several", 32, 7)])
def test_shared_selection_and_a_numpy_gather_equal_create_input(layouts, name, batch_size, seed):
    files, records = layouts[name]
    cfg = G.configs(files, batch_size)
    steps = -(-3 * records // batch_size) + 1                        # a little over three epochs
    host = inputs.create_input(cfg["train_config"], cfg["train_dataset"], is_training=True, seed=seed)
    plan = device_inputs.WindowPlan(cfg["train_config"], cfg["train_dataset"], seed=seed)
    assert plan.window == 240 and plan.motion.shape[1] == 225 and plan.audio.shape[1] == 35
    table = np.concatenate([plan.rows(5) for _ in range(-(-steps // 5))])  # drawn in blocks, as the device does
    seen = set()
    for s in range(steps):
        want, rows = next(host), table[s]
        got = numpy_gather(plan, rows)
        assert list(got) == list(want)
        for k, v in want.items():
            if isinstance(v, np.ndarray):
                assert got[k].dtype == v.dtype and np.array_equal(got[k], v), (s, k)
            else:
                assert got[k] == v, (s, k)
        # every window lies inside its own sequence
        seq = rows[2]
        assert np.all(rows[0] >= plan.motion_offset[seq])
        assert np.all(rows[0] + plan.window <= plan.motion_offset[seq] + plan.motion_frames[seq])
        assert np.all(rows[1] + plan.audio_len <= plan.audio_offset[seq] + plan.audio_frames[seq])
        seen.update(seq.tolist())
    assert seen == set(range(records))


def test_construction_errors(tmp_path):
    window = 240
    for sub, clips, what in (("short", [(300, 300), (window - 1, window - 1)], "shorter than the 240-frame window"),
                             ("audio", [(300, 300), (300, 300 - window + 240 - 1)], "audio track of")):
        root = tmp_path / sub
        root.mkdir()
        with inputs.TFRecordWriter(str(root / "x_tfrecord-train-0")) as w:
            for i, (tm, ta) in enumerate(clips):
                w.write(inputs.to_tfexample(np.zeros((tm, 219), np.float32), np.zeros((ta, 35), np.float32),
                                            f"m{i}", f"a{i}").SerializeToString())
        cfg = G.configs(str(root / "*"), 2)
        with pytest.raises(ValueError, match=what):
            device_inputs.WindowPlan(cfg["train_config"], cfg["train_dataset"], seed=0)
    # the longest audio window a 300-frame sequence allows needs exactly 300 audio frames: accepted
    ok = tmp_path / "ok"
    ok.mkdir()
    with inputs.TFRecordWriter(str(ok / "x_tfrecord-train-0")) as w:
        w.write(inputs.to_tfexample(np.zeros((300, 219), np.float32), np.zeros((300, 35), np.float32),
                                    "m", "a").SerializeToString())
    cfg = G.configs(str(ok / "*"), 2)
    device_inputs.WindowPlan(cfg["train_config"], cfg["train_dataset"], seed=0)
    (tmp_path / "empty").mkdir()
    open(tmp_path / "empty" / "x_tfrecord-train-0", "wb").close()
    cfg = G.configs(str(tmp_path / "empty" / "*"), 2)
    with pytest.raises(ValueError, match="hold no records"):
        device_inputs.WindowPlan(cfg["train_config"], cfg["train_dataset"], seed=0)
    cfg = G.configs(str(tmp_path / "nothing_here_*"), 2)
    with pytest.raises(FileNotFoundError):
        device_inputs.WindowPlan(cfg["train_config"], cfg["train_dataset"], seed=0)
    cfg = G.configs(str(ok / "*"), 2)
    cfg["train_dataset"].ClearField("data_augmentation_options")
    with pytest.raises(ValueError, match="fact_preprocessor"):
        device_inputs.WindowPlan(cfg["train_config"], cfg["train_dataset"], seed=0)
