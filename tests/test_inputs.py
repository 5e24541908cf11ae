"""TFRecord / tf.train.Example reader-writer and the reference's fact_preprocessing windowing (no TensorFlow)."""
import os
import struct

import numpy as np
import pytest

from mint_b200 import config_util, inputs


def test_crc32c_known_answers():
    assert inputs.crc32c(b"123456789") == 0xE3069283            # standard CRC-32C check value
    assert inputs.crc32c(b"") == 0
    assert inputs.crc32c(bytes(32)) == 0x8A9136AA               # RFC 3720 B.4: 32 zero bytes
    assert inputs.crc32c(bytes([0xFF] * 32)) == 0x62A8AB43      # RFC 3720 B.4: 32 0xFF bytes


def test_example_wire_format_is_tf_train_example():
    """Hand-built wire bytes of a tf.train.Example (field numbers of tensorflow/core/example/{example,feature}.proto)."""
    ex = inputs.Example()
    ex.features.feature["n"].int64_list.value.extend([3, 2])
    # Example{1: Features{1: entry{1: "n", 2: Feature{3: Int64List{1: packed [3, 2]}}}}}
    want = bytes([0x0A, 0x0D, 0x0A, 0x0B, 0x0A, 0x01, ord("n"), 0x12, 0x06, 0x1A, 0x04, 0x0A, 0x02, 0x03, 0x02])
    assert ex.SerializeToString(deterministic=True) == want
    back = inputs.Example.FromString(want)
    assert list(back.features.feature["n"].int64_list.value) == [3, 2]


def _write(tmp_path, name, clips):
    path = str(tmp_path / name)
    with inputs.TFRecordWriter(path) as w:
        for i, (t_m, t_a) in enumerate(clips):
            rng = np.random.default_rng(i)
            ex = inputs.to_tfexample(rng.standard_normal((t_m, 219)).astype(np.float32),
                                     rng.standard_normal((t_a, 35)).astype(np.float32), f"gBR_sBM_c{i:02d}", f"mBR{i}")
            w.write(ex.SerializeToString())
    return path


def test_tfrecord_roundtrip_and_corruption(tmp_path):
    path = _write(tmp_path, "a_tfrecord-train-0", [(300, 600), (260, 520)])
    recs = list(inputs.read_tfrecords(path, verify_payload_crc=True))
    assert len(recs) == 2
    ex = inputs.parse_example(recs[1])
    assert ex["motion_sequence"].shape == (260, 219) and ex["audio_sequence"].shape == (520, 35)
    assert ex["motion_name"] == b"gBR_sBM_c01" and ex["audio_name"] == b"mBR1"
    raw = bytearray(open(path, "rb").read())
    raw[20] ^= 0xFF
    open(path, "wb").write(bytes(raw))
    with pytest.raises(IOError):
        list(inputs.read_tfrecords(path, verify_payload_crc=True))
    (length,) = struct.unpack("<Q", bytes(raw[:8]))
    assert length == len(recs[0])


def test_fact_preprocessing_matches_reference_rules(tmp_path):
    cfg = config_util.get_configs_from_pipeline_file(config_util.DEFAULT_CONFIG)
    params = inputs.get_modality_to_param_dict(cfg["train_dataset"])
    assert params["motion"]["input_length"] == 120 and params["audio"]["input_length"] == 240
    assert params["motion"]["target_length"] == 20 and params["motion"]["target_shift"] == 120
    rng = np.random.default_rng(0)
    seq = rng.standard_normal((400, 219)).astype(np.float32)
    audio = rng.standard_normal((400, 35)).astype(np.float32)
    ex = {"motion_sequence": seq, "audio_sequence": audio, "motion_name": b"m", "audio_name": b"a"}
    tr = inputs.fact_preprocessing(ex, params, True, np.random.default_rng(1))
    assert tr["motion_input"].shape == (120, 225) and tr["target"].shape == (20, 225) and tr["audio_input"].shape == (240, 35)
    assert np.all(tr["motion_input"][:, :6] == 0)
    # locate the window: target must be the 20 frames that follow the 120 input frames, audio starts at the same frame
    start = int(np.where((seq == tr["motion_input"][0, 6:]).all(1))[0][0])
    assert 0 <= start <= 400 - 240
    assert np.array_equal(tr["motion_input"][:, 6:], seq[start:start + 120])
    assert np.array_equal(tr["target"][:, 6:], seq[start + 120:start + 140])
    assert np.array_equal(tr["audio_input"], audio[start:start + 240])
    ev = inputs.fact_preprocessing(ex, params, False)
    assert np.array_equal(ev["motion_input"][:, 6:], seq[:120]) and "target" not in ev
    assert ev["audio_input"].shape == (400, 35)               # eval keeps the whole track (inputs_util.py:104-105)


def test_create_input_train_and_eval(tmp_path):
    _write(tmp_path, "x_tfrecord-train-0", [(300, 300)] * 5)
    _write(tmp_path, "x_tfrecord-testval-0", [(300, 300), (280, 280), (290, 290)])
    cfg = config_util.get_configs_from_pipeline_file(
        config_util.DEFAULT_CONFIG,
        'train_dataset { data_files: "%s/*_tfrecord-train*" } eval_dataset { data_files: "%s/*_tfrecord-testval*" } '
        'train_config { batch_size: 4 }' % (tmp_path, tmp_path))
    it = inputs.create_input(cfg["train_config"], cfg["train_dataset"], is_training=True, seed=0)
    for _ in range(3):                                            # repeats forever, fixed shapes
        b = next(it)
        assert b["motion_input"].shape == (4, 120, 225) and b["audio_input"].shape == (4, 240, 35)
        assert b["target"].shape == (4, 20, 225) and len(b["motion_name"]) == 4
    ev = list(inputs.create_input(cfg["eval_config"], cfg["eval_dataset"], is_training=False))
    assert [e["audio_input"].shape for e in ev] == [(1, 300, 35), (1, 280, 35), (1, 290, 35)]   # ordered, batch 1
    assert ev[0]["motion_input"].shape == (1, 120, 225)


def test_fact_preprocessing_matches_the_references_own_code():
    """tests/golden/inputs_reference.npz: outputs of the reference's mint/utils/inputs_util.py (run over the TF shim)
    on a self-describing sequence, for forced window starts and for eval; the parameter dict comes from the
    reference's get_modality_to_param_dict on its pipeline_pb2 parse of the fact_v5 config."""
    import json
    import os
    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "inputs_reference.npz"))
    ref_params = json.loads(bytes(g["params_json"]).decode())
    cfg = config_util.get_configs_from_pipeline_file(config_util.DEFAULT_CONFIG)
    params = inputs.get_modality_to_param_dict(cfg["train_dataset"])
    for mod in ("motion", "audio"):
        for k in ("feature_dim", "input_length", "target_length", "target_shift"):
            assert params[mod][k] == ref_params[mod][k], (mod, k)
    seq, audio = g["motion_sequence"], g["audio_sequence"]
    lo, hi = g["uniform_bounds"][0]

    class Forced:
        def __init__(self, start):
            self.start, self.calls = start, []

        def integers(self, a, b=None):
            self.calls.append((a, b))
            return self.start

    for i, start in enumerate(g["starts"]):
        rng = Forced(int(start))
        ex = inputs.fact_preprocessing({"motion_sequence": seq, "audio_sequence": audio}, params, True, rng)
        assert rng.calls == [(int(lo), int(hi))]              # same draw range as tf.random.uniform([], 0, T - 240 + 1)
        for k in ("motion_input", "target", "audio_input"):
            assert ex[k].dtype == g[f"train{i}_{k}"].dtype
            np.testing.assert_array_equal(ex[k], g[f"train{i}_{k}"])
        assert "motion_sequence" not in ex and "audio_sequence" not in ex
    ev = inputs.fact_preprocessing({"motion_sequence": seq, "audio_sequence": audio}, params, False)
    np.testing.assert_array_equal(ev["motion_input"], g["eval_motion_input"])
    np.testing.assert_array_equal(ev["audio_input"], g["eval_audio_input"])
    assert "target" not in ev


# ---------------------------------------------------------------------------- pinned to TensorFlow-written record files
def _tfrecord_manifest():
    import json
    with open(os.path.join(os.path.dirname(__file__), "golden", "tfrecord_manifest.json")) as f:
        return json.load(f)


def test_masked_crc_matches_every_length_checksum_tensorflow_wrote():
    """14 TF-written known answers: masked crc32c of the 8-byte little-endian record length."""
    import struct
    man = _tfrecord_manifest()
    n = 0
    for info in man["files"].values():
        for rec in info["records"]:
            assert inputs.masked_crc(struct.pack("<Q", rec["length"])) == rec["length_masked_crc32c"]
            n += 1
    assert n == 14


def test_reader_and_writer_on_a_record_tensorflow_wrote(tmp_path):
    """tests/golden/tf_written_record.bin is one framed record copied bit for bit out of a TensorFlow-written file
    (tests/golden/make_tfrecord_golden.py): the reader verifies both checksums, the Example parser reproduces the
    manifest's feature table, and the writer re-frames the payload into the identical bytes."""
    import hashlib
    from tests.golden.make_tfrecord_golden import feature_summary
    man = _tfrecord_manifest()
    fx = man["fixture"]
    path = os.path.join(os.path.dirname(__file__), "golden", fx["path"])
    raw = open(path, "rb").read()
    assert hashlib.sha256(raw).hexdigest() == fx["sha256"]
    recs = list(inputs.read_tfrecords(path, verify_payload_crc=True))
    assert len(recs) == 1
    want = man["files"][fx["file"]]["records"][fx["record"]]
    assert len(recs[0]) == want["length"] and hashlib.sha256(recs[0]).hexdigest() == want["payload_sha256"]
    assert inputs.masked_crc(recs[0]) == want["payload_masked_crc32c"]
    got = {k: list(v) for k, v in feature_summary(recs[0]).items()}
    assert got == {k: list(v) for k, v in want["features"].items()}
    out = tmp_path / "again.record"
    with inputs.TFRecordWriter(str(out)) as w:
        w.write(recs[0])
    assert out.read_bytes() == raw
    # a flipped payload bit must be caught
    bad = bytearray(raw)
    bad[40] ^= 1
    (tmp_path / "bad.record").write_bytes(bytes(bad))
    with pytest.raises(IOError):
        list(inputs.read_tfrecords(str(tmp_path / "bad.record"), verify_payload_crc=True))


def test_every_record_of_the_tensorflow_written_sample(tmp_path):
    """tests/golden/tf_written_records.bin holds whole records of a TensorFlow-written file, framed as TensorFlow wrote
    them and in file order: the reader walks the stream with both checksums verified, every payload matches its
    manifest entry, and the writer re-frames the payloads into the identical stream."""
    import hashlib
    from tests.golden.make_tfrecord_golden import feature_summary
    man = _tfrecord_manifest()
    sample = man["sample"]
    path = os.path.join(os.path.dirname(__file__), "golden", sample["path"])
    raw = open(path, "rb").read()
    assert hashlib.sha256(raw).hexdigest() == sample["sha256"]
    recs = list(inputs.read_tfrecords(path, verify_payload_crc=True))
    assert len(recs) == len(sample["records"]) > 1
    for payload, i in zip(recs, sample["records"]):
        want = man["files"][sample["file"]]["records"][i]
        assert len(payload) == want["length"] and hashlib.sha256(payload).hexdigest() == want["payload_sha256"]
        assert inputs.masked_crc(payload) == want["payload_masked_crc32c"]
        assert {k: list(v) for k, v in feature_summary(payload).items()} == \
               {k: list(v) for k, v in want["features"].items()}
    out = tmp_path / "again.record"
    with inputs.TFRecordWriter(str(out)) as w:
        for payload in recs:
            w.write(payload)
    assert out.read_bytes() == raw
