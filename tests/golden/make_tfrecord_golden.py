#!/usr/bin/env python
"""Golden for the TFRecord reader / tf.train.Example parser of mint_b200/inputs.py from record files WRITTEN BY
TENSORFLOW that ship inside the reference tree (third_party/tf_models test data: 10 + 1 + 3 records).

Build container only (reads /root/reference).  With this repo's reader -- length AND payload checksums verified --
it walks every record and commits
  * tfrecord_manifest.json : per file sha256 / size / record count; per record: payload length, the two masked
    crc32c values TensorFlow stored (TF-written known answers for masked_crc), sha256 of the payload, and per feature
    key: kind, value count, sha256 of the canonical value bytes;
  * tf_written_record.bin : ONE framed record (the smallest, 11 KB: length | crc | payload | crc) exactly as TensorFlow
    wrote it, so that the GPU box (no /root/reference) still reads TensorFlow-written bytes, and the writer can be
    required to reproduce the frame byte for byte;
  * tf_written_records.bin : the SAMPLE_RECORDS smallest records of the first file, framed exactly as TensorFlow wrote
    them and kept in file order (64 KB), so that the tests read a multi-record stream of TensorFlow-written bytes
    without the source files (the three files hold 2.8 MB of mostly compressed images).

    python tests/golden/make_tfrecord_golden.py
"""
import hashlib
import json
import os
import struct
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
from mint_b200 import inputs as I  # noqa: E402

BASE = "/root/reference/third_party/tf_models/research/"
FILES = ["object_detection/test_data/pets_examples.record",
         "object_detection/test_data/snapshot_serengeti_sequence_examples.record",
         "deeplab/testing/pascal_voc_seg/val-00000-of-00001.tfrecord"]
HERE = os.path.dirname(os.path.abspath(__file__))
SAMPLE_RECORDS = 4


def feature_summary(payload: bytes) -> dict:
    """key -> [kind, count, sha256 of the values in a canonical byte form]."""
    ex = I.Example.FromString(payload)
    out = {}
    for key, feat in sorted(ex.features.feature.items()):
        kind = feat.WhichOneof("kind")
        if kind == "bytes_list":
            vals = list(feat.bytes_list.value)
            raw = b"".join(struct.pack("<Q", len(v)) + v for v in vals)
        elif kind == "float_list":
            vals = feat.float_list.value
            raw = np.asarray(vals, "<f4").tobytes()
        elif kind == "int64_list":
            vals = feat.int64_list.value
            raw = np.asarray(vals, "<i8").tobytes()
        else:
            vals, raw = [], b""
        out[key] = [kind, len(vals), hashlib.sha256(raw).hexdigest()]
    return out


def frames(path):
    """(header, stored length crc, payload, stored payload crc) for every record, checksums verified."""
    data = open(path, "rb").read()
    pos = 0
    while pos < len(data):
        header = data[pos:pos + 8]
        (n,) = struct.unpack("<Q", header)
        (lcrc,) = struct.unpack("<I", data[pos + 8:pos + 12])
        payload = data[pos + 12:pos + 12 + n]
        (pcrc,) = struct.unpack("<I", data[pos + 12 + n:pos + 16 + n])
        assert lcrc == I.masked_crc(header) and pcrc == I.masked_crc(payload)
        yield header, lcrc, payload, pcrc
        pos += 16 + n


def main():
    manifest = {"source_root": BASE, "files": {}}
    smallest = None
    framed = {}
    for rel in FILES:
        path = BASE + rel
        raw = open(path, "rb").read()
        recs = []
        via_reader = list(I.read_tfrecords(path, verify_payload_crc=True))
        for i, (header, lcrc, payload, pcrc) in enumerate(frames(path)):
            assert payload == via_reader[i]
            framed[rel, i] = header + struct.pack("<I", lcrc) + payload + struct.pack("<I", pcrc)
            recs.append({"length": len(payload), "length_masked_crc32c": lcrc, "payload_masked_crc32c": pcrc,
                         "payload_sha256": hashlib.sha256(payload).hexdigest(), "features": feature_summary(payload)})
            if smallest is None or len(payload) < len(smallest[2]):
                smallest = (rel, i, payload, header + struct.pack("<I", lcrc) + payload + struct.pack("<I", pcrc))
        assert len(via_reader) == len(recs)
        manifest["files"][rel] = {"sha256": hashlib.sha256(raw).hexdigest(), "bytes": len(raw), "records": recs}
    manifest["fixture"] = {"file": smallest[0], "record": smallest[1], "path": "tf_written_record.bin",
                           "sha256": hashlib.sha256(smallest[3]).hexdigest()}
    with open(os.path.join(HERE, "tf_written_record.bin"), "wb") as f:
        f.write(smallest[3])
    first = manifest["files"][FILES[0]]["records"]
    picked = sorted(sorted(range(len(first)), key=lambda i: first[i]["length"])[:SAMPLE_RECORDS])
    sample = b"".join(framed[FILES[0], i] for i in picked)
    manifest["sample"] = {"file": FILES[0], "records": picked, "path": "tf_written_records.bin",
                          "sha256": hashlib.sha256(sample).hexdigest()}
    with open(os.path.join(HERE, "tf_written_records.bin"), "wb") as f:
        f.write(sample)
    with open(os.path.join(HERE, "tfrecord_manifest.json"), "w") as f:
        json.dump(manifest, f, indent=1)
    print({k: len(v["records"]) for k, v in manifest["files"].items()}, manifest["fixture"], manifest["sample"])


if __name__ == "__main__":
    main()
