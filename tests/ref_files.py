"""The reference's own JPEG files kept under tests/golden/ref/.

manifest.json records the length and SHA-256 of each reference file.  The digests were taken from these copies
while they were being checked byte for byte against the reference tree, so they pin the copies to the files as
they were then.  A file whose tail after the EOI marker is zero padding is stored without that tail; read() puts
the recorded length back, so every reader sees the reference's bytes."""
import json
import os

DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref")
with open(os.path.join(DIR, "manifest.json")) as _f:
    MANIFEST = json.load(_f)
NAMES = sorted(MANIFEST)


def read(name: str) -> bytes:
    """the reference file `name`: the stored copy, zero-padded to the recorded length"""
    with open(os.path.join(DIR, name), "rb") as f:
        data = f.read()
    pad = MANIFEST[name]["bytes"] - len(data)
    if pad < 0:
        raise ValueError(f"{name}: stored copy is longer than the reference file")
    return data + bytes(pad)
