"""Payload bits of the reference scripts as a golden INPUT vector -> tests/golden/eagle_bits.bin.

`file_reader('eagle.tiff', n)` (`Task 5/file_reader.m:2-12`: imread -> imbinarize -> first n entries, column-major)
restated by `oracle.chains.read_payload_bits`; 129,600 bits packed MSB-first (numpy.packbits) = 16,200 bytes.  Needs
the image from a checkout of the reference (it is not copied into this repository); the tests read the committed file.
`eagle_bits_digest.json` holds the SHA-256 of exactly these bytes.

    python tests/golden/make_eagle_bits.py "<reference checkout>/Task 5/eagle.tiff"
"""
import hashlib
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
from oracle import chains as OC  # noqa: E402

if __name__ == "__main__":
    b = OC.read_payload_bits(sys.argv[1], 129600)
    raw = np.packbits(b).tobytes()
    want = json.load(open(os.path.join(HERE, "eagle_bits_digest.json")))["sha256_of_packbits"]
    assert hashlib.sha256(raw).hexdigest() == want
    open(os.path.join(HERE, "eagle_bits.bin"), "wb").write(raw)
    print(len(raw), "bytes written")
