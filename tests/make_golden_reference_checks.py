#!/usr/bin/env python3
"""Record the compiled reference's answers for the cross-checks in test_oracle.py and
test_stream_windows.py as tests/golden/reference_checks.json.

Needs the UNMODIFIED reference C extension in oracle/_ref (`make -C oracle ref REF=<reference
checkout>`).  The inputs are regenerated from seeds (golden_inputs.py); for every case the file
holds the input's sha256 and the length and sha256 of what the reference produced, so the tests
compare the oracle port with the reference byte for byte without the reference being present.

usage:  python tests/make_golden_reference_checks.py
"""
import hashlib
import json
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, HERE)

import numpy as np  # noqa: E402

from golden_inputs import REFERENCE_CHECKS, WINDOW_CASE, huf_block_cases, stream_cases, window_case_bytes  # noqa: E402
from oracle import oracle as O  # noqa: E402


def sha(b) -> str:
    return hashlib.sha256(bytes(b)).hexdigest()


def hdr():
    h = bytearray(32)
    h[0:2] = b"ZN"
    return h


def main():
    ref, cdll = O.ref_core(), O.ref_cdll()
    if ref is None or cdll is None:
        sys.exit("oracle/_ref is not built: make -C oracle ref REF=<reference checkout>")
    blocks = []
    for src, cap in huf_block_cases():
        r, out = O.ref_huf_compress(src, cap)
        blocks.append(dict(input_sha256=sha(src), ret=int(r), out_sha256=sha(out)))
    streams = []
    for data, G, bits, bm, chunk in stream_cases():
        n = data.size
        r = bytes(ref.zipnn_core(bytes(hdr()), bytearray(data.tobytes()), G, bits, bm, 0, chunk, 0.95, 10, 4))
        assert bytes(ref.combine_dtype(r[32:], G, bits, bm, chunk, n, 2)) == data.tobytes()
        streams.append(dict(input_sha256=sha(data), stream_len=len(r), stream_sha256=sha(r)))
    data = window_case_bytes()
    chunk = WINDOW_CASE["chunk"]
    windows = []
    for c0, c1 in WINDOW_CASE["windows"]:
        r = bytes(ref.zipnn_core(bytes(hdr()), bytearray(data[c0 * chunk: c1 * chunk].tobytes()), WINDOW_CASE["G"], 1, 10, 0,
                                 chunk, 0.95, 10, 4))
        windows.append(dict(chunks=[c0, c1], stream_len=len(r), stream_sha256=sha(r)))
    with open(REFERENCE_CHECKS, "w") as f:
        json.dump(dict(reference="zipnn/zipnn v0.5.3 (0e9beed), C extension built -O3", numpy=np.__version__,
                       window_input_sha256=sha(data), huf_blocks=blocks, streams=streams, windows=windows), f, indent=1)
    print(f"wrote {len(blocks)} blocks, {len(streams)} streams, {len(windows)} windows to {REFERENCE_CHECKS}")


if __name__ == "__main__":
    main()
