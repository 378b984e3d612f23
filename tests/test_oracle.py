"""The oracle (our C restatement) against the reference: committed golden streams, and the
compiled reference's answers on seeded blocks and streams (golden/reference_checks.json).  CPU only."""
import hashlib

import numpy as np
import pytest

from conftest import golden_stream, load_manifest
from golden_inputs import huf_block_cases, load_reference_checks, make_input, raw_bytes, stream_cases
from oracle import oracle as O
from zipnn_b200 import ZipNN

CASES = load_manifest()
REF = load_reference_checks()


def sha(b):
    return hashlib.sha256(bytes(b)).hexdigest()


@pytest.mark.parametrize("rec", CASES, ids=[c["name"] for c in CASES])
def test_port_reproduces_reference_stream(rec):
    data = make_input(rec["input"])
    raw = raw_bytes(data)
    if sha(raw) != rec["input_sha256"]:
        pytest.skip("input generator drifted on this machine (numpy/torch RNG or cast)")
    z = ZipNN(**rec["ctor"])
    plan = z.plan(data if rec["ctor"]["input_format"] == "torch" else raw)
    assert plan["header"][:24].hex() == rec["header_hex"][:48]
    stream = O.zipnn_compress(plan["header"], np.frombuffer(raw, dtype=np.uint8), plan["num_buf"], plan["bit_reorder"],
                              plan["byte_reorder"], plan["chunk"], plan["threshold"], threads=4).tobytes()
    assert len(stream) == rec["stream_len"]
    assert sha(stream) == rec["stream_sha256"]
    gold = golden_stream(rec)
    if gold is not None:
        assert stream == gold
    body = np.frombuffer(stream, dtype=np.uint8)[len(plan["header"]):]
    back = O.zipnn_decompress(body, plan["num_buf"], plan["bit_reorder"], plan["byte_reorder"], plan["chunk"], len(raw), threads=4)
    assert back.tobytes() == raw


def test_port_matches_compiled_reference_blocks():
    for i, ((src, cap), want) in enumerate(zip(huf_block_cases(), REF["huf_blocks"], strict=True)):
        assert sha(src) == want["input_sha256"], f"block {i}: input generator drifted"
        r, out = O.huf_compress(src, cap)
        assert (r, sha(out)) == (want["ret"], want["out_sha256"]), f"block {i}: {src.size} bytes, cap {cap}"


def test_port_matches_compiled_reference_streams():
    h = bytearray(32)
    h[0:2] = b"ZN"
    for i, ((data, G, bits, bm, chunk), want) in enumerate(zip(stream_cases(), REF["streams"], strict=True)):
        assert sha(data) == want["input_sha256"], f"stream {i}: input generator drifted"
        o = O.zipnn_compress(h, data, G, bits, bm, chunk, 0.95, threads=2).tobytes()
        assert (len(o), sha(o)) == (want["stream_len"], want["stream_sha256"]), f"stream {i}: G={G} bits={bits} chunk={chunk} n={data.size}"
        assert O.zipnn_decompress(np.frombuffer(o, dtype=np.uint8)[32:], G, bits, bm, chunk, data.size, threads=2).tobytes() == data.tobytes()
