"""The bit-packer (k_encode_write_warp and the ragged-tail k_encode_write) against the oracle, byte for byte,
on inputs built to reach its edge cases:

- coded planes whose symbols are mostly rare ones in whole stretches of every bitstream, so that the
  length-limited Huffman table gives them the longest codes (11 bits) and every lane of a tile builds
  runs of the worst-case length;
- every destination alignment of the four bitstreams (a = 0..3) and of the raw plane quarters (0..15),
  obtained by stepping the header length over 32..47 bytes behind payloads of varying sizes;
- chunk sizes 1024 .. 262144, a short last chunk that still takes the warp kernel with a tile count
  that is not a power of two, and a ragged last chunk;
- G = 1, 2, 4 with bits = 0 and 1, raw, RLE and coded planes at every group index.
"""
import ctypes as C

import numpy as np
import pytest
import torch

from oracle import oracle as O
from zipnn_b200 import _native

pytestmark = pytest.mark.gpu


def _plane(rng, kind, n):
    if kind == 0:
        # coded: four frequent bytes (1- to 3-bit codes take 15/16 of the code space), and a sixteenth of every
        # quarter made of the other 252, which get the longest codes the table allows (11 bits)
        p = rng.choice(np.array([0x3C, 0x3D, 0x3E, 0x3F], dtype=np.uint8), n, p=[0.5, 0.25, 0.125, 0.125])
        q = max(n // 4, 1)
        for s in range(4):
            a = s * q
            b = min(n, a + max(q // 16, 1))
            p[a:b] = rng.integers(0, 256, b - a, dtype=np.uint8)
        return p
    if kind == 1:  # incompressible: stays raw
        return rng.integers(0, 256, n, dtype=np.uint8)
    return np.full(n, 0xA5, dtype=np.uint8)  # one byte: RLE


def _input(rng, G, chunk, n):
    """Chunk c, plane g gets kind (c + g) % 3 (coded, raw, RLE)."""
    out = np.empty(n, dtype=np.uint8)
    for c0 in range(0, n, chunk):
        m = min(chunk, n - c0)
        ci = c0 // chunk
        for g in range(G):
            idx = np.arange(g, m, G)
            out[c0 + idx] = _plane(rng, (ci + g) % 3, idx.size)
    return out


def _compress(L, d_in, n, hdr, G, bits, bm, chunk):
    bound = _native.compress_bound(n, G, chunk, len(hdr))
    d_out = torch.zeros(bound, dtype=torch.uint8, device="cuda")
    ws = torch.empty(_native.compress_workspace_size(n, G, chunk), dtype=torch.uint8, device="cuda")
    out_len = C.c_size_t(0)
    hbuf = (C.c_char * len(hdr)).from_buffer_copy(bytes(hdr))
    st = L.zipnn_b200_compress(d_in.data_ptr(), n, hbuf, len(hdr), G, bits, bm, chunk, 0.95, d_out.data_ptr(), bound,
                               C.byref(out_len), ws.data_ptr(), ws.numel(), torch.cuda.current_stream().cuda_stream)
    assert st == 0, st
    return d_out[: out_len.value]


def _decompress(L, body, n, G, bits, bm, chunk):
    d_dec = torch.zeros(n + 16, dtype=torch.uint8, device="cuda")
    ws = torch.empty(_native.decompress_workspace_size(n, G, chunk), dtype=torch.uint8, device="cuda")
    st = L.zipnn_b200_decompress(body.data_ptr(), body.numel(), G, bits, bm, chunk, n, d_dec.data_ptr(), ws.data_ptr(),
                                 ws.numel(), torch.cuda.current_stream().cuda_stream, 1)
    assert st == 0, st
    return d_dec[:n].cpu().numpy()


@pytest.mark.parametrize("chunk", [1024, 4096, 65536, 262144])
@pytest.mark.parametrize("G,bits", [(1, 0), (1, 1), (2, 0), (2, 1), (4, 0), (4, 1)])
def test_packer_matches_oracle(G, bits, chunk):
    rng = np.random.default_rng(7 + 100 * G + 10 * bits + chunk)
    L = _native.lib()
    bm = 220 if G == 4 else 10
    # last chunk: 4 * G * 2576 bytes = three warp steps of 1024 plane bytes per bitstream, the first
    # one holding 528 (less when the chunk is small), then the same plus a ragged 3 * G bytes
    short = 4 * G * 2576 if 4 * G * 2576 < chunk else chunk // 2 + 64 * G
    for n in (3 * chunk, 3 * chunk + short, 3 * chunk + short + 3 * G):
        data = _input(rng, G, chunk, n)
        d_in = torch.from_numpy(data.copy()).cuda()
        for hl in range(32, 48):
            hdr = bytearray(hl)
            hdr[0:2] = b"ZN"
            want = O.zipnn_compress(hdr, data, G, bits, bm, chunk, 0.95, threads=4)
            got = _compress(L, d_in, n, hdr, G, bits, bm, chunk)
            assert got.numel() == want.size, (n, hl, got.numel(), want.size)
            assert np.array_equal(got.cpu().numpy(), want), (n, hl)
            if hl in (32, 47):
                back = _decompress(L, got[hl:].contiguous(), n, G, bits, bm, chunk)
                assert np.array_equal(back, data), (n, hl)
        # the inputs reach both paths (type bytes follow the header): coded planes unless they are over
        # 128 KiB (always raw, huf_compress.c:658); raw planes unless the sign-bit rotation (bits = 1) has
        # moved structure into the random ones
        types = want[hl: hl + G * ((n + chunk - 1) // chunk)]
        if bits == 0:
            assert (types == 0).any()
        if chunk // G <= 131072:
            assert (types == 1).any()
