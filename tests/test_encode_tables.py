"""Pass A of compress (k_encode_hist, k_encode_table) against the oracle, byte for byte, on byte planes built
to reach every branch of the block decision and of the table description:

- the six distribution families of test_device_serial_routines_match_oracle;
- trees deeper than 11 bits (geometric and Fibonacci-like counts), so the depth limit repays its debt;
- both table-description forms (tANS weights and nibbles) and the raw fallback of a wide alphabet;
- single-symbol (RLE) planes and two-symbol planes;
- the "not compressible" early-out with the largest count exactly at and one above (plen >> 7) + 4;
- G = 1, 2, 4 with bits = 0 and 1, and a ragged last chunk (the histogram's byte-wise path);
- a stream quarter of one byte value, whose count (32768) fills the 16-bit half of a folded counter.

The GPU tests compare the whole stream with the oracle and decode it back; the CPU test checks, with the
oracle alone, that the inputs do reach each of those forms.
"""
import ctypes as C

import numpy as np
import pytest
import torch

from oracle import oracle as O

N_CASES = 16


def _spread(rng, counts):
    """A plane holding counts[i] copies of symbol sym[i], shuffled; symbols scattered over 0..255."""
    syms = (np.arange(len(counts)) * 37 + 11) % 256
    p = np.repeat(syms.astype(np.uint8), counts)
    rng.shuffle(p)
    return p


def _plane(rng, case, m):
    if case == 0:  # f32 exponents of small normals
        x = (rng.standard_normal(m) * 0.02).astype(np.float32)
        return (x.view(np.uint32) >> 23).astype(np.uint8)
    if case == 1:
        k = int(rng.integers(2, 20))
        return rng.choice(k, m, p=rng.dirichlet(np.ones(k) * rng.uniform(0.05, 2))).astype(np.uint8)
    if case == 2:
        k = int(rng.integers(2, 256))
        return rng.choice(k, m, p=rng.dirichlet(np.ones(k) * rng.uniform(0.01, 1))).astype(np.uint8)
    if case == 3:
        return np.minimum(rng.geometric(rng.uniform(0.02, 0.9), m), 255).astype(np.uint8)
    if case == 4:
        return (rng.standard_normal(m) * rng.uniform(0.5, 40) + 128).clip(0, 255).astype(np.uint8)
    if case == 5:
        return np.minimum(rng.zipf(rng.uniform(1.1, 3), m), 255).astype(np.uint8)
    if case in (6, 7):  # deep trees: halving or Fibonacci-like counts down to 1
        r = 2.0 if case == 6 else 1.618
        c = np.maximum((m * (r - 1) / r) / r ** np.arange(40), 1).astype(np.int64)
        c = c[: int(np.searchsorted(-c, -1, side="right")) + 3]
        c[0] += m - c.sum()
        return _spread(rng, c)
    if case == 8:  # RLE
        return np.full(m, int(rng.integers(0, 256)), dtype=np.uint8)
    if case == 9:  # two symbols
        return np.where(rng.random(m) < rng.uniform(0.5, 0.99), 0x40, 0x41).astype(np.uint8)
    if case == 10:  # two symbols, one of them once
        p = np.full(m, 0x7F, dtype=np.uint8)
        p[int(rng.integers(0, m))] = 0x80
        return p
    if case in (11, 12):  # largest count at / one above the "not compressible" limit
        top = (m >> 7) + 4 + (case - 11)
        rest = m - top
        c = np.full(256, rest // 255, dtype=np.int64)
        c[0] = top
        c[1: 1 + rest % 255] += 1
        return _spread(rng, c)
    if case == 13:  # wide, nearly flat alphabet: weights do not pay in tANS and do not fit the nibble form
        return rng.choice(256, m, p=rng.dirichlet(np.ones(256) * 40)).astype(np.uint8)
    if case == 14:  # incompressible
        return rng.integers(0, 256, m, dtype=np.uint8)
    # few symbols low in the alphabet: nibble form
    k = int(rng.integers(3, 9))
    return rng.choice(k, m, p=rng.dirichlet(np.ones(k))).astype(np.uint8) * 3


def _input(rng, G, chunk, n, first_case=0):
    """Plane g of chunk c gets case (first_case + c * G + g) % N_CASES."""
    out = np.empty(n, dtype=np.uint8)
    for c0 in range(0, n, chunk):
        m = min(chunk, n - c0)
        for g in range(G):
            idx = np.arange(g, m, G)
            out[c0 + idx] = _plane(rng, (first_case + (c0 // chunk) * G + g) % N_CASES, idx.size)
    return out


def _forms(stream, hl, G, K):
    """Kind of every item's block: raw, rle, tans or nibble."""
    nitems = G * K
    types = stream[hl: hl + nitems]
    cum = stream[hl + nitems: hl + 9 * nitems].view("<u8")
    out = set()
    base = hl + 9 * nitems
    for g in range(G):
        prev = 0
        for c in range(K):
            i = g * K + c
            size = int(cum[i]) - prev
            if types[i] == 0:
                out.add("raw")
            elif size == 1:
                out.add("rle")
            else:
                out.add("tans" if stream[base + prev] < 128 else "nibble")
            prev = int(cum[i])
        base += prev
    return out


def _case_input(G, bits, chunk):
    rng = np.random.default_rng(31 + 100 * G + 10 * bits)
    n = 2 * N_CASES * chunk + 77 * G  # every case at every group index, then a ragged last chunk
    return _input(rng, G, chunk, n), n


CHUNK = 65536
PARAMS = [(1, 0), (1, 1), (2, 0), (2, 1), (4, 0), (4, 1)]


def test_inputs_reach_every_form():
    """CPU: the oracle's streams for the GPU test inputs hold raw, RLE, tANS and nibble blocks."""
    hdr = bytearray(32)
    seen = set()
    for G, bits in PARAMS:
        data, n = _case_input(G, bits, CHUNK)
        want = O.zipnn_compress(hdr, data, G, bits, 220 if G == 4 else 10, CHUNK, 0.95, threads=4)
        seen |= _forms(want, 32, G, (n + CHUNK - 1) // CHUNK)
    assert seen == {"raw", "rle", "tans", "nibble"}, seen


def _roundtrip(G, bits, chunk, data):
    from zipnn_b200 import _native
    L = _native.lib()
    n = data.size
    bm = 220 if G == 4 else 10
    hdr = bytearray(32)
    hdr[0:2] = b"ZN"
    want = O.zipnn_compress(hdr, data, G, bits, bm, chunk, 0.95, threads=4)
    d_in = torch.from_numpy(data.copy()).cuda()
    bound = _native.compress_bound(n, G, chunk, len(hdr))
    d_out = torch.zeros(bound, dtype=torch.uint8, device="cuda")
    ws = torch.empty(_native.compress_workspace_size(n, G, chunk), dtype=torch.uint8, device="cuda")
    out_len = C.c_size_t(0)
    hbuf = (C.c_char * len(hdr)).from_buffer_copy(bytes(hdr))
    st = L.zipnn_b200_compress(d_in.data_ptr(), n, hbuf, len(hdr), G, bits, bm, chunk, 0.95, d_out.data_ptr(), bound,
                               C.byref(out_len), ws.data_ptr(), ws.numel(), torch.cuda.current_stream().cuda_stream)
    assert st == 0, st
    got = d_out[: out_len.value].cpu().numpy()
    assert got.size == want.size, (got.size, want.size)
    assert np.array_equal(got, want)
    body = d_out[len(hdr): out_len.value].contiguous()
    d_dec = torch.zeros(n + 16, dtype=torch.uint8, device="cuda")
    ws = torch.empty(_native.decompress_workspace_size(n, G, chunk), dtype=torch.uint8, device="cuda")
    st = L.zipnn_b200_decompress(body.data_ptr(), body.numel(), G, bits, bm, chunk, n, d_dec.data_ptr(), ws.data_ptr(),
                                 ws.numel(), torch.cuda.current_stream().cuda_stream, 1)
    assert st == 0, st
    assert np.array_equal(d_dec[:n].cpu().numpy(), data)


@pytest.mark.gpu
@pytest.mark.parametrize("G,bits", PARAMS)
def test_tables_match_oracle(G, bits):
    data, _ = _case_input(G, bits, CHUNK)
    _roundtrip(G, bits, CHUNK, data)


@pytest.mark.gpu
@pytest.mark.parametrize("G", [1, 2])
def test_full_quarter_of_one_byte(G):
    """Planes of 128 KiB whose first stream quarter is one byte value (a count of 32768 in one quarter),
    then coded, raw and RLE remainders."""
    chunk = 131072 * G
    rng = np.random.default_rng(5 + G)
    data = _input(rng, G, chunk, 3 * chunk, first_case=3)
    for c in range(3):
        for g in range(G):
            plane = data[c * chunk + g: (c + 1) * chunk: G]
            plane[: plane.size // 4] = 0x3C + c
            data[c * chunk + g: (c + 1) * chunk: G] = plane
    _roundtrip(G, 0, chunk, data)
