"""Window-by-window comparison of large streams with the oracle (tools/stream_windows.py).

CPU part: the window logic itself, on oracle streams (whole stream vs the same chunks compressed
alone; port vs the compiled reference's recorded window streams).  GPU part: streams far larger
than anything a whole-stream oracle run could cover in seconds -- 9 GiB bf16 (the group-0 size table passes 2^32 at chunk 32768)
and 6 GiB fp32 (groups 2 and 3 start beyond 2^32) -- compared with the oracle on windows that
include the chunks around every 2^32 crossing (u64 size table, csrc/zipnn_core.c:145-153)."""
import hashlib

import numpy as np
import pytest

from golden_inputs import WINDOW_CASE, gauss_bytes, load_reference_checks, window_case_bytes
from oracle import oracle as O
from tools.stream_windows import StreamTables, check_stream_windows, compare_window


def _hdr():
    h = bytearray(32)
    h[0:2] = b"ZN"
    return h


@pytest.mark.parametrize("G,bits,chunk", [(2, 1, 4096), (4, 1, 65536), (1, 0, 131072), (2, 0, 262144)])
def test_windows_of_an_oracle_stream_match_the_chunks_compressed_alone(G, bits, chunk):
    rng = np.random.default_rng(5 + G)
    K = 37
    n = (K - 1) * chunk + (chunk // 2 // G) * G          # ragged last chunk
    data = gauss_bytes(rng, n, 2 if G <= 2 else 4)
    data[3 * chunk: 4 * chunk] = 0                        # an RLE chunk
    data[5 * chunk: 6 * chunk] = rng.integers(0, 256, chunk, dtype=np.uint8)   # an all-raw chunk
    bm = 220 if G == 4 else 10
    whole = O.zipnn_compress(_hdr(), data, G, bits, bm, chunk, 0.95, threads=4)

    def comp(win):
        return O.zipnn_compress(bytearray(40), win, G, bits, bm, chunk, 0.95, threads=2), 40

    res = check_stream_windows(whole, 32, G, K, chunk, n, lambda a, b: data[a:b], [(0, 5), (3, 7), (30, K), (0, K)], comp)
    assert res["windows"] == [[0, 5], [3, 7], [30, K], [0, K]]
    assert res["bytes_compared"] > whole.size            # overlapping windows: more than the stream once
    # a flipped payload byte inside a window must be noticed
    tab = StreamTables(whole, 32, G, K)
    bad = whole.copy()
    bad[int(tab.base[G - 1]) + int(tab.cum[G - 1, 3]) + 1] ^= 0x40
    with pytest.raises(AssertionError):
        check_stream_windows(bad, 32, G, K, chunk, n, lambda a, b: data[a:b], [(3, 7)], comp)


def test_windows_against_the_compiled_reference():
    """The reference's streams for two chunk ranges alone (recorded in golden/reference_checks.json) are
    windows of the port's whole stream."""
    want = load_reference_checks()
    data = window_case_bytes()
    assert hashlib.sha256(data.tobytes()).hexdigest() == want["window_input_sha256"], "input generator drifted"
    chunk, G, K = WINDOW_CASE["chunk"], WINDOW_CASE["G"], WINDOW_CASE["K"]
    whole = O.zipnn_compress(_hdr(), data, G, 1, 10, chunk, 0.95, threads=4)
    tab = StreamTables(whole, 32, G, K)
    for (c0, c1), rec in zip(WINDOW_CASE["windows"], want["windows"], strict=True):
        assert rec["chunks"] == [c0, c1]
        # the port's stream for the window equals the reference's, so it can stand in for it
        r = O.zipnn_compress(_hdr(), data[c0 * chunk: c1 * chunk], G, 1, 10, chunk, 0.95, threads=4)
        assert (r.size, hashlib.sha256(r.tobytes()).hexdigest()) == (rec["stream_len"], rec["stream_sha256"])
        assert compare_window(tab, c0, c1, r, 32) > 0


@pytest.mark.gpu
@pytest.mark.parametrize("dtype_name,gib", [("bfloat16", 9), ("float32", 6)])
def test_large_gpu_stream_matches_oracle_window_by_window(dtype_name, gib):
    import torch
    from zipnn_b200 import ZipNN
    dtype = getattr(torch, dtype_name)
    esz = torch.empty(0, dtype=dtype).element_size()
    nbytes = gib << 30
    free, _ = torch.cuda.mem_get_info()
    if free < 2.4 * nbytes + (4 << 30):
        pytest.skip("not enough device memory for this size")
    g = torch.Generator(device="cuda").manual_seed(77 + gib)
    t = torch.empty(nbytes // esz, dtype=dtype, device="cuda")
    slab = 1 << 27
    for i in range(0, t.numel(), slab):
        m = min(slab, t.numel() - i)
        t[i:i + m] = (torch.randn(m, generator=g, device="cuda", dtype=torch.float32) * 0.02).to(dtype)
    # a few chunks of the other item kinds inside the windows that get compared
    tb = t.view(torch.uint8)
    chunk = 262144
    tb[7 * chunk: 8 * chunk] = 0
    tb[9 * chunk: 10 * chunk] = torch.randint(0, 256, (chunk,), dtype=torch.uint8, device="cuda", generator=g)
    z = ZipNN(input_format="torch")
    stream = z.compress(t)
    plan = z._last_plan
    G, hdr_len = plan["num_buf"], len(plan["header"])
    K = (nbytes + chunk - 1) // chunk
    tab = StreamTables(stream, hdr_len, G, K)
    assert tab.total == stream.numel()
    wins = [(0, 96), (K - 64, K)]
    crossings = 0
    for grp in range(G):
        lim = 1 << 32
        if int(tab.base[grp]) < lim:
            cx = tab.first_chunk_past(grp, lim - int(tab.base[grp]))
            if 0 < cx < K:
                wins.append((cx - 48, cx + 48))
                crossings += 1
        else:
            crossings += 1                                  # the whole group lies beyond 2^32
            wins.append((K // 2 - 16, K // 2 + 16))
        cy = tab.first_chunk_past(grp, lim)
        if 0 < cy < K:
            wins.append((cy - 48, cy + 48))
            crossings += 1
    assert crossings >= 1, "this size was chosen to have offsets beyond 2^32"

    def comp(win):
        return O.zipnn_compress(bytearray(32), win, G, plan["bit_reorder"], plan["byte_reorder"], chunk, plan["threshold"], threads=8), 32

    res = check_stream_windows(stream, hdr_len, G, K, chunk, nbytes, lambda a, b: tb[a:b].cpu().numpy(), wins, comp)
    assert res["max_stream_offset"] > (1 << 32)
    assert res["bytes_compared"] > 32 << 20
    back = ZipNN(input_format="torch").decompress(stream)
    assert torch.equal(back.view(torch.uint8), tb)
