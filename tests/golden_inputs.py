"""Deterministic input generators shared by the golden generators (make_golden*.py) and the tests.

Inputs are regenerated from a seed rather than committed; each manifest record
carries the input sha256 so a test can tell "generator drifted" (skip) from
"codec wrong" (fail).
"""
import json
import os

import numpy as np
import torch

_TORCH_DT = {
    "bfloat16": torch.bfloat16, "float16": torch.float16, "float32": torch.float32,
    "float8_e4m3fn": torch.float8_e4m3fn, "float8_e5m2": torch.float8_e5m2, "uint8": torch.uint8,
}


def torch_dtype(name: str):
    return _TORCH_DT[name]


def make_input(spec: dict):
    """-> torch tensor for float dtypes, bytes for dtype == 'uint8'."""
    gen, n = spec["gen"], spec["n"]
    rng = np.random.default_rng(spec.get("seed", 1234))
    dt = _TORCH_DT[spec["dtype"]]
    if gen == "randn":
        x = rng.standard_normal(n, dtype=np.float32) * np.float32(spec["sigma"])
        t = torch.from_numpy(x).to(dt)
    elif gen == "rand_pm1":
        x = (rng.random(n, dtype=np.float32) * np.float32(2) - np.float32(1))
        t = torch.from_numpy(x).to(dt)
    elif gen == "randn_bf16_as_fp32":
        x = rng.standard_normal(n, dtype=np.float32) * np.float32(spec["sigma"])
        t = torch.from_numpy(x).to(torch.bfloat16).to(torch.float32)
    elif gen == "zeros_ones":
        t = torch.cat([torch.zeros(n // 2, dtype=dt), torch.ones(n - n // 2, dtype=dt)])
    elif gen == "choice":
        p = np.asarray(spec["p"], dtype=np.float64)
        return rng.choice(len(p), n, p=p / p.sum()).astype(np.uint8).tobytes()
    elif gen == "bytes":
        return rng.integers(0, 256, n, dtype=np.uint8).tobytes()
    elif gen == "half_zero":
        b = rng.integers(0, 256, n, dtype=np.uint8)
        b[rng.random(n) >= spec["frac"]] = 0
        return b.tobytes()
    else:
        raise ValueError(gen)
    if "shape" in spec:
        t = t.reshape(spec["shape"])
    return t


def raw_bytes(data) -> bytes:
    if isinstance(data, (bytes, bytearray)):
        return bytes(data)
    if data.numel() == 0:
        return b""
    return data.contiguous().reshape(-1).view(torch.uint8).numpy().tobytes()


# ---- inputs of the checks against the compiled reference (make_golden_reference_checks.py records
#      the reference's answers for them in golden/reference_checks.json)
REFERENCE_CHECKS = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_checks.json")


def load_reference_checks() -> dict:
    with open(REFERENCE_CHECKS) as f:
        return json.load(f)


def gauss_bytes(rng, n, esz):
    """n bytes of randn*0.02 as bf16 (esz 2) or fp32 (esz 4)."""
    x = (rng.standard_normal(n // esz + 2) * 0.02).astype(np.float32)
    if esz == 2:
        return np.ascontiguousarray((x.view(np.uint32) >> 16).astype(np.uint16).view(np.uint8)[:n])
    return np.ascontiguousarray(x.view(np.uint8)[:n])


def huf_block_cases():
    """-> [(src uint8 array, dst capacity)]: single HUF blocks of every symbol distribution the codec meets."""
    rng = np.random.default_rng(3)
    cases = []
    for it in range(300):
        size = int(rng.choice([12, 13, 64, 257, 1500, 4096, 65536, 131072, int(rng.integers(1, 131073))]))
        kind = it % 5
        if kind == 0:
            x = (rng.standard_normal(size) * 0.02).astype(np.float32)
            src = (x.view(np.uint32) >> 23).astype(np.uint8)
        elif kind == 1:
            src = rng.integers(0, 256, size, dtype=np.uint8)
        elif kind == 2:
            k = int(rng.integers(2, 256))
            src = rng.choice(k, size, p=rng.dirichlet(np.ones(k) * rng.uniform(0.01, 1))).astype(np.uint8)
        elif kind == 3:
            src = np.full(size, 7, dtype=np.uint8)
        else:
            src = np.minimum(rng.geometric(rng.uniform(0.02, 0.9), size), 255).astype(np.uint8)
        cases.append((src, 256 * 1024 if it % 2 else 128 * 1024))
    return cases


def stream_cases():
    """-> [(data uint8 array, num_buf, bits_mode, bytes_mode, chunk)]: whole streams over layouts and sizes."""
    rng = np.random.default_rng(11)
    cases = []
    for it in range(40):
        G = [1, 2, 4][it % 3]
        bits = (it // 3) % 2
        bm = 220 if G == 4 else 10
        chunk = 128 * 1024 if G == 1 else int(rng.choice([256 * 1024, 65536, 4096]))
        nelem = int(rng.choice([1, 3, 13, 4096, chunk // G + 1, int(rng.integers(1, 200000))]))
        n = nelem * G
        if it % 4 == 3:
            data = rng.integers(0, 256, n, dtype=np.uint8)
        else:
            x = (rng.standard_normal(max(n // 2, 1) + 2) * 0.02).astype(np.float32)
            data = np.ascontiguousarray((x.view(np.uint32) >> 16).astype(np.uint16).view(np.uint8)[:n])
        cases.append((data, G, bits, bm, chunk))
    return cases


WINDOW_CASE = dict(chunk=262144, G=2, K=9, windows=[(0, 3), (4, 9)])


def window_case_bytes():
    """The bf16 input of the window check: K chunks of WINDOW_CASE."""
    return gauss_bytes(np.random.default_rng(8), WINDOW_CASE["K"] * WINDOW_CASE["chunk"], 2)
