#!/usr/bin/env python3
"""bench.py -- throughput of the ZipNN hot path (compress + decompress) on B200.

Contract (see the task statement):  python bench.py --gpus N --steps K --warmup W [--impl reference]
prints ONE JSON line on rank 0.

  step      one pass of the hot path over one batch: compress the resident tensor, then
            decompress the stream that came out (both through zipnn_b200.ZipNN -> C ABI).
  value     whole-job GB/s = (uncompressed bytes all ranks coded in a step) / (t_compress +
            t_decompress), inputs resident in HBM, CUDA events, max over ranks.
  e2e       the same metric through the host-buffer API (pinned host tensors; H2D and D2H
            inside the timed region).
  roofline  for the dominant kernel of the step, timed with CUDA events on its own stream.
  cpu_baseline / --impl reference : the reference's own C path (oracle/_ref, compiled from
            /root/reference) or, if that binary is absent, the oracle port, on the host cores.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "compress+decompress GB/s on bf16 tensors"
GIB = 1 << 30


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--size-gib", type=float, default=16.0, help="uncompressed bytes per GPU")
    ap.add_argument("--dtype", default="bfloat16")
    ap.add_argument("--e2e-gib", type=float, default=-1.0, help="-1: size-gib if the host has the RAM, else 4")
    ap.add_argument("--cpu-sample-gib", type=float, default=1.0)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-sharded", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step returned on rank 0 (the stream and the decompressed tensor) "
                         "as DIR/<name>.npy in float32, so that two builds can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs records the outputs of --impl ours")
    return args


# ------------------------------------------------------------------ helpers
def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks/throttle reasons sampled every 200 ms while the timed region runs."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200",
                                          "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.lines.append(ln.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons, pw = [], [], set(), []
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2])); pw.append(float(f[3]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        busy = sorted(sm)[len(sm) // 2:]  # upper half = samples under load
        return {"sm_mhz": sorted(busy)[len(busy) // 2], "sm_max_mhz": max(mx), "power_w_max": max(pw),
                "samples": len(sm), "reasons": sorted(reasons)}


def make_tensor(nbytes, dtype, device, seed):
    import torch
    esz = torch.empty(0, dtype=dtype).element_size()
    n = nbytes // esz
    sigma = 0.5 if esz == 1 else 0.02
    g = torch.Generator(device=device).manual_seed(seed)
    out = torch.empty(n, dtype=dtype, device=device)
    slab = 1 << 27
    for i in range(0, n, slab):
        m = min(slab, n - i)
        out[i:i + m] = (torch.randn(m, generator=g, device=device, dtype=torch.float32) * sigma).to(dtype)
    return out


DUMP_ELEMS = 1 << 22      # per output: 16 MiB of float32, so both outputs stay well under 64 MB


def dump_outputs(out_dir, outputs):
    """Each tensor of `outputs` ({name: tensor}) -> out_dir/<name>.npy as float32 (exact for every dtype the
    bench codes).  A tensor with more than DUMP_ELEMS elements is sampled at DUMP_ELEMS positions drawn from a
    fixed seed, in ascending order: the same positions for every tensor of the same length."""
    import numpy as np
    import torch
    os.makedirs(out_dir, exist_ok=True)
    for name, x in outputs.items():
        x = x.reshape(-1)
        if x.numel() > DUMP_ELEMS:
            g = torch.Generator().manual_seed(20240601)
            idx = torch.randint(0, x.numel(), (DUMP_ELEMS,), generator=g).sort().values
            x = x[idx.to(x.device)]
        np.save(os.path.join(out_dir, name + ".npy"), x.float().cpu().numpy())


def cpu_reference_codec(num_buf=2, bits=1, bytes_mode=10, chunk=262144):
    """-> (kind, compress(bytes, threads) -> stream, decompress(stream, n, threads), release(buffer)).
    Layout defaults = bf16 (zipnn/zipnn.py:803-808); fp16 (2,0,10), fp32 (4,1,220), fp8 (1,1,10, chunk 131072)."""
    from oracle import oracle as O
    ref = O.ref_core()
    hdr = bytearray(32)
    hdr[0:2] = b"ZN"
    if ref is not None:
        import ctypes
        import numpy as np
        libc_free = ctypes.CDLL(None).free
        libc_free.argtypes = [ctypes.c_void_p]
        libc_free.restype = None

        def comp(buf, th):
            return ref.zipnn_core(bytes(hdr), buf, num_buf, bits, bytes_mode, 0, chunk, 0.95, 10, th)

        def dec(stream, n, th):
            return ref.combine_dtype(memoryview(stream)[32:], num_buf, bits, bytes_mode, chunk, n, th)

        def release(mv):
            # the reference wraps a malloc'ed buffer in an owner-less memoryview (csrc/zipnn_core.c:122,594-595,
            # 1119-1120): every call leaks its result.  The harness gives the block back (outside the timed
            # region) so that full-size steps can repeat inside one process.
            if mv is None or len(mv) == 0:
                return
            arr = np.frombuffer(mv, dtype=np.uint8)
            addr = arr.ctypes.data
            del arr                      # drops the buffer export, so the view can be released
            mv.release()
            libc_free(ctypes.c_void_p(addr))
        return "reference", comp, dec, release
    import numpy as np

    def comp(buf, th):
        return O.zipnn_compress(hdr, np.frombuffer(buf, dtype=np.uint8), num_buf, bits, bytes_mode, chunk, 0.95, threads=th)

    def dec(stream, n, th):
        return O.zipnn_decompress(np.asarray(stream)[32:], num_buf, bits, bytes_mode, chunk, n, threads=th)
    return "port", comp, dec, (lambda mv: None)


def time_cpu(sample_bytes, threads, reps=1, keep_stream=False):
    """Round-trip GB/s of the CPU path on `sample_bytes` (bytearray; the reference rotates it in place)."""
    import numpy as np
    kind, comp, dec, release = cpu_reference_codec()
    n = len(sample_bytes)
    best = None
    kept = None
    for _ in range(reps):
        work = bytearray(sample_bytes)  # clone outside the timed region (SURVEY Q1)
        t0 = time.perf_counter()
        s = comp(work, threads)
        t1 = time.perf_counter()
        d = dec(s, n, threads)
        t2 = time.perf_counter()
        assert len(d) == n
        cur = (t1 - t0, t2 - t1, len(s))
        if keep_stream and kept is None:
            kept = np.frombuffer(s, dtype=np.uint8).copy()
        if isinstance(d, memoryview):
            release(d)
        if isinstance(s, memoryview):
            release(s)
        del work
        if best is None or cur[0] + cur[1] < best[0] + best[1]:
            best = cur
    tc, td, slen = best
    return kind, n / (tc + td) / 1e9, n / tc / 1e9, n / td / 1e9, slen / n, kept


def host_cpu_info():
    """What the CPU arm can actually use on this box (explains run-to-run differences between boxes)."""
    info = {"logical_cores": os.cpu_count()}
    try:
        info["affinity"] = len(os.sched_getaffinity(0))
    except Exception:
        pass
    for path in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            info["cgroup_" + os.path.basename(path)] = open(path).read().strip()
            break
        except Exception:
            pass
    try:
        info["loadavg_1m"] = os.getloadavg()[0]
    except Exception:
        pass
    try:
        for ln in open("/proc/cpuinfo"):
            if ln.startswith("model name"):
                info["model"] = ln.split(":", 1)[1].strip()
                break
    except Exception:
        pass
    return info


def workload_text(dtype_name, nbytes):
    return (f"synthetic {dtype_name} tensor, {nbytes / GIB:.2f} GiB per GPU, randn*0.02 (seed 1234+rank), 256 KiB chunks; "
            "step = compress the tensor + decompress the stream that came out")


def thread_candidates(cores):
    return sorted({t for t in (16, 32, 64, cores) if 1 <= t <= cores} | {min(16, cores)})


# ------------------------------------------------------------------ reference arm
def run_reference(args, rank, world):
    if rank != 0:
        return
    try:
        import resource
        resource.setrlimit(resource.RLIMIT_STACK, (resource.RLIM_INFINITY, resource.RLIM_INFINITY))
    except Exception:
        pass
    import psutil
    import torch
    cores = os.cpu_count() or 1
    dtype = getattr(torch, args.dtype)
    full = int(args.size_gib * GIB)
    # the same bytes our arm codes on rank 0 (generated on the GPU when there is one: seconds instead of minutes)
    gen_dev = "cuda" if torch.cuda.is_available() else "cpu"
    avail = psutil.virtual_memory().available
    nbytes = full
    while nbytes > (1 << 28) and 3.2 * nbytes + (8 << 30) > avail:      # input + working clone + stream/result
        nbytes //= 2
    t = make_tensor(nbytes, dtype, gen_dev, 1234)
    whole = bytearray(t.view(torch.uint8).cpu().numpy().tobytes())
    del t
    if gen_dev == "cuda":
        torch.cuda.empty_cache()
    # ---- thread sweep on a bounded sample: the reference's default (min(cpu,16), zipnn/zipnn.py:176-177) and the best of {16,32,64,all}
    sweep_bytes = min(len(whole), 2 * GIB)
    sweep = {}
    for th in thread_candidates(cores):
        _, v, vc, vd, _, _ = time_cpu(whole[:sweep_bytes], th)
        sweep[th] = {"round_trip_gbs": round(v, 3), "compress_gbs": round(vc, 3), "decompress_gbs": round(vd, 3)}
    best_th = max(sweep, key=lambda k: sweep[k]["round_trip_gbs"])
    default_th = min(16, cores)
    # ---- size of one step: the full workload unless the K + W steps would not end within a few minutes
    budget_s = 240.0
    sample = len(whole)
    per_byte = 1.0 / (sweep[best_th]["round_trip_gbs"] * 1e9)
    while sample > GIB and (args.steps + args.warmup) * sample * per_byte * 1.15 > budget_s:
        sample //= 2
    data = whole if sample == len(whole) else whole[:sample]
    kind = "reference"
    for _ in range(args.warmup):
        kind, *_ = time_cpu(data, best_th)
    t0 = time.perf_counter()
    vals = [time_cpu(data, best_th) for _ in range(args.steps)]
    wall = time.perf_counter() - t0
    v = sum(x[1] for x in vals) / len(vals)
    sample_txt = (f"{sample / GIB:.2f} GiB of the workload per step" + ("" if sample == full else f" (bounded: the full {full / GIB:.0f} GiB x {args.steps + args.warmup} steps would not end within {budget_s:.0f} s"
                  + (" or does not fit host RAM" if len(whole) < full else "") + ")")
                  + f", {best_th} threads = best of {sorted(sweep)} on a {sweep_bytes / GIB:.0f} GiB sweep; reference default is {default_th} threads")
    line = {
        "impl": "reference", "metric": METRIC, "value": round(v, 4), "unit": "GB/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(1e3 * sample / (v * 1e9), 3),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": {"workload": workload_text(args.dtype, full),
                   "l2": "inputs are far larger than the 126 MB L2 (no flush needed)", "sharding": "one tensor shard per GPU, no data-path collective"},
        "timing": "host wall clock; the reference C path (zipnn_core.zipnn_core + combine_dtype) called directly, input clone outside the timed region, leaked result buffers freed by the harness between steps",
        "compress_gbs": round(sum(x[2] for x in vals) / len(vals), 4), "decompress_gbs": round(sum(x[3] for x in vals) / len(vals), 4),
        "ratio": round(vals[0][4], 6),
        "cpu_baseline": {"value": round(v, 4), "unit": "GB/s", "cores": best_th, "kind": kind, "sample": sample_txt,
                         "threads_sweep": {str(k): sweep[k] for k in sorted(sweep)}, "default_threads": default_th,
                         "default_threads_value": sweep[default_th]["round_trip_gbs"], "host": host_cpu_info()},
        "e2e": {"value": round(v, 4), "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0, "wall_s": round(wall, 2),
    }
    print(json.dumps(line), flush=True)



def bind_to_gpu_numa(local_rank):
    """Pin this process (and the threads / pinned buffers it creates afterwards) to the CPUs that share a
    NUMA node with its GPU: 8 ranks that all stage through node 0's memory halve each other's PCIe rate."""
    info = {"bound": False}
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(local_rank)
        ncpu = os.cpu_count() or 1
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (ncpu + 63) // 64)
        cpus = [64 * i + b for i, w in enumerate(words) for b in range(64) if (int(w) >> b) & 1]
        cpus = [c for c in cpus if c < ncpu]
        if cpus:
            os.sched_setaffinity(0, cpus)
            info = {"bound": True, "cpus": f"{min(cpus)}-{max(cpus)} ({len(cpus)})"}
            try:
                for node in sorted(os.listdir("/sys/devices/system/node")):
                    if node.startswith("node") and os.path.exists(f"/sys/devices/system/node/{node}/cpu{cpus[0]}"):
                        info["numa_node"] = int(node[4:])
            except Exception:
                pass
    except Exception as exc:  # no NVML / not permitted: run unbound and say so
        info["error"] = str(exc)[:120]
    return info


def run_sharded(args, rank, world, dev, total_bytes, dtype):
    """ONE tensor of `total_bytes`, chunk ranges partitioned over the ranks (zipnn_b200.sharded): local codec
    with no communication, then the per-rank payloads gathered into rank 0's buffer with point-to-point
    NCCL sends (NVLink), giving the byte-identical single-GPU stream; the way back scatters payload ranges.
    Codec time and exchange time are reported separately (SURVEY.md section 8e)."""
    import torch
    import torch.distributed as dist
    from zipnn_b200 import ZipNN
    from zipnn_b200.sharded import HEADER_LEN, ShardedZipNN, byte_range
    esz = torch.empty(0, dtype=dtype).element_size()
    n_elems = total_bytes // esz
    chunk = 131072 if esz == 1 else 262144
    b0, b1 = byte_range(n_elems * esz, chunk, rank, world)
    # every rank draws the same stream of random numbers, slab by slab, and keeps its own byte range
    g = torch.Generator(device=dev).manual_seed(4321)
    local = torch.empty((b1 - b0) // esz, dtype=dtype, device=dev)
    full = torch.empty(n_elems, dtype=dtype, device=dev) if rank == 0 else None
    slab = 1 << 27
    for i in range(0, n_elems, slab):
        m = min(slab, n_elems - i)
        piece = (torch.randn(m, generator=g, device=dev, dtype=torch.float32) * (0.5 if esz == 1 else 0.02)).to(dtype)
        lo, hi = max(i, b0 // esz), min(i + m, b1 // esz)
        if hi > lo:
            local[lo - b0 // esz: hi - b0 // esz] = piece[lo - i: hi - i]
        if full is not None:
            full[i: i + m] = piece
        del piece
    z = ShardedZipNN()
    ev = lambda: torch.cuda.Event(enable_timing=True)
    res = {}
    reps = 3
    tc, tg, ts, td = [], [], [], []
    stream = None
    for it in range(reps + 1):
        torch.cuda.synchronize(); dist.barrier()
        e0, e1, e2 = ev(), ev(), ev()
        e0.record()
        lstream, plan = z.compress_local(local)
        e1.record()
        n_local = local.numel() * esz
        stream = z.gather(lstream, plan, n_local, (n_elems,), 0)
        e2.record()
        torch.cuda.synchronize(); dist.barrier()
        e3, e4 = ev(), ev()
        e3.record()
        back = z.decompress(stream if rank == 0 else None, src=0, device=dev)
        e4.record()
        torch.cuda.synchronize()
        if it:
            tc.append(e0.elapsed_time(e1)); tg.append(e1.elapsed_time(e2)); td.append(e3.elapsed_time(e4))
        if it == 0:
            ok_local = bool(torch.equal(back.view(torch.uint8), local.view(torch.uint8)))
        if it < reps:
            del lstream, back
            if rank != 0:
                stream = None
    vals = torch.tensor([sum(tc) / reps, sum(tg) / reps, sum(td) / reps, 0.0 if ok_local else 1.0], device=dev, dtype=torch.float64)
    dist.all_reduce(vals, op=dist.ReduceOp.MAX)
    codec_ms, gather_ms, dec_total_ms, bad = [float(x) for x in vals.tolist()]
    if rank == 0:
        want = ZipNN(input_format="torch").compress(full)
        same = stream.numel() == want.numel() and bool(torch.equal(stream, want))
        # decompress side: local decode time of rank 0's shard alone, to split scatter from codec
        own = ShardedZipNN()
        ls0, _ = own.compress_local(local)
        a, b = ev(), ev()
        a.record()
        own._codec()[1](ls0[HEADER_LEN:], plan["num_buf"], plan["bit_reorder"], plan["byte_reorder"], plan["chunk"], local.numel() * esz)
        b.record()
        torch.cuda.synchronize()
        dec_codec_ms = a.elapsed_time(b)
        C = int(stream.numel())
        moved = C * (world - 1) // world
        N = n_elems * esz
        res = {"tensor_bytes": N, "stream_bytes": C, "ranks": world, "stream_equals_single_gpu": bool(same), "round_trip_exact": bad == 0.0,
               "compress": {"codec_ms": round(codec_ms, 3), "gather_ms": round(gather_ms, 3), "nvlink_bytes_into_owner": moved,
                            "gather_gbs_into_owner": round(moved / (gather_ms * 1e-3) / 1e9, 1) if gather_ms > 0 else None,
                            "gbs_of_N": round(N / ((codec_ms + gather_ms) * 1e-3) / 1e9, 1), "codec_only_gbs_of_N": round(N / (codec_ms * 1e-3) / 1e9, 1)},
               "decompress": {"scatter_plus_codec_ms": round(dec_total_ms, 3), "codec_ms_rank0": round(dec_codec_ms, 3),
                              "scatter_ms_estimate": round(max(dec_total_ms - dec_codec_ms, 0.0), 3),
                              "gbs_of_N": round(N / (dec_total_ms * 1e-3) / 1e9, 1)},
               "transport": "CUDA IPC: every rank copies its payload slices straight into (out of) the owner's buffer -- peer copies over NVLink, no send/recv pairing",
               "limiter": "the exchange: C*(R-1)/R bytes enter / leave ONE GPU over its NVLink ports (~0.75 TB/s measured peer rate), while the codec side scales with R",
               "note": "the reference has no distributed path; this is the design BASELINE.json's north_star describes (chunks partition, NCCL only gathers the stream)"}
        del want, full
    del local, stream
    torch.cuda.empty_cache()
    return res


# ------------------------------------------------------------------ our arm
def run_ours(args, rank, local_rank, world):
    import torch
    import torch.distributed as dist
    from zipnn_b200 import ZipNN, _native

    numa = bind_to_gpu_numa(local_rank) if world > 1 or os.environ.get("ZIPNN_BENCH_BIND") else {"bound": False}
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    dtype = getattr(torch, args.dtype)
    nbytes = int(args.size_gib * GIB)
    t = make_tensor(nbytes, dtype, dev, 1234 + rank)
    nbytes = t.numel() * t.element_size()

    def step():
        s = ZipNN(input_format="torch").compress(t)
        d = ZipNN(input_format="torch").decompress(s)
        return s, d

    # ---- warm-up + exactness check (outside the timed region)
    for _ in range(max(args.warmup, 1)):
        s, d = step()
    assert torch.equal(d.view(torch.uint8), t.view(torch.uint8)), "round trip is not exact"
    stream_bytes = s.numel()
    del s, d
    barrier = (lambda: dist.barrier()) if world > 1 else (lambda: None)

    # ---- timed region: device-resident
    clocks = ClockSampler(local_rank)
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2 * args.steps + 1)]
    _native.timing_enable(True)
    launches0 = _native.launch_count()
    barrier()
    torch.cuda.synchronize()
    if rank == 0:
        clocks.start()
    ev[0].record()
    for i in range(args.steps):
        s = ZipNN(input_format="torch").compress(t)
        ev[2 * i + 1].record()
        d = ZipNN(input_format="torch").decompress(s)
        ev[2 * i + 2].record()
        if i + 1 < args.steps:
            del s, d
    torch.cuda.synchronize()
    barrier()
    clk = clocks.stop() if rank == 0 else None
    launches = _native.launch_count() - launches0
    ktimes = _native.timing_collect()
    _native.timing_enable(False)
    total_ms = ev[0].elapsed_time(ev[-1])
    tc_ms = sum(ev[2 * i].elapsed_time(ev[2 * i + 1]) for i in range(args.steps)) / args.steps
    td_ms = sum(ev[2 * i + 1].elapsed_time(ev[2 * i + 2]) for i in range(args.steps)) / args.steps
    step_ms = total_ms / args.steps
    if world > 1:
        tt = torch.tensor([step_ms, tc_ms, td_ms], device=dev, dtype=torch.float64)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        step_ms, tc_ms, td_ms = [float(x) for x in tt.tolist()]
    value = world * nbytes / (step_ms * 1e-3) / 1e9
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"stream": s, "decompressed": d})
    del s, d

    # ---- e2e: host buffers through the public API (rank-local; reported for the whole job)
    e2e = None
    if not args.no_e2e:
        import psutil
        want = args.e2e_gib if args.e2e_gib > 0 else (args.size_gib if psutil.virtual_memory().available > (6 * args.size_gib + 16) * GIB * world else min(4.0, args.size_gib))
        eb = int(want * GIB)
        torch.cuda.empty_cache()
        ht = torch.empty(eb // t.element_size(), dtype=dtype, pin_memory=True)
        ht.copy_(t[: ht.numel()])
        torch.cuda.synchronize()
        # staging buffers a real caller would keep across tensors (pinned once, outside the step)
        hs_buf = torch.empty(eb + (eb >> 6) + 4096, dtype=torch.uint8, pin_memory=True)
        hd_buf = torch.empty(ht.numel(), dtype=dtype, pin_memory=True)
        zs = ZipNN(input_format="torch").compress(ht, out=hs_buf)          # warm-up
        hd = ZipNN(input_format="torch").decompress(zs, out=hd_buf)
        assert torch.equal(hd.view(torch.uint8), ht.view(torch.uint8))
        c_e2e = len(zs)
        del zs, hd
        reps = max(2, min(args.steps, 3))
        barrier()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(reps):
            zs = ZipNN(input_format="torch").compress(ht, out=hs_buf)     # H2D N, kernels, D2H C
            hd = ZipNN(input_format="torch").decompress(zs, out=hd_buf)   # H2D C, kernels, D2H N
            _ = hd.view(torch.uint8)[-1].item()                           # the result is read on the host
            del zs, hd
        torch.cuda.synchronize()
        e_ms = (time.perf_counter() - t0) * 1e3 / reps
        if world > 1:
            tt = torch.tensor([e_ms], device=dev, dtype=torch.float64)
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            e_ms = float(tt.item())
        e2e = {"value": round(world * eb / (e_ms * 1e-3) / 1e9, 3), "unit": "GB/s", "h2d_bytes_per_step": world * (eb + c_e2e),
               "d2h_bytes_per_step": world * (c_e2e + eb), "ms_per_step": round(e_ms, 2), "bytes_per_gpu": eb,
               "api": "zipnn_b200.ZipNN(input_format='torch').compress(pinned cpu tensor, out=pinned) / .decompress(host stream, out=pinned) -> C ABI zipnn_b200_compress_host / zipnn_b200_decompress_host (include/zipnn_b200.h): the library moves the data through the device slab by slab, H2D copy, kernels and D2H copy overlapped"}
        e2e["numa"] = numa
        # per-rank one-way PCIe rates of the e2e region (the limiter at 8 GPUs is host memory / root ports, not the codec)
        del ht, hs_buf, hd_buf

    # ---- the sharded path (N > 1): one tensor partitioned by chunk range, NCCL gathers / scatters the stream
    sharded = None
    if world > 1 and not args.no_sharded:
        del t                      # (the CPU leg below runs at N = 1 only)
        t = None
        torch.cuda.empty_cache()
        sharded = run_sharded(args, rank, world, dev, nbytes, dtype)

    # ---- CPU baseline beside it (rank 0, single-GPU runs only) + stream == reference stream at the bench scale
    cpu = None
    parity = None
    if rank == 0 and world == 1 and not args.no_cpu:
        try:
            import resource
            resource.setrlimit(resource.RLIMIT_STACK, (resource.RLIM_INFINITY, resource.RLIM_INFINITY))
        except Exception:
            pass
        import numpy as np
        from tools.stream_windows import StreamTables, check_stream_windows
        chunk = 262144
        sb = int(min(args.cpu_sample_gib * GIB, nbytes)) // chunk * chunk
        sample = bytearray(t.view(torch.uint8)[:sb].cpu().numpy().tobytes())
        cores = os.cpu_count() or 1
        kind, v, vc, vd, ratio_cpu, ref_stream = time_cpu(sample, cores, reps=2, keep_stream=True)
        cpu = {"value": round(v, 4), "unit": "GB/s", "cores": cores, "kind": kind, "compress_gbs": round(vc, 4),
               "decompress_gbs": round(vd, 4), "ratio": round(ratio_cpu, 6),
               "sample": f"first {sb / GIB:.2f} GiB of the same tensor, {cores} threads (all logical cores), best of 2"}
        # The checker's stream for the first sb bytes is a window of ours; so are the chunks whose cumulative
        # offsets straddle 2^32 in every group (u64 size table, csrc/zipnn_core.c:145-153, 1002-1005).
        z = ZipNN(input_format="torch")
        gs = z.compress(t)
        torch.cuda.synchronize()
        hdr_len = len(z._last_plan["header"])
        G = z._last_plan["num_buf"]
        K = (nbytes + chunk - 1) // chunk
        tab = StreamTables(gs, hdr_len, G, K)
        first = True
        _, comp, _, release = cpu_reference_codec()

        def compress_window(data):
            nonlocal first
            if first and data.size == sb:       # the stream time_cpu kept: no second CPU pass over the first GiB
                first = False
                return ref_stream, 32
            mv = comp(bytearray(data.tobytes()), cores)
            out = np.frombuffer(mv, dtype=np.uint8).copy()
            if isinstance(mv, memoryview):
                release(mv)
            return out, 32

        wins = [(0, sb // chunk)]
        for g in range(G):
            lim = 1 << 32
            if lim > int(tab.base[g]):
                cx = tab.first_chunk_past(g, lim - int(tab.base[g]))   # the absolute stream offset passes 2^32 inside this group
                if 0 < cx < K:
                    wins.append((cx - 128, cx + 128))
            cy = tab.first_chunk_past(g, lim)                          # the group's own cumulative size passes 2^32
            if 0 < cy < K:
                wins.append((cy - 128, cy + 128))
        wins.append((K - 256, K))
        uniq = []
        for w in wins:
            w = (max(0, w[0]), min(K, w[1]))
            if w not in uniq and w[1] > w[0]:
                uniq.append(w)
        try:
            res = check_stream_windows(gs, hdr_len, G, K, chunk, nbytes,
                                       lambda a, b: t.view(torch.uint8)[a:b].cpu().numpy(), uniq, compress_window)
            parity = {"stream_equals_reference": True, "checker": kind, "stream_bytes": int(gs.numel()), **res}
        except AssertionError as exc:
            parity = {"stream_equals_reference": False, "checker": kind, "error": str(exc)}
        del gs

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- roofline of the dominant kernel
    peak, peak_src = peaks()
    per_launch = {k: (ms / max(cnt, 1), cnt) for k, (ms, cnt) in ktimes.items() if cnt}
    dom = max(per_launch, key=lambda k: per_launch[k][0] * per_launch[k][1])
    N, Cb = nbytes, stream_bytes
    esz_t = torch.empty(0, dtype=dtype).element_size()
    G = 1 if esz_t == 1 else (2 if esz_t == 2 else 4)
    huf_payload = Cb - (N // G) * (G - 1) if G > 1 else Cb  # bytes of the Huffman-coded group(s) (the others are stored raw)
    algo = {  # algorithmic bytes per launch, see DESIGN.md "kernels"
        "k_encode_hist": N,                     # reads every input byte once
        "k_encode_write_warp": N + Cb,               # reads the input again, writes the stream
        "k_huf_decode_fused": Cb + N,           # reads the whole stream, writes the elements (fused decode + regroup)
    }
    dom_ms = per_launch[dom][0]
    achieved = algo.get(dom, N) / (dom_ms * 1e-3) / 1e9
    kernels = {k: {"ms_per_launch": round(v[0], 4), "launches": v[1],
                   "algo_gbs": round(algo[k] / (v[0] * 1e-3) / 1e9, 1) if k in algo and v[0] > 0 else None,
                   "roofline_frac": round(algo[k] / (v[0] * 1e-3) / 1e9 / peak, 4) if k in algo and v[0] > 0 else None}
               for k, v in per_launch.items()}
    # DRAM bytes per launch of the dominant kernel: recorded from one `ncu --set full` capture of the same
    # workload (never measured under this run: ncu serialises and replays kernels); null when the
    # workload differs from the recorded one.
    traffic, traffic_src = None, None
    try:
        rec = json.load(open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "profiles", "traffic.json"))).get(dom)
        if rec and rec.get("n_bytes") == N and dtype == torch.bfloat16:
            traffic, traffic_src = rec["traffic_bytes_per_launch"], rec["source"]
    except Exception:
        pass
    # The north-star kernel (BASELINE.json: decompress) is no longer the longest one: its roofline next to `roofline`,
    # which stays the dominant kernel of the step as the contract says.
    north_star = None
    try:
        ns = "k_huf_decode_fused"
        if ns in per_launch and per_launch[ns][0] > 0:
            ns_ms = per_launch[ns][0]
            ns_rec = json.load(open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "profiles", "traffic.json"))).get(ns) or {}
            ns_traffic = ns_rec.get("traffic_bytes_per_launch") if (ns_rec.get("n_bytes") == N and dtype == torch.bfloat16) else None
            north_star = {"kernel": ns, "bound": "hbm", "achieved": round(algo[ns] / (ns_ms * 1e-3) / 1e9, 1), "peak": peak, "unit": "GB/s",
                          "frac": round(algo[ns] / (ns_ms * 1e-3) / 1e9 / peak, 4), "ms_per_launch": round(ns_ms, 4),
                          "algorithmic_bytes_per_launch": algo[ns], "traffic": ns_traffic}
    except Exception:
        north_star = None
    line = {
        "metric": METRIC, "value": round(value, 3), "unit": "GB/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": round(step_ms, 3), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "u8", "data": "synthetic",
        "config": {"workload": workload_text(args.dtype, nbytes),
                   "l2": "inputs are far larger than the 126 MB L2 (no flush needed)", "sharding": "one tensor shard per GPU, no data-path collective"},
        "compress_gbs": round(world * N / (tc_ms * 1e-3) / 1e9, 2), "decompress_gbs": round(world * N / (td_ms * 1e-3) / 1e9, 2),
        "ratio": round(Cb / N, 6),
        "path_roofline": {"compress_frac": round((N + Cb) / (tc_ms * 1e-3) / 1e9 / peak, 4),
                          "decompress_frac": round((N + Cb) / (td_ms * 1e-3) / 1e9 / peak, 4),
                          "note": "(N + C) / t / peak: SURVEY.md section 8d definition for the whole direction"},
        "roofline": {"bound": "hbm", "kernel": dom, "achieved": round(achieved, 1), "peak": peak, "unit": "GB/s",
                     "frac": round(achieved / peak, 4), "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src,
                     "algorithmic_bytes_per_launch": algo.get(dom, N), "ms_per_launch": round(dom_ms, 4)},
        "kernels": kernels,
        "north_star_kernel": north_star,
        "gpu_launches": int(launches),
        "clocks": clk,
    }
    if e2e:
        line["e2e"] = e2e
    if cpu:
        line["cpu_baseline"] = cpu
    if parity:
        line["parity_check"] = parity
    if sharded:
        line["sharded"] = sharded
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    args = parse()
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank, world)
    else:
        run_ours(args, rank, local_rank, world)


if __name__ == "__main__":
    main()
