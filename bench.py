#!/usr/bin/env python
"""bench.py -- the benchmarks BASELINE.json names, one JSON line per run.

  python bench.py [--config c2] --gpus N --steps K --warmup W     our arm (CUDA path through the C ABI)
  python bench.py --impl reference [--config ...] ...             the reference's own CPU code on the host cores

  c2 (default, the headline)  10 000 x 64 KiB synthetic text units per GPU, -m2, one compressBlock per unit
  c3  100 MB enwik-shaped synthetic corpus per GPU in 64 KiB blocks, -m3, compress + decompress round trip
  c4  dedup fragmenter + fragment SHA-1 + per-file BLAKE3 over a synthetic filesystem image (--c4-gb in total,
      files dealt to the GPUs, digests exchanged for the global unique-fragment count)
  c5  mixed-entropy 64 KiB units, -m5 (--c5-units per GPU; BASELINE's 1 000 000 do not fit a few-minute run)

A "step" = one pass of the hot path over one batch of synthetic input.  Per rank the batch is fixed (weak scaling)
except c4 (strong: one image, files dealt to the ranks).  `value` = work of all ranks / max-over-ranks device time.
  value : inputs and outputs resident in HBM (device-pointer entry points) where the path has one
  e2e   : the reference-facing call with HOST buffers: H2D of the batch and D2H of the results inside the timed region.
c2 runs with `--inflight` (default 2) steps outstanding through zq_pipe_* -- the counterpart of CompressJob's block
queue.  Bracket: barrier + device synchronize, CUDA event, K steps, device synchronize, CUDA event, barrier; max over
ranks.  `stage_ms` / `roofline` come from a serial pass on ONE context whose stream is torch's current stream, so
the per-kernel CUDA events there time exactly one kernel each.  Inputs exceed L2 (126 MB) in every config.
Parity: every block / digest / fragment table of the timed batch is compared with the reference (oracle/_ref, run once
on all host cores, outside the timed region) -- config.parity says how many matched.
--dump-outputs DIR: after the timed steps, what the last timed step returned is written as DIR/<name>.npy (float32 /
float64, at most 64 MB): block offsets and lengths, the SHA-256 of every block and a fixed sample of whole blocks; c4
the fragment tables and digests.  The inputs depend on the arguments only, so two builds can be compared file by file.
"""
import argparse
import hashlib
import importlib.util
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True     # the tree may be read-only; nothing is written into it

UNIT = 65536
MB = 1e6
METRICS = {
    "c2": ("MB/s compressed (-m2, 64 KiB frags)", "MB/s", "2"),
    "c3": ("MB/s round trip (-m3 compress + decompress, 64 KiB blocks)", "MB/s", "3"),
    "c4": ("GB/s fragmenter + fragment SHA-1 + file BLAKE3 (-fragment 6)", "GB/s", None),
    "c5": ("MB/s compressed (-m5, 64 KiB mixed-entropy frags)", "MB/s", "5"),
}
# state bytes read+written per coded bit (SURVEY.md section 8d): S = sum over the model's components
S_BYTES = {"3": 28, "4": 157, "5": 573}
DUMP_CAP = 64 << 20       # --dump-outputs: bytes written at most
DUMP_SAMPLE = 128         # --dump-outputs: blocks of a batch written whole (a seeded choice; all by SHA-256)


def load_corpus():
    """zpaqfranz_b200/corpus.py by path: pure numpy, does not load the CUDA library (the reference arm must not)."""
    spec = importlib.util.spec_from_file_location("zq_corpus", os.path.join(ROOT, "zpaqfranz_b200", "corpus.py"))
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    return m


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler(threading.Thread):
    """Samples nvidia-smi clocks / throttle reasons while the timed region runs."""

    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self.stop_flag = index, [], False

    def run(self):
        while not self.stop_flag:
            try:
                r = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                    "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5)
                if r.returncode == 0 and r.stdout.strip():
                    self.rows.append([x.strip() for x in r.stdout.strip().split(",")])
            except Exception:
                pass
            time.sleep(0.2)

    def summary(self):
        sm = sorted(int(r[0]) for r in self.rows if r[0].isdigit())
        mx = [int(r[1]) for r in self.rows if r[1].isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for k, n in enumerate(names) if any(len(r) > 2 + k and r[2 + k] == "Active" for r in self.rows)]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "samples": len(self.rows)}


def block_outputs(data, ooff, olen, prefix=""):
    """What a caller of a batch entry point receives -- blocks data[ooff[i]:ooff[i]+olen[i]], their offsets and lengths --
    as float arrays for --dump-outputs: every block by its SHA-256, a seeded sample of DUMP_SAMPLE blocks byte for byte."""
    n = len(olen)
    blocks = [data[int(ooff[i]): int(ooff[i]) + int(olen[i])] for i in range(n)]
    pick = np.sort(np.random.default_rng(0).choice(n, size=min(n, DUMP_SAMPLE), replace=False))
    sha = np.frombuffer(b"".join(hashlib.sha256(b).digest() for b in blocks), dtype=np.uint8).reshape(n, 32)
    return {prefix + "offsets": np.asarray(ooff, dtype=np.float64), prefix + "lengths": np.asarray(olen, dtype=np.float64),
            prefix + "sha256": sha.astype(np.float32), prefix + "sample_index": pick.astype(np.float64),
            prefix + "sample_bytes": np.concatenate([blocks[i] for i in pick] + [np.zeros(0, np.uint8)]).astype(np.float32)}


def dump_outputs(directory, arrays):
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_CAP:
        raise SystemExit("--dump-outputs: %d bytes exceed the %d-byte cap (a smaller workload dumps less)" % (total, DUMP_CAP))
    os.makedirs(directory, exist_ok=True)
    for name, a in arrays.items():
        assert a.dtype in (np.float32, np.float64), name
        np.save(os.path.join(directory, name + ".npy"), a)


# ---- synthetic workloads (same bytes for both arms) ------------------------------------------------------------
def make_units(corpus, cfg, rank, args):
    """(arena u8, offsets u64, lengths u32) of the compression configs."""
    if cfg == "c2":
        U = args.units
        arena = corpus.text_corpus(U, UNIT, seed0=rank)
    elif cfg == "c3":
        U = args.c3_mb * 1000000 // UNIT
        arena = enwik_like(corpus, U * UNIT, 7000 + rank)
    else:
        U = args.c5_units
        arena = np.empty(U * UNIT, dtype=np.uint8)
        for u in range(U):
            arena[u * UNIT:(u + 1) * UNIT] = np.frombuffer(corpus.mixed_unit(rank * 1000003 + u, UNIT), dtype=np.uint8)
    return arena, np.arange(U, dtype=np.uint64) * UNIT, np.full(U, UNIT, dtype=np.uint32)


def enwik_like(corpus, nbytes, seed):
    """XML-ish markup around word-soup paragraphs with ~2 % digits (SURVEY.md section 8d, C3)."""
    rng = np.random.Generator(np.random.PCG64([seed, 33]))
    text = corpus.text_bytes(seed, nbytes).copy()
    # a <tag attr="1234"> ... </tag> frame every ~600 bytes, digits sprinkled over 2 % of the bytes
    tags = [b"<page>\n  <title>", b"</title>\n  <id>", b"</id>\n  <revision>\n    <timestamp>", b"</timestamp>\n    <text xml:space=\"preserve\">",
            b"</text>\n  </revision>\n</page>\n", b"[[", b"]]", b"{{", b"}}", b"&quot;", b"&amp;"]
    pos = np.cumsum(rng.integers(200, 1000, nbytes // 600 + 2))
    for k, p in enumerate(pos):
        t = tags[int(rng.integers(0, len(tags)))]
        if p + len(t) < nbytes:
            text[p:p + len(t)] = np.frombuffer(t, dtype=np.uint8)
    dig = rng.integers(0, nbytes, nbytes // 50)
    text[dig] = rng.integers(48, 58, len(dig)).astype(np.uint8)
    return text


def make_image(corpus, total_bytes, seed=4):
    """File list of the synthetic filesystem image (SURVEY.md section 8d, C4): log-normal sizes (median 16 KiB, capped
    at 64 MiB), content classes 40 % text / 30 % random / 20 % copies of earlier files / 10 % zero pages.  Returns
    (sizes, kinds, srcs): contents are a pure function of the file id, so every rank can build its own files."""
    rng = np.random.Generator(np.random.PCG64(seed))
    n = int(total_bytes / 60000) + 64
    sizes = np.minimum(rng.lognormal(np.log(16384), 2.0, n), 64 << 20).astype(np.int64) + 1
    k = int(np.searchsorted(np.cumsum(sizes), total_bytes)) + 1
    sizes = sizes[:k]
    kinds = rng.integers(0, 10, k)
    srcs = (rng.random(k) * np.arange(k)).astype(np.int64)
    return sizes, kinds, srcs


_POOLS = {}


def file_bytes(corpus, f, sizes, kinds, srcs, depth=0):
    """Content of file f.  Text and random files are windows of two fixed 64 MiB pools at a per-file offset."""
    s = int(sizes[f])
    kd = int(kinds[f])
    if not _POOLS:
        _POOLS["t"] = corpus.text_bytes(991, (64 << 20) + (1 << 20))
        _POOLS["r"] = np.random.Generator(np.random.PCG64(992)).integers(0, 256, (64 << 20) + (1 << 20), dtype=np.uint8)
    if kd >= 7 and kd < 9 and f > 10 and depth < 4:      # copy of an earlier file (dedup hit), zero tail if longer
        out = np.zeros(s, dtype=np.uint8)
        src = file_bytes(corpus, int(srcs[f]), sizes, kinds, srcs, depth + 1)
        k = min(s, len(src))
        out[:k] = src[:k]
        return out
    if kd >= 9 or (kd >= 7 and kd < 9):
        return np.zeros(s, dtype=np.uint8)
    pool = _POOLS["t"] if kd < 4 else _POOLS["r"]
    o = (f * 2654435761) % (len(pool) - s) if len(pool) > s else 0
    return pool[o:o + s]


# ---- the reference on the host cores ---------------------------------------------------------------------------
def ref_lib():
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle_bindings as ob
    return ob.load_ref()


def ref_compress_list(ref, arena, offs, lens, method, threads, digests=False, roundtrip=False):
    """(MB/s, seconds, total compressed bytes, sha256 digests [n,32] or None, lengths) through zref_compress_list_mt."""
    import ctypes as C
    n = len(offs)
    off = np.ascontiguousarray(offs, dtype=np.uint64)
    ln = np.ascontiguousarray(lens, dtype=np.uint32)
    dg = np.zeros((n, 32), dtype=np.uint8) if digests else None
    ol = np.zeros(n, dtype=np.uint32)
    f = ref.lib.zref_compress_list_mt
    f.restype = C.c_longlong
    t0 = time.perf_counter()
    tot = f(arena.ctypes.data_as(C.c_void_p), off.ctypes.data_as(C.c_void_p), ln.ctypes.data_as(C.c_void_p), C.c_int(n),
            method.encode(), C.c_int(threads), dg.ctypes.data_as(C.c_void_p) if digests else None, ol.ctypes.data_as(C.c_void_p),
            C.c_int(1 if roundtrip else 0))
    dt = time.perf_counter() - t0
    if tot < 0:
        raise RuntimeError("reference failed on the batch")
    return float(ln.sum()) / MB / dt, dt, int(tot), dg, ol


def best_threads(ref, arena, offs, lens, method):
    """The reference's pthread pool does not scale linearly (allocator contention): probe a few thread counts on a
    small sample and keep the fastest, so the baseline is the reference at its best."""
    ncpu = os.cpu_count() or 1
    best, best_v = ncpu, 0.0
    for t in sorted({max(1, ncpu >> k) for k in range(0, 4)}, reverse=True):
        k = min(len(offs), max(t * 2, 16))
        v = ref_compress_list(ref, arena, offs[:k], lens[:k], method, t)[0]
        if v > best_v:
            best, best_v = t, v
    return best


def ref_c4(ref, arena, offs, lens, threads):
    """Fragmenter + SHA-1 of every fragment + BLAKE3 of every file with the reference's own code on `threads` host
    threads (zref_fragment_hash_mt).  Returns seconds."""
    import ctypes as C
    f = ref.lib.zref_fragment_hash_mt
    f.restype = C.c_longlong
    off = np.ascontiguousarray(offs, dtype=np.uint64)
    ln = np.ascontiguousarray(lens, dtype=np.uint64)
    t0 = time.perf_counter()
    f(arena.ctypes.data_as(C.c_void_p), off.ctypes.data_as(C.c_void_p), ln.ctypes.data_as(C.c_void_p), C.c_int(len(off)), C.c_int(6), C.c_int(threads))
    return time.perf_counter() - t0


def build_files(corpus, files, sizes, kinds, srcs, out=None):
    msz = sizes[files].astype(np.uint64)
    moff = np.concatenate([[0], np.cumsum(msz)[:-1]]).astype(np.uint64)
    if out is None:
        out = np.empty(int(msz.sum()), dtype=np.uint8)
    for o, f in zip(moff, files):
        d = file_bytes(corpus, int(f), sizes, kinds, srcs)
        out[int(o):int(o) + len(d)] = d
    return out, moff, msz


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    corpus = load_corpus()
    ref = ref_lib()
    cfg = args.config
    metric, unit, method = METRICS[cfg]
    if ref is None:
        print(json.dumps({"impl": "reference", "unavailable": "oracle/_ref/libzpaqref.so missing"}))
        return 0
    ncpu = os.cpu_count() or 1
    if cfg == "c4":
        sizes, kinds, srcs = make_image(corpus, int(args.c4_gb * 1e9))
        threads = ncpu
        k = int(np.searchsorted(np.cumsum(sizes), args.ref_sample_mb * 1e6 * 8)) + 1   # hashing is far faster than compressing
        files = list(range(min(k, len(sizes))))
        arena, moff, msz = build_files(corpus, files, sizes, kinds, srcs)
        tot = int(msz.sum())
        times = []
        for _ in range(args.warmup + args.steps):
            times.append(ref_c4(ref, arena, moff, msz, threads))
        times = times[args.warmup:]
        v = tot / 1e9 / (sum(times) / len(times))
        sample = "%d files, %.0f MB of the %.1f GB image per step" % (len(files), tot / 1e6, args.c4_gb)
        workload = "dedup fragmenter + fragment SHA-1 + file BLAKE3, %s, reference code on %d host threads" % (sample, threads)
    else:
        arena, offs, lens = make_units(corpus, cfg, 0, args)
        threads = best_threads(ref, arena, offs, lens, method)      # doubles as warm-up
        k = max(threads * 4, int(args.ref_sample_mb * 1e6 / UNIT / (1 if cfg == "c2" else 4 if cfg == "c3" else 40)))
        k = min(len(offs), k)
        times = []
        for _ in range(args.warmup + args.steps):
            times.append(ref_compress_list(ref, arena, offs[:k], lens[:k], method, threads, roundtrip=(cfg == "c3"))[1])
        times = times[args.warmup:]
        v = k * UNIT / MB / (sum(times) / len(times))
        sample = "%d of the %d units (64 KiB each) per step" % (k, len(offs))
        workload = "%s, bounded sample: %s, reference libzpaq::compressBlock%s on %d host threads" % (
            WORKLOADS[cfg] % len(offs), sample, " + libzpaq::decompress" if cfg == "c3" else "", threads)
    line = {
        "impl": "reference", "metric": metric, "value": round(v, 3), "unit": unit, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": round(1000 * sum(times) / len(times), 2), "higher_is_better": True,
        "scaling": "strong" if cfg == "c4" else "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": {"workload": workload, "method": method, "unit_bytes": UNIT},
        "cpu_baseline": {"value": round(v, 3), "unit": unit, "cores": threads, "kind": "reference", "sample": sample},
        "e2e": {"value": round(v, 3), "unit": unit, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))
    return 0


WORKLOADS = {
    "c2": "%d x 64KiB synthetic text fragments per GPU, -m2 (x0,1,4,0,7,21,1), one compressBlock per unit",
    "c3": "%d x 64KiB blocks of an enwik-shaped synthetic corpus per GPU, -m3 (LZ77 + ICM/ISSE model), compress then decompress",
    "c5": "%d x 64KiB mixed-entropy fragments (text / random / repeats / zeros) per GPU, -m5 (22-23 component model)",
}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours")
    ap.add_argument("--config", default="c2", choices=sorted(METRICS))
    ap.add_argument("--units", type=int, default=10000, help="c2: units per GPU per step (configs[1]: 10000)")
    ap.add_argument("--c3-mb", type=int, default=100)
    ap.add_argument("--c4-gb", type=float, default=10.0, help="c4: image size, all GPUs together")
    ap.add_argument("--c5-units", type=int, default=2048, help="c5: units per GPU per step")
    ap.add_argument("--ref-sample-mb", type=float, default=400.0, help="reference arm / cpu_baseline: input MB per step (c2 scale)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-parity", action="store_true")
    ap.add_argument("--inflight", type=int, default=4,
                    help="c2: batches in flight (zq_pipe lanes): the next step's copies/kernels fill the tail of the current one")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step returned to DIR/<name>.npy")
    args = ap.parse_args()
    if args.impl == "reference":
        return run_reference(args)

    import torch
    import torch.distributed as dist
    import zpaqfranz_b200 as zq
    corpus = load_corpus()

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        print(json.dumps({"error": "no CUDA device; this benchmark has no CPU fallback"}))
        return 2
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    cfg = args.config
    metric, unit, method = METRICS[cfg]
    stream = torch.cuda.current_stream()
    ctx = zq.Context(local)
    ctx.set_stream(stream.cuda_stream)
    # the library's own communicator (zq_dist_*, NCCL): rank 0's unique id travels through the launcher's process group
    uid = None
    if world > 1:
        t = torch.zeros(128, dtype=torch.uint8, device="cuda")
        if rank == 0:
            t.copy_(torch.frombuffer(bytearray(zq.dist_unique_id()), dtype=torch.uint8))
        dist.broadcast(t, 0)
        uid = bytes(t.cpu().numpy().tobytes())
    zd = zq.Dist(local, rank, world, unique_id=uid)

    def sync_all():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    def max_over_ranks(ms):
        if world > 1:
            tt = torch.tensor([ms], device="cuda", dtype=torch.float64)
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            return float(tt.item())
        return ms

    def bracket(fn, steps):
        """device-clock ms of `steps` calls of fn(k), max over ranks"""
        sync_all()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for k in range(steps):
            fn(k)
        torch.cuda.synchronize()
        e1.record(stream)
        sync_all()
        return max_over_ranks(e0.elapsed_time(e1))

    peak, peak_src = load_peaks()
    ref = None if args.no_parity and args.no_cpu_baseline else ref_lib()
    line = None
    outputs = {}

    if cfg == "c4":
        line = run_c4(args, zq, corpus, ctx, zd, ref, rank, world, local, dist, torch, bracket, sync_all, peak, peak_src, outputs)
    else:
        arena_np, offs, lens = make_units(corpus, cfg, rank, args)
        U = len(offs)
        nbytes = U * UNIT
        h_in = torch.empty(nbytes, dtype=torch.uint8, pin_memory=True)
        h_in.numpy()[:] = arena_np
        d_in = h_in.cuda()
        cap = int(zq.lib.zq_compress_bound(UNIT)) * U
        depth = max(1, min(args.inflight, 4)) if cfg == "c2" else 1
        d_outs = [torch.empty(cap, dtype=torch.uint8, device="cuda") for _ in range(depth)]
        h_outs = [torch.empty(cap, dtype=torch.uint8, pin_memory=True) for _ in range(depth)]
        pipe = zq.Pipe(local, depth) if cfg == "c2" else None
        state = {}

        def step_device(k=0):
            state["dev"] = ctx.compress_blocks_device(d_in.data_ptr(), offs, lens, d_outs[0].data_ptr(), cap, method=method, filename="", comment="")

        def exchange(olen):
            # archive offsets of every block of every rank: all-gather of the 4-byte sizes (zq_dist_exchange_sizes, NCCL)
            state["sizes"], state["goff"] = zd.exchange_sizes(olen, U * world)

        def step_host(k=0):
            state["host"] = ctx.compress_blocks(h_in.numpy(), offs, lens, method=method, filename="", comment="", out=h_outs[0].numpy())
            if world > 1:
                exchange(state["host"][2])

        def piped(steps, device):
            sync_all()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            l0 = pipe.launch_count()
            e0.record(stream)
            tickets = []
            for k in range(steps):
                done = pipe.wait(tickets[k - depth]) if k >= depth else None
                if device:
                    tickets.append(pipe.submit(d_in.data_ptr(), offs, lens, d_outs[k % depth].data_ptr(), cap, method=method, filename="", comment="", device=True))
                else:
                    tickets.append(pipe.submit(h_in.data_ptr(), offs, lens, h_outs[k % depth].data_ptr(), cap, method=method, filename="", comment="", device=False))
                if done is not None and world > 1 and not device:
                    exchange(done[1])      # (the freed lane is already copying the next batch in)
            for t in tickets[-depth:]:
                r_ = pipe.wait(t)
                if world > 1 and not device:
                    exchange(r_[1])
            state["last"] = ((steps - 1) % depth, r_)      # the last step's output buffer, (offsets, lengths)
            torch.cuda.synchronize()
            e1.record(stream)
            sync_all()
            return max_over_ranks(e0.elapsed_time(e1)), pipe.launch_count() - l0

        sampler = ClockSampler(local)
        if cfg == "c2":
            for _ in range(max(1, args.warmup - 2)):
                step_device()
            piped(max(args.warmup, depth), True)
            sampler.start()
            ms_dev, launches = piped(args.steps, True)
            if args.dump_outputs:
                k, (ooff, olen) = state["last"]
                outputs.update(block_outputs(d_outs[k][:int((ooff + olen).max())].cpu().numpy(), ooff, olen))
            piped(max(args.warmup, depth), False)
            ms_e2e, _ = piped(args.steps, False)
            d2h_extra = h2d_extra = 0
        else:
            # c3 / c5: one context, serial steps (the model state of one batch already fills the device's parallelism)
            dstate = {}
            for _ in range(args.warmup):
                step_device()
            sampler.start()
            l0 = ctx.launch_count()
            ms_dev = bracket(step_device, args.steps)
            launches = ctx.launch_count() - l0
            if args.dump_outputs:
                ooff, olen = state["dev"]
                outputs.update(block_outputs(d_outs[0][:int((ooff + olen).max())].cpu().numpy(), ooff, olen))
            for _ in range(max(1, args.warmup - 1)):
                step_host()
            ms_e2e = bracket(step_host, args.steps)
            d2h_extra = h2d_extra = 0
            if cfg == "c3":     # the decompress half of the round trip: host buffers in and out (its only entry point)
                comp, coff, clen = state["host"]

                def step_dec(k=0):
                    dstate["dec"] = ctx.decompress_blocks(comp, coff, clen, expect_len=lens)
                for _ in range(max(1, args.warmup - 1)):
                    step_dec()
                l0 = ctx.launch_count()
                ms_dec = bracket(step_dec, args.steps)
                launches += ctx.launch_count() - l0
                if args.dump_outputs:
                    outputs.update(block_outputs(*dstate["dec"], prefix="decoded_"))
                ms_dev += ms_dec
                ms_e2e += ms_dec
                h2d_extra, d2h_extra = int(clen.sum()), nbytes
        # serial pass on one context: device time of each stage (the roofline's kernel time)
        ser_steps = min(args.steps, 3)
        stage = np.zeros(len(zq.TIMING_KEYS_EX))
        sync_all()
        for _ in range(ser_steps):
            step_device()
            t = ctx.last_timings(ex=True)
            stage += np.array([t[k] for k in zq.TIMING_KEYS_EX])
        stage /= ser_steps
        sampler.stop_flag = True
        sampler.join(timeout=3)
        step_host()
        out_np, ooff, olen = state["host"]
        out_bytes = int(olen.astype(np.int64).sum())

        # ---- parity over the WHOLE batch (outside the timed region; the checker is oracle/_ref, never the product path)
        parity, threads, cpu = "unchecked", None, None
        if rank == 0 and ref is not None and not args.no_parity:
            threads = best_threads(ref, arena_np, offs, lens, method)
            budget = U if cfg == "c2" else min(U, max(threads * 4, int(args.ref_sample_mb * 1e6 / UNIT / (4 if cfg == "c3" else 40))))
            v, dt, tot, dg, ol = ref_compress_list(ref, arena_np, offs[:budget], lens[:budget], method, threads, digests=True)
            bad = 0
            for i in range(budget):
                blk = out_np[int(ooff[i]): int(ooff[i]) + int(olen[i])]
                if int(olen[i]) != int(ol[i]) or hashlib.sha256(blk).digest() != dg[i].tobytes():
                    bad += 1
            parity = ("bit-exact, %d/%d blocks of the timed batch" % (budget - bad, budget)) if bad == 0 else "MISMATCH: %d of %d blocks differ" % (bad, budget)
            if cfg == "c3":
                back = dstate["dec"][0][:nbytes]
                parity += "; round trip " + ("restores all %d bytes" % nbytes if bytes(back) == arena_np.tobytes() else "MISMATCH")
            cpu = (v, dt, budget)

        total_units = U * world
        value = total_units * UNIT / MB / (ms_dev / 1000 / args.steps)
        e2e_v = total_units * UNIT / MB / (ms_e2e / 1000 / args.steps)
        st = dict(zip(zq.TIMING_KEYS_EX, [float(x) for x in stage]))
        kernels = {"k_sha1_units": st["sha1"], "k_suffix_sort": st["sufsort"], "k_lz_scan<0>": st["lz_scan0"], "k_lz_scan<1>": st["lz_scan1"],
                   "k_lz_walk": st["lz_walk"], "k_lz_emit": st["lz_emit"], "k_frame": st["frame"], "k_cm_encode (+k_cm_init)": st["model"]}
        if st["lz_scan0"] == 0 and st["lzparse"] > 0:
            kernels["k_lz77 (hash / general parser)"] = st["lzparse"]
        dom = max(kernels, key=lambda k: kernels[k])
        # algorithmic bytes per launch of the path (SURVEY.md section 8d): A_io = bytes_in + bytes_out; modeled methods add
        # the component state read+written per coded bit, 8 * S bytes per coded byte
        coded = 0
        if method in S_BYTES:
            coded = out_bytes   # the coder's input is the pre-pass stream: bounded below by its output; use the LZ stream when present
        a_io = nbytes + out_bytes
        algo = a_io + (8 * S_BYTES[method] * coded if method in S_BYTES else 0)
        achieved = algo / 1e9 / (kernels[dom] / 1000) if kernels[dom] > 0 else 0.0
        traffic, traffic_src = None, None
        tp = os.path.join(ROOT, "profiles", "traffic_r04.json")
        if os.path.exists(tp):
            try:
                tj = json.load(open(tp))
                e = tj.get(cfg, {}).get(dom)
                if e and int(e.get("units", 0)) == U:
                    traffic, traffic_src = int(e["dram_bytes"]), e.get("source")
            except Exception:
                pass
        line = {
            "metric": metric, "value": round(value, 2), "unit": unit, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": round(ms_dev / args.steps, 3), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "u8", "data": "synthetic",
            "config": {"workload": WORKLOADS[cfg] % U, "method": method, "units_per_gpu": U, "unit_bytes": UNIT,
                       "parallelism": "units sharded over the ranks, no data-path collective; per step one all-gather of the 4-byte block sizes "
                                      "(zq_dist_exchange_sizes over NCCL, inside the e2e region) -> global archive offsets" if world > 1 else
                                      "one rank: units on one GPU, no collective",
                       "exchanged_bytes_per_rank": zd.bytes_exchanged(),
                       "l2": "inputs %.0f MB per step > 126 MB L2 (no flush needed)" % (nbytes / MB), "parity": parity,
                       "inflight": depth, "serial_ms_per_step": round(float(st["total"]), 3),
                       "compressed_ratio": round(out_bytes / nbytes, 4)},
            "e2e": {"value": round(e2e_v, 2), "unit": unit, "h2d_bytes_per_step": nbytes + h2d_extra, "d2h_bytes_per_step": out_bytes + d2h_extra,
                    "ms_per_step": round(ms_e2e / args.steps, 3)},
            "gpu_launches": int(launches),
            "stage_ms": {k: round(v, 3) for k, v in st.items()},
            "roofline": {"bound": "hbm", "kernel": dom, "achieved": round(achieved, 2), "peak": peak, "unit": "GB/s",
                         "frac": round(achieved / peak, 5), "traffic": traffic, "traffic_source": traffic_src,
                         "algorithmic_bytes_per_launch": int(algo),
                         "algorithmic_bytes_rule": "A_io = bytes_in + bytes_out of the batch" + (" + 8*S*coded bytes, S=%d" % S_BYTES[method] if method in S_BYTES else ""),
                         "kernel_ms": round(float(kernels[dom]), 3), "kernel_ms_all": {k: round(v, 3) for k, v in kernels.items() if v > 0},
                         "whole_step_frac": round(a_io / 1e9 / (st["total"] / 1000) / peak, 5) if st["total"] > 0 else None,
                         "peak_source": peak_src},
            "clocks": sampler.summary(),
        }
        if cfg == "c3":
            line["config"]["note"] = "decompress has no device-pointer entry point: its time is host-to-host in value and e2e alike"
        if rank == 0 and cpu is not None and not args.no_cpu_baseline:
            line["cpu_baseline"] = {"value": round(cpu[0], 2), "unit": unit, "cores": threads, "kind": "reference",
                                    "sample": "%d of the %d units (64 KiB each), compress only, all host threads, %.1f s" % (cpu[2], U, cpu[1])}
        if pipe is not None:
            pipe.close()
    if rank == 0:
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, outputs)
        print(json.dumps(line))
    zd.close()
    ctx.close()
    if world > 1:
        dist.destroy_process_group()
    return 0


def run_c4(args, zq, corpus, ctx, zd, ref, rank, world, local, dist, torch, bracket, sync_all, peak, peak_src, outputs):
    """Fragmenter + fragment SHA-1 + per-file BLAKE3 over this rank's share of the image; digests all-gathered."""
    sizes, kinds, srcs = make_image(corpus, int(args.c4_gb * 1e9))
    # files dealt to the ranks longest first (LPT): every rank computes the same assignment
    order = np.argsort(-sizes, kind="stable")
    load = np.zeros(world, dtype=np.int64)
    mine = []
    for f in order:
        r = int(np.argmin(load))
        load[r] += sizes[f]
        if r == rank:
            mine.append(int(f))
    mine.sort()
    msz = sizes[mine].astype(np.uint64)
    nbytes = int(msz.sum())
    h_in = torch.empty(nbytes, dtype=torch.uint8, pin_memory=True)
    a, moff, msz = build_files(corpus, mine, sizes, kinds, srcs, out=h_in.numpy())
    res = {}

    def step(k=0):
        res["frag"] = ctx.fragment(a, moff, msz, fragment=6, want_sha1=True)
        res["b3"] = ctx.blake3(a, moff, msz)
    for _ in range(args.warmup):
        step()
    sampler = ClockSampler(local)
    sampler.start()
    l0 = ctx.launch_count()
    ms = bracket(step, args.steps)
    launches = ctx.launch_count() - l0
    sampler.stop_flag = True
    sampler.join(timeout=3)
    fl, fh, fs, first = res["frag"]
    if args.dump_outputs:
        outputs.update({"fragment_lengths": fl.astype(np.float64), "fragment_hits": fh.astype(np.float64),
                        "fragment_sha1": fs.astype(np.float32), "file_first_fragment": first.astype(np.float64),
                        "file_blake3": np.asarray(res["b3"]).astype(np.float32)})
    # dedup key exchange: 20-byte digests of every rank's fragments -> global unique count (the index the archiver keeps)
    nfrag = len(fl)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    is_first, uniq = zd.dedup(fs)            # zq_dist_dedup: all-gather of the 20-byte digests over NCCL, first occurrence wins
    t_x = time.perf_counter() - t0
    cnt = torch.tensor([nfrag, int(is_first.sum())], device="cuda", dtype=torch.int64)
    if world > 1:
        dist.all_reduce(cnt)
    tot_frag = int(cnt[0].item())
    assert int(cnt[1].item()) == uniq, "dedup bookkeeping differs between the ranks"
    # parity: every fragment table and digest of a bounded prefix of this rank's files against the reference
    parity, cpu = "unchecked", None
    if rank == 0 and ref is not None and not args.no_parity:
        budget_bytes, bad, k, checked = args.ref_sample_mb * 1e6 * 2, 0, 0, 0
        t0 = time.perf_counter()
        for j, f in enumerate(mine):
            d = a[int(moff[j]): int(moff[j]) + int(msz[j])].tobytes()
            rl, rh = ref.fragment(d, 6)
            x, y = int(first[j]), int(first[j + 1])
            ok = (y - x == len(rl)) and bool((fl[x:y] == rl).all()) and bool((fh[x:y] == rh).all())
            o = 0
            for q in range(x, y if ok else x):
                ok = ok and fs[q].tobytes() == ref.sha1(d[o:o + int(fl[q])])
                o += int(fl[q])
            ok = ok and res["b3"][j].tobytes() == ref.blake3(d)
            bad += 0 if ok else 1
            k += 1
            checked += len(d)
            if checked >= budget_bytes:
                break
        dt = time.perf_counter() - t0
        parity = ("bit-exact, %d/%d files (fragment tables, hit counts, SHA-1 of every fragment, BLAKE3), %.0f MB" % (k - bad, k, checked / 1e6)
                  if bad == 0 else "MISMATCH in %d of %d files" % (bad, k))
        nthr = os.cpu_count() or 1
        kk = int(np.searchsorted(np.cumsum(msz.astype(np.int64)), args.ref_sample_mb * 1e6 * 8)) + 1
        kk = min(kk, len(mine))
        ref_c4(ref, a, moff[:8], msz[:8], nthr)
        dt2 = ref_c4(ref, a, moff[:kk], msz[:kk], nthr)
        cpu = (float(msz[:kk].sum()) / 1e9 / dt2, dt2, kk, nthr)
    total = float(sizes.sum())
    value = total / 1e9 / (ms / 1000 / args.steps)
    out_b = tot_frag * 28 + len(sizes) * 32     # fragment length + hits + 20-byte digest, 32-byte file digest
    line = {
        "metric": METRICS["c4"][0], "value": round(value, 3), "unit": "GB/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": round(ms / args.steps, 3), "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "u8",
        "data": "synthetic",
        "config": {"workload": "dedup fragmenter (-fragment 6) + SHA-1 of every fragment + BLAKE3 of every file over a %.1f GB synthetic "
                               "filesystem image of %d files (log-normal sizes <= 64 MiB; text / random / copies / zero pages), files dealt to "
                               "the ranks longest first" % (total / 1e9, len(sizes)),
                   "files": int(len(sizes)), "image_bytes": int(total), "fragments": tot_frag, "unique_fragments": int(uniq),
                   "parallelism": "files sharded over the ranks; one all-gather of the 20-byte fragment digests (zq_dist_dedup over NCCL: %.1f ms, %d bytes received per rank, outside the step)" % (t_x * 1e3, zd.bytes_exchanged()),
                   "l2": "inputs %.0f MB per rank per step > 126 MB L2" % (nbytes / MB), "parity": parity,
                   "note": "host buffers in, tables out: value == e2e (this path has no device-pointer entry point); a file is never split across GPUs"},
        "e2e": {"value": round(value, 3), "unit": "GB/s", "h2d_bytes_per_step": int(2 * nbytes), "d2h_bytes_per_step": int(out_b // world),
                "ms_per_step": round(ms / args.steps, 3)},
        "gpu_launches": int(launches),
        "roofline": {"bound": "hbm", "kernel": "k_fragment_round + k_sha1_many + k_blake3_chunks (whole step)", "achieved": round(2 * total / 1e9 / (ms / 1000 / args.steps), 2),
                     "peak": peak, "unit": "GB/s", "frac": round(2 * total / 1e9 / (ms / 1000 / args.steps) / peak / world, 5), "traffic": None,
                     "algorithmic_bytes_per_launch": int(2 * total), "algorithmic_bytes_rule": "1.0003 B per input byte for fragmenter + SHA-1, 1 B per byte for BLAKE3; the step includes the H2D copies",
                     "peak_source": peak_src},
        "clocks": sampler.summary(),
    }
    if cpu is not None and not args.no_cpu_baseline:
        line["cpu_baseline"] = {"value": round(cpu[0], 3), "unit": "GB/s", "cores": cpu[3], "kind": "reference",
                                "sample": "%d of this rank's files (fragmenter loop + libzpaq::SHA1 per fragment + BLAKE3 per file), all host threads, %.1f s" % (cpu[2], cpu[1])}
    return line


if __name__ == "__main__":
    sys.exit(main())
