#!/usr/bin/env python
"""bench.py — model-load throughput of the kukeon GPU weight loader (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W            # our arm  (torchrun for N > 1)
    python bench.py --impl reference --gpus N --steps K ...   # CPU arm: the oracle port on host cores
    python bench.py ... --dump-outputs DIR                    # also write a seeded sample of the pool after the timed steps

Workload (config.workload): Llama-3-8B bf16, 291 tensors / 4 safetensors shards / 16,060,522,496 B, synthetic
content, files warm in tmpfs/page cache.  A "step" = one pass of the hot path over the whole checkpoint:

* `value`  (GB/s): kernel stage with the checkpoint bytes already resident in HBM — one convert/fan-out launch
  per shard, timed with CUDA events on the launching stream inside the library (kk_convert_resident), max over
  ranks.  At N > 1 every rank converts 1/N of the checkpoint and the same kernel stores it into all N pools over
  NVLink (P2P), so value counts N x checkpoint bytes made resident per step ("weak": bytes per pool fixed).
* `e2e`    (GB/s): the same through the public call a user makes (modelhub.Load -> kk_load_part) with HOST
  buffers: CPU copy from the warm files into the pinned ring, H2D copies, kernels, and a device->host read of a
  result (pool checksum word) plus kk_export, all inside the timed region.
* `roofline`: dominant kernel kk_convert_kernel.  N = 1: bound "hbm", algorithmic bytes = 2 x shard bytes (2 B read + 2 B written
  per bf16 element) / its CUDA-event duration, against MEASURED_PEAKS.json's hbm_gbs.  N > 1 broadcast: bound "nvlink", the
  bytes every GPU has to receive ((N-1)/N of the pool) / the fan-out stage's CUDA-event time, against a peer-copy rate measured
  in the same run (every rank reading from its ring neighbour at once, kk_probe_peer) and against 900 GB/s nominal.
* `cpu_baseline`: the oracle's C port (oracle/kk_oracle.c, OpenMP, all host threads) over the WHOLE checkpoint.
* `secondary` (N = 1, default workload): the same kernel stage on a 4-layer Mixtral q4_K GGUF — the expanding conversion for which
  the north_star's HBM-write fraction is meaningful (a bf16 copy has to read what it writes and tops out near 0.5 of it).

The reference (eminwux/kukeon) has no loader and Go is absent, so `--impl reference` times that same CPU port
(kind "port") — see DESIGN.md.
"""
from __future__ import annotations

import argparse
import gc
import json
import os
import shutil
import statistics
import subprocess
import sys
import threading
import time
import zlib

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

METRIC = "model_load_GBps"
UNIT = "GB/s"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5, help="timed steps of every timed loop (kernel stage, e2e, CPU baseline, secondary records)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--dump-outputs", default="", metavar="DIR",
                    help="after the timed steps, write what the last one made resident (rank 0's pool, tensor by tensor as its manifest describes it) "
                         "to DIR/<tensor name>.npy, a seeded sample of large tensors, at most 64 MB in all (see dump_outputs)")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="llama3-8b", choices=["llama3-8b", "mixtral-q4k", "gpt2", "llama3-70b-scatter"])
    ap.add_argument("--qtype", default="Q4_K", help="mixtral-q4k: block type of the weights (Q4_K = the BASELINE config; Q4_0, Q5_K, IQ4_XS, ... "
                    "measure the other dequantisers at the same shapes)")
    ap.add_argument("--layers", type=int, default=0, help="override the layer count (reported in config; 0 = full size)")
    ap.add_argument("--data-dir", default="")
    ap.add_argument("--gen-only", action="store_true", help="internal: write the synthetic checkpoint into --data-dir and exit (run as a child process by make_files)")
    ap.add_argument("--no-interleave", action="store_true", help="do not spread the synthetic files' page-cache pages over the NUMA nodes")
    ap.add_argument("--keep-data", action="store_true")
    ap.add_argument("--readers", type=int, default=0)
    ap.add_argument("--slots", type=int, default=0)
    ap.add_argument("--slot-mb", type=int, default=0)
    ap.add_argument("--zerocopy", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--nccl-compare", action="store_true", help="also time an NCCL all-gather of the pools (comparison collective)")
    ap.add_argument("--nvls-compare", action="store_true", help="N > 1: also time the kernel stage with KK_FANOUT_NVLS (multimem.st through the NVSwitch multicast object) "
                    "against KK_FANOUT_P2P, both in the one-process-all-GPUs shape (rank 0)")
    ap.add_argument("--kernel-only", action="store_true", help="profiling aid: skip the streaming load / e2e legs (every kk_convert launch is a resident one)")
    ap.add_argument("--e2e-only", action="store_true", help="tuning aid: skip the resident kernel leg")
    ap.add_argument("--no-numa-pin", action="store_true")
    ap.add_argument("--eager-peers", action="store_true", help="enable peer access to every GPU in kk_open (A/B for time-to-ready)")
    ap.add_argument("--no-exchange", action="store_true", help="scatter: every rank gathers its own column runs from the file (no NVLink row exchange)")
    ap.add_argument("--no-single-process", action="store_true", help="skip the one-process-all-GPUs time-to-ready measurement at N > 1")
    ap.add_argument("--no-secondary", action="store_true", help="N = 1 default workload: skip the short Mixtral q4_K record (`secondary`)")
    ap.add_argument("--fanout", default="auto", choices=["auto", "p2p", "raw", "pull"],
                    help="broadcast order: fused convert+fan-out by P2P stores (p2p), all-gather the file bytes then convert locally (raw), or convert into own "
                         "pool + slice buffer and pull the peers' slices (pull: peers map 1/N of the bytes).  auto = p2p (measured best on every count at N = 8)")
    a = ap.parse_args()
    if a.dump_outputs and a.impl == "reference":
        ap.error("--dump-outputs writes the GPU pool; the CPU arm (--impl reference) has none")
    if a.fanout == "auto":
        # Measured at N = 8 (profiles/README.md, round 2): with pools in 2 MiB multiples the seven 16 GB pool mappings of the P2P-store order take
        # 0.05-0.07 s (3.6 s in round 1), so it has the shorter time-to-ready, the faster kernel stage (20.0 vs 25.2 ms) and the faster e2e step
        # (156 vs 183 ms: its fan-out overlaps the ingest).  PULL stays available for deployments where peers must not map whole pools.
        a.fanout = "p2p"
    return a


# ---------------------------------------------------------------------------------------------
# workload files
# ---------------------------------------------------------------------------------------------
def workload_spec(args):
    from tools import synth
    if args.workload == "llama3-8b":
        cfg = dict(synth.LLAMA3_8B)
        if args.layers:
            cfg["layers"] = args.layers
        t = synth.llama_tensors(**cfg)
        name = "Llama-3-8B bf16 safetensors" + (f" (REDUCED to {args.layers} layers)" if args.layers else "")
        return dict(kind="llama", cfg=cfg, tensors=t, name=name, mode="broadcast")
    if args.workload == "llama3-70b-scatter":
        cfg = dict(synth.LLAMA3_70B)
        if args.layers:
            cfg["layers"] = args.layers
        t = synth.llama_tensors(**cfg)
        name = "Llama-3-70B bf16 safetensors scatter" + (f" (REDUCED to {args.layers} layers)" if args.layers else "")
        return dict(kind="llama", cfg=cfg, tensors=t, name=name, mode="scatter")
    if args.workload == "mixtral-q4k":
        kw = dict(layers=args.layers) if args.layers else {}
        if args.qtype not in synth.GGML or synth.GGML[args.qtype][1] == 1:
            raise SystemExit(f"--qtype {args.qtype}: not a block-quantised GGUF type this tool can write")
        t = synth.mixtral_gguf_tensors(qtype=args.qtype, **kw)
        name = f"Mixtral-8x7B GGUF {args.qtype.lower()} -> bf16" + (f" (REDUCED to {args.layers} layers)" if args.layers else "")
        return dict(kind="gguf", tensors=t, name=name, mode="broadcast")
    if args.layers:  # test-sized: the reduced model also gets a 4096-entry vocabulary (wte is 154 of the full model's 498 MB)
        t = synth.gpt2_tensors(n_layer=args.layers, vocab=4096)
        return dict(kind="gpt2", tensors=t, name=f"GPT-2-small f32 safetensors (REDUCED to {args.layers} layers, vocabulary 4096)", mode="broadcast")
    t = synth.gpt2_tensors()
    return dict(kind="gpt2", tensors=t, name="GPT-2-small f32 safetensors", mode="broadcast")


def pick_data_dir(args, need_bytes: int) -> str:
    if args.data_dir:
        return args.data_dir
    for base in ("/dev/shm", "/tmp"):
        try:
            st = os.statvfs(base)
            if st.f_bavail * st.f_frsize > need_bytes * 1.15 + (2 << 30):
                return os.path.join(base, f"kk_bench_{args.workload}_{args.layers}")
        except OSError:
            pass
    raise SystemExit(f"no directory with {need_bytes / 1e9:.1f} GB free for the synthetic checkpoint")


def interleave_new_pages(on: bool) -> bool:
    """set_mempolicy(MPOL_INTERLEAVE over every online node) for this thread while the synthetic checkpoint is written, so that its tmpfs /
    page-cache pages are spread over the host's NUMA nodes — the neutral placement for a file that N readers on both sockets are about to read
    (a checkpoint read from disk by the per-GPU reader threads would even land on each reader's own node).  Written from one process without
    this, every page sits on the writer's node and the four ranks of the other socket pull their parts through the inter-socket link.
    Returns whether the policy was applied (False: single node, or the syscall is unavailable)."""
    import ctypes
    try:
        nodes = []
        for part in open("/sys/devices/system/node/online").read().strip().split(","):
            lo, _, hi = part.partition("-")
            nodes += list(range(int(lo), int(hi or lo) + 1))
        if len(nodes) < 2:
            return False
        mask = ctypes.c_ulong(sum(1 << n for n in nodes) if on else 0)
        libc = ctypes.CDLL(None, use_errno=True)
        rc = libc.syscall(238, 3 if on else 0, ctypes.byref(mask) if on else None, 65 if on else 0)  # x86-64 set_mempolicy; MPOL_INTERLEAVE = 3, MPOL_DEFAULT = 0
        return rc == 0
    except Exception:  # noqa: BLE001
        return False


def warm_page_cache(d: str, rank: int, world: int, passes: int = 2, threads: int = 8, block: int = 32 << 20) -> int:
    """Read this rank's stripe (blocks i with i % world == rank) of every regular file under d `passes` times; returns the bytes read per pass."""
    files = sorted(os.path.join(d, f) for f in os.listdir(d) if os.path.isfile(os.path.join(d, f)) and not f.startswith("."))
    jobs, i = [], 0
    for f in files:
        n = os.path.getsize(f)
        for off in range(0, n, block):
            if i % world == rank:
                jobs.append((f, off, min(block, n - off)))
            i += 1

    def work(k):
        buf = bytearray(block)
        fds = {}
        for _ in range(passes):
            for f, off, ln in jobs[k::threads]:
                fd = fds.get(f)
                if fd is None:
                    fd = fds[f] = os.open(f, os.O_RDONLY)
                got = 0
                while got < ln:
                    r = os.preadv(fd, [memoryview(buf)[got:ln]], off + got)
                    if r <= 0:
                        break
                    got += r
        for fd in fds.values():
            os.close(fd)

    th = [threading.Thread(target=work, args=(k,)) for k in range(threads)]
    for t in th:
        t.start()
    for t in th:
        t.join()
    return sum(j[2] for j in jobs)


_INTERLEAVED = None


def make_files(spec, d: str, args=None) -> str:
    """Synthetic checkpoint under d (once; `.complete` marks it).  Written by a CHILD process (`bench.py --gen-only`): the NUMA interleave policy
    it sets — inherited by the generator's OpenMP workers — must not stay on this process's threads, whose first-touch placement the CPU arm
    depends on."""
    global _INTERLEAVED
    marker = os.path.join(d, ".complete")
    if not os.path.exists(marker):
        if args is None or getattr(args, "gen_only", False):
            generate_files_here(spec, d)
        else:
            cmd = [sys.executable, os.path.abspath(__file__), "--gen-only", "--workload", args.workload, "--qtype", args.qtype, "--layers", str(args.layers), "--data-dir", d]
            if getattr(args, "no_interleave", False):
                cmd.append("--no-interleave")
            subprocess.run(cmd, check=True, stdout=subprocess.DEVNULL)
    _INTERLEAVED = open(marker).read().strip() == "interleaved"
    return d if spec["kind"] != "gguf" else os.path.join(d, "model.gguf")


def generate_files_here(spec, d: str, interleave: bool = True) -> None:
    from tools import synth
    shutil.rmtree(d, ignore_errors=True)
    os.makedirs(d)
    il = interleave_new_pages(True) if interleave else False
    _write_files(spec, d, synth)
    open(os.path.join(d, ".complete"), "w").write("interleaved" if il else "ok")


def _write_files(spec, d: str, synth) -> None:
    if spec["kind"] == "llama":
        synth.write_sharded(d, spec["tensors"], 8001, 5_000_000_000)
    elif spec["kind"] == "gguf":
        synth.write_gguf(os.path.join(d, "model.gguf"), spec["tensors"], 8007)
    else:
        synth.write_safetensors(os.path.join(d, "model.safetensors"), spec["tensors"], 1234)


# ---------------------------------------------------------------------------------------------
# clocks
# ---------------------------------------------------------------------------------------------
class ClockSampler:
    Q = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, gpu: int):
        self.gpu, self.rows, self.p = gpu, [], None

    def start(self):
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100", "-i", str(self.gpu)],
                                      stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except OSError:
            self.p = None

    def _read(self):
        for line in self.p.stdout:
            self.rows.append((time.time(), [x.strip() for x in line.split(",")]))

    def stop(self, t0: float, t1: float) -> dict:
        if self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.p.terminate()
        rows = [r for t, r in self.rows if t0 - 0.05 <= t <= t1 + 0.15 and len(r) >= 8] or [r for _, r in self.rows if len(r) >= 8]
        if not rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        sm = [float(r[1]) for r in rows]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({n for r in rows for n, v in zip(names, r[4:8]) if v.lower().startswith("active")})
        return {"sm_mhz": statistics.median(sm), "sm_max_mhz": float(rows[0][2]), "reasons": reasons, "samples": len(rows),
                "power_w_max": max(float(r[3]) for r in rows)}


# ---------------------------------------------------------------------------------------------
# CPU arm (oracle port) — the only place bench.py touches oracle/
# ---------------------------------------------------------------------------------------------
def cpu_port_setup(path: str, sample_bytes: int | None = None):
    """Jobs over the whole checkpoint (sample_bytes None) and an UNTOUCHED output buffer: its pages are first touched by the untimed warm-up
    pass, i.e. by the OpenMP thread that writes them in every later pass (orc_cpu_load schedules jobs statically), so the buffer ends up
    spread over both sockets.  Round 1 touched it from one thread — everything on one NUMA node — and the same port read 9 GB/s on one box
    and 50 GB/s on the next."""
    from oracle import coracle, oracle
    shards, recs = oracle.index_path(path)
    plan, total = oracle.plan_pool(recs)
    jobs, src = coracle.make_jobs(recs, plan, job_bytes=8 << 20, max_src_bytes=sample_bytes)
    hi = max((j.dst_off + j.nbytes // coracle._UNITS[j.op][0] * coracle._UNITS[j.op][1] for j in jobs), default=0)
    pool = np.empty(min(total, hi) + 4096, np.uint8)
    return coracle, shards, jobs, src, pool


def cpu_port_step(ctx) -> float:
    coracle, shards, jobs, src, pool = ctx
    t = time.perf_counter()
    coracle.cpu_load(shards, jobs, pool, threads=os.cpu_count() or 1)  # explicit: torchrun exports OMP_NUM_THREADS=1
    return time.perf_counter() - t


def run_reference(args, spec, path, file_bytes):
    """--impl reference: the CPU port of the load path on all host threads (kind "port": the reference has no
    loader and cannot be built here)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    ctx = cpu_port_setup(path, None if file_bytes <= (40 << 30) else 40 << 30)  # whole checkpoint for every BASELINE config that fits a step into seconds
    cores = os.cpu_count() or 1
    for _ in range(max(min(args.warmup, 3), 1)):  # the first pass is also the parallel first touch of the output buffer
        cpu_port_step(ctx)
    ts = [cpu_port_step(ctx) for _ in range(args.steps)]
    tot = sum(ts)
    v = ctx[3] * args.steps / tot / 1e9
    line = {
        "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": tot / args.steps * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16",
        "data": "synthetic", "config": {"workload": spec["name"], "file_bytes": file_bytes,
                                        "files": "warm in tmpfs/page cache" + (", pages interleaved over the host's NUMA nodes" if _INTERLEAVED else ""),
                                        "same_config": ctx[3] == file_bytes},
        "cpu_baseline": {"value": v, "unit": UNIT, "cores": cores, "kind": "port",
                         "sample": (("the whole checkpoint" if ctx[3] == file_bytes else f"first {ctx[3] / 1e9:.2f} GB of the checkpoint") +
                                    f" ({ctx[3] / 1e9:.2f} GB) per step, pread + convert into host memory (oracle/kk_oracle.c, OpenMP static schedule, "
                                    "output pages first-touched by their writers)")},
        "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


# ---------------------------------------------------------------------------------------------
# our arm
# ---------------------------------------------------------------------------------------------
_REAL_STDOUT = None


def emit(line: dict) -> None:
    """The one JSON line goes to the real stdout; fd 1 itself is pointed at stderr while the benchmark runs so that
    native libraries (NCCL's version banner, ...) cannot interleave with it."""
    data = (json.dumps(line) + "\n").encode()
    if _REAL_STDOUT is not None:
        os.write(_REAL_STDOUT, data)
    else:
        sys.stdout.write(data.decode())
        sys.stdout.flush()


DUMP_BYTES = 48 << 20  # --dump-outputs: values written for all tensors together (the files, .npy headers included, stay under 64 MB)
DUMP_RUN = 4096        # elements per sampled run of a large tensor
# pool dtype -> (element type as stored, type written); FP8, sub-byte and block-quantised types are written as their bytes, one value per byte
_DUMP_TYPES = {"BF16": (np.uint16, np.float32), "F16": (np.float16, np.float32), "F32": (np.float32, np.float32), "F64": (np.float64, np.float64),
               **{k: (v, np.float64) for k, v in (("BOOL", np.uint8), ("U8", np.uint8), ("I8", np.int8), ("U16", np.uint16), ("I16", np.int16),
                                                  ("U32", np.uint32), ("I32", np.int32), ("U64", np.uint64), ("I64", np.int64))}}
_DUMP_BYTEWISE = (np.uint8, np.float32)


def _dump_values(raw: np.ndarray, dtype: str) -> np.ndarray:
    src, dst = _DUMP_TYPES.get(dtype, _DUMP_BYTEWISE)
    v = raw.view(src)
    if dtype == "BF16":
        return (v.astype(np.uint32) << 16).view(np.float32)
    return v.astype(dst)


def dump_outputs(out_dir: str, tensors, read) -> None:
    """--dump-outputs: what a caller of the timed path receives — every tensor of the pool, as the manifest describes it — written as
    out_dir/<tensor name>.npy.  `read(offset, nbytes)` returns pool bytes.  A tensor whose values fit its share of DUMP_BYTES is written whole in
    its shape; a larger one as the 1-D concatenation of runs of DUMP_RUN elements drawn with a seed taken from its name, so that the same
    arguments select the same elements in every run and two builds can be compared output for output."""
    os.makedirs(out_dir, exist_ok=True)
    share = DUMP_BYTES // max(len(tensors), 1)
    for t in tensors:
        src, dst = _DUMP_TYPES.get(t["dtype"], _DUMP_BYTEWISE)
        isz = np.dtype(src).itemsize
        n, per = t["nbytes"] // isz, share // np.dtype(dst).itemsize
        if n <= per:
            vals = _dump_values(read(t["offset"], n * isz), t["dtype"])
            if n == int(np.prod(t["shape"])):
                vals = vals.reshape(t["shape"])
        else:
            run = min(DUMP_RUN, per)
            rng = np.random.default_rng(zlib.crc32(t["name"].encode()))
            starts = np.sort(rng.choice(n // run, per // run, replace=False)) * run
            vals = np.concatenate([_dump_values(read(t["offset"] + int(s) * isz, run * isz), t["dtype"]) for s in starts])
        with open(os.path.join(out_dir, t["name"].replace(os.sep, "_") + ".npy"), "wb") as f:
            np.save(f, vals)


def main():
    global _REAL_STDOUT
    args = parse()
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    spec = workload_spec(args)
    from tools import synth
    if args.gen_only:
        generate_files_here(spec, args.data_dir, interleave=not args.no_interleave)
        return
    file_bytes = synth.total_bytes(spec["tensors"])
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    N = args.gpus
    if world != N and not (world == 1 and N == 1):
        if args.impl == "reference" and world == 1:
            pass
        else:
            raise SystemExit(f"--gpus {N} but WORLD_SIZE={world}: launch with torchrun --nproc-per-node {N}")

    d = pick_data_dir(args, file_bytes)
    if args.impl == "reference":
        if rank == 0:
            path = make_files(spec, d, args)
            run_reference(args, spec, path, file_bytes)
            if not args.keep_data:
                shutil.rmtree(d, ignore_errors=True)
        return

    import torch
    import torch.distributed as dist
    from kukeon_b200 import gpupool, modelhub

    gpupool.lib()
    if not torch.cuda.is_available():
        raise SystemExit("bench.py (our arm) needs a CUDA device: the loader has no CPU path")
    torch.cuda.set_device(local)
    gloo = None
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
        gloo = dist.new_group(backend="gloo")

    def barrier():
        if world > 1:
            dist.barrier(group=gloo)

    def allmax(x: float) -> float:
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX, group=gloo)
        return float(t.item())

    def allsum(x: float) -> float:
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.SUM, group=gloo)
        return float(t.item())

    t_gen = time.time()
    if rank == 0:
        path = make_files(spec, d, args)
    barrier()
    path = d if spec["kind"] != "gguf" else os.path.join(d, "model.gguf")
    t_gen = time.time() - t_gen
    # "files warm in the page cache" means they have been READ before, not only written: the first read of freshly written tmpfs pages by 8 x 16
    # threads is an order of magnitude slower than every later one (measured on a fresh 8-GPU box: 1.33 s of pread per reader thread in the cold
    # load against 0.11 s when the same files had been loaded once before — profiles/r02/bench_n8_first_vs_second_run.txt; the kernel promotes
    # pages to the active LRU list on re-reference, under a lock all readers share).  So every rank reads its stripe of the files twice, untimed.
    t_warm = time.time()
    warm_page_cache(d, rank, world)
    barrier()
    t_warm = time.time() - t_warm

    mode = gpupool.MODE_SINGLE if world == 1 else (gpupool.MODE_SCATTER if spec["mode"] == "scatter" else gpupool.MODE_BROADCAST)
    flags = (gpupool.CFG_ZEROCOPY if args.zerocopy else 0) | (gpupool.CFG_NO_NUMA_PIN if args.no_numa_pin else 0)
    if world > 1 and args.eager_peers:
        flags |= gpupool.CFG_PEER_ALL  # measured: does not shorten cudaIpcOpenMemHandle (the mapping itself is the cost)
    t0 = time.time()
    pool = gpupool.Pool([local], n_staging_buffers=args.slots, staging_buffer_bytes=args.slot_mb << 20, n_reader_threads=args.readers, flags=flags)
    t_open = time.time() - t0

    # ---- cold path once: index + plan + pool allocation (+ peer exchange), then time-to-agent-ready ----------
    barrier()
    t_ready0 = time.time()
    brk = {}
    ref = modelhub.Pull(path)
    brk["pull_s"] = time.time() - t_ready0
    lflags = gpupool.LOAD_DEFER | (gpupool.LOAD_GPT2_CONV1D_T if spec["kind"] == "gpt2" else 0)
    exchange = world > 1 and mode == gpupool.MODE_SCATTER and not args.no_exchange
    if exchange:
        lflags |= gpupool.LOAD_SCATTER_EXCHANGE
    t1 = time.time()
    raw_order = args.fanout == "raw" and world > 1 and mode == gpupool.MODE_BROADCAST
    pull_order = args.fanout == "pull" and world > 1 and mode == gpupool.MODE_BROADCAST
    two_stage = raw_order or pull_order  # kk_load_part / kk_convert_resident = stage 1, barrier, kk_convert_local = stage 2
    m = modelhub.Load(pool, ref, mode=mode, fanout=gpupool.FANOUT_RAW if raw_order else gpupool.FANOUT_PULL if pull_order else gpupool.FANOUT_P2P, flags=lflags,
                      part_index=rank if world > 1 else 0, part_count=world if world > 1 else 0)
    brk["plan_alloc_s"] = time.time() - t1
    t1 = time.time()
    which = gpupool.BUF_RAW if raw_order else gpupool.BUF_SLICE if pull_order else gpupool.BUF_POOL
    attach_thread = None
    if world > 1 and (mode == gpupool.MODE_BROADCAST or exchange):
        h = m.export_buffer(local, which)
        hs = [None] * world
        dist.all_gather_object(hs, h, group=gloo)
        brk["handle_exchange_s"] = time.time() - t1
        t1 = time.time()

        def attach_all():
            ta = time.time()
            for k in range(1, world):  # ring order: the ranks do not all open rank 0's buffer first
                r = (rank + k) % world
                m.peer_attach_buffer(r, which, hs[r])
            brk["peer_attach_s"] = time.time() - ta

        if pull_order and not args.kernel_only:
            # PULL: stage 1 writes only this rank's own pool and slice buffer, so the peers' slice buffers are mapped (cudaIpcOpenMemHandle,
            # the expensive part of time-to-ready in this shape) on a second thread WHILE the part is being read, copied and converted
            attach_thread = threading.Thread(target=attach_all)
            attach_thread.start()
        else:
            attach_all()
    t1 = time.time()
    if attach_thread is None:
        barrier()
    if args.kernel_only:
        m.stage_resident()
        barrier()
        m.convert_resident()
        if two_stage:
            barrier()
            m.convert_local()
    else:
        brk["barrier_s"] = time.time() - t1
        t1 = time.time()
        m.load_part()
        brk["stage1_s"] = time.time() - t1
        if attach_thread is not None:
            attach_thread.join()
            brk["attach_wait_after_stage1_s"] = time.time() - t1 - brk["stage1_s"]
        if two_stage:
            barrier()
            m.convert_local()
        brk["load_part_s"] = time.time() - t1
    t1 = time.time()
    handle, manifest = m.export(local)
    brk["export_s"] = time.time() - t1
    brk["wall_before_final_barrier_s"] = time.time() - t_ready0
    barrier()
    t_ready = None if args.kernel_only else allmax(time.time() - t_ready0)
    t_ready_incl_open = None if t_ready is None else allmax(time.time() - t_ready0 + t_open)
    st0 = m.stats()
    rd = st0.get("readers") or {}
    if rd.get("threads"):  # where the reader threads of the cold load spent their time: average seconds per thread
        for k in ("slot_wait_s", "pread_s", "issue_s", "drain_s"):
            brk["readers_avg_" + k] = rd[k] / rd["threads"]
    brk_max = None
    if world > 1:  # the slowest rank decides time-to-ready: per component, the maximum over ranks and the rank that had it
        allb = [None] * world
        dist.all_gather_object(allb, brk, group=gloo)
        brk_max = {k: (lambda vals: {"s": max(vals), "rank": vals.index(max(vals))})([b.get(k, 0.0) for b in allb]) for k in brk}

    # pinned H2D probe (plumbing; tells what the PCIe link of this box can do for the e2e leg)
    h2d_probe = None
    try:
        hb = torch.empty(1 << 30, dtype=torch.uint8).pin_memory()
        db = torch.empty(1 << 30, dtype=torch.uint8, device=f"cuda:{local}")
        db.copy_(hb, non_blocking=True)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(3):
            db.copy_(hb, non_blocking=True)
        e1.record()
        torch.cuda.synchronize()
        h2d_probe = 3 * (1 << 30) / (e0.elapsed_time(e1) / 1e3) / 1e9
        del hb, db
    except Exception:  # noqa: BLE001
        pass

    # ---- verification against the files (product-only: bf16 passthrough == file bytes) -------------------
    verified = None
    if spec["kind"] == "llama":
        verified = True
        picks = [ref.tensors[0], ref.tensors[1], ref.tensors[len(ref.tensors) // 2], ref.tensors[-1]]
        picks += [t for t in ref.tensors if t["name"].endswith(("o_proj.weight", "down_proj.weight"))][-2:]
        for r in picks:
            pl = m.placements(r["name"])[0]
            if pl.slice_dim == 1:  # column slice: compare the last 64 rows run by run
                R = r["shape"][0]
                row_bytes, w = r["nbytes"] // R, pl.nbytes // R
                es = row_bytes // r["shape"][1]
                mm = np.memmap(ref.shards[r["shard"]], np.uint8, "r", offset=r["file_offset"], shape=(R, row_bytes))
                want = np.ascontiguousarray(mm[R - 64:, pl.slice_begin * es: pl.slice_begin * es + w]).reshape(-1)
                got = m.read(local, pl.pool_offset + (R - 64) * w, 64 * w)
                verified = verified and bool(np.array_equal(want, got))
                del mm
                continue
            row_bytes = r["nbytes"] // r["shape"][0] if r["shape"] else r["nbytes"]
            base = r["file_offset"] + (pl.slice_begin * row_bytes if pl.slice_dim == 0 else 0)
            n = min(pl.nbytes, 8 << 20)
            raw = np.fromfile(ref.shards[r["shard"]], np.uint8, count=n, offset=base + pl.nbytes - n)
            got = m.read(local, pl.pool_offset + pl.nbytes - n, n)
            verified = verified and bool(np.array_equal(raw, got))
        if not verified:
            raise SystemExit("pool contents differ from the checkpoint files")

    info = m.info()
    pool_bytes = info["pool_bytes"]
    part = st0["parts"][0]
    local_src = part["src_bytes"]

    # ---- e2e: public API with host buffers (pread -> pinned -> H2D -> kernels -> export + D2H result) ---------
    first = m.placements(ref.tensors[0]["name"])[0]

    step_detail = []

    def e2e_step():
        barrier()
        t = time.perf_counter()
        m.load_part()
        t_lp = time.perf_counter() - t
        if two_stage:
            barrier()
            m.convert_local()
        t_e0 = time.perf_counter()
        m.export(local)
        t_e1 = time.perf_counter()
        m.checksum(local, first.pool_offset, min(first.nbytes, 1 << 20))  # 8-byte D2H result read
        dt = time.perf_counter() - t
        if True:  # where this step's time went (recorded outside the timed region)
            st = m.stats()
            rd = st.get("readers") or {}
            n = max(rd.get("threads", 1), 1)
            step_detail.append({"ms": dt * 1e3, "load_part_ms": t_lp * 1e3, "export_ms": (t_e1 - t_e0) * 1e3, "checksum_ms": (time.perf_counter() - t_e1) * 1e3, "load_s": st.get("load_s"), "files_open_s": rd.get("files_open_s"), "files_close_s": rd.get("files_close_s"),
                                "reader_avg": {k: rd.get(k, 0) / n for k in ("slot_wait_s", "pread_s", "issue_s", "drain_s")}})
        barrier()
        return dt

    if args.kernel_only:
        e2e_ts = [float("nan")]
    else:
        # The harness's own garbage collector stays out of the timed steps: a generation-2 pass over a torch-sized heap is 50-150 ms, a third of a
        # step (it showed as one step in six taking 0.46 s while kk_load_part took its usual 0.30 s, profiles/r02/e2e_read_modes_q.jsonl); a Go or
        # C++ caller of the C ABI has no such pause.
        gc.collect()
        gc.freeze()
        gc.disable()
        try:
            for _ in range(args.warmup):
                e2e_step()
            e2e_ts = [allmax(e2e_step()) for _ in range(args.steps)]
        finally:
            gc.enable()
            gc.unfreeze()
    e2e_time = sum(e2e_ts)
    delivered = (pool_bytes if mode == gpupool.MODE_SCATTER else file_bytes) * (1 if mode == gpupool.MODE_SCATTER else world)
    if mode == gpupool.MODE_SCATTER:
        delivered = allsum(float(part["out_bytes"]))
    e2e_val = delivered * args.steps / e2e_time / 1e9
    file_read = allsum(float(local_src))  # bytes all ranks read from the files per step (= the checkpoint once, whatever N)
    chunks_per_load = part["chunks"]

    # ---- value: kernel stage from the HBM-resident image ---------------------------------------------------
    if args.e2e_only:
        line = {"metric": METRIC, "e2e_only": True, "n_gpus": N, "e2e": {"value": e2e_val, "unit": UNIT, "ms_per_step": e2e_time / args.steps * 1e3},
                "time_to_agent_ready_s": t_ready, "h2d_probe_GBps": h2d_probe, "verified_vs_files": verified, "readers_last_step": m.stats().get("readers"),
                "read_mode": os.environ.get("KUKEON_GPULOAD_READ", "auto"), "e2e_ms_each": [t * 1e3 for t in e2e_ts], "steps_detail": step_detail[-args.steps:],
                "config": {"readers": args.readers, "slots": args.slots, "slot_mb": args.slot_mb, "zerocopy": args.zerocopy, "numa_pin": not args.no_numa_pin,
                           "chunks_per_load": chunks_per_load, "kk_open_s": t_open}}
        if args.dump_outputs and rank == 0:
            dump_outputs(args.dump_outputs, m.manifest(local)["tensors"], lambda off, n: m.read(local, off, n))
        m.release()
        pool.close()
        barrier()
        if rank == 0:
            emit(line)
            if not args.keep_data:
                shutil.rmtree(d, ignore_errors=True)
        if world > 1:
            dist.destroy_process_group()
        return
    if not args.kernel_only:
        m.stage_resident()
    barrier()
    for _ in range(max(args.warmup, 3)):
        barrier()
        m.convert_resident()
        if two_stage:
            barrier()
            m.convert_local()
    clocks = ClockSampler(local)
    clocks.start()
    time.sleep(0.25)
    torch.cuda.synchronize()
    barrier()
    tc0 = time.time()
    step_ms, launch_ms = [], []
    wall0 = time.perf_counter()
    raw_ms = []
    for _ in range(args.steps):
        barrier()
        tot, per = m.convert_resident()
        if two_stage:  # stage 1 was just timed; stage 2 after every rank's stage 1 has landed
            barrier()
            t2 = m.convert_local()
            raw_ms.append((tot, t2))
            tot, per = tot + t2, [tot, t2]
        step_ms.append(tot)
        launch_ms.append(per)
    torch.cuda.synchronize()
    barrier()
    wall = time.perf_counter() - wall0
    tc1 = time.time()
    ck = clocks.stop(tc0, tc1)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, m.manifest(local)["tensors"], lambda off, n: m.read(local, off, n))
    dev_ms = allmax(sum(step_ms))
    value = delivered * args.steps / (dev_ms / 1e3) / 1e9
    n_launch = len(launch_ms[0])

    # ---- roofline of the dominant kernel (this rank's launches) -------------------------------------------
    peaks = {}
    pk = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(pk):
        peaks = json.load(open(pk))
    peak, peak_src = (peaks["hbm_gbs"], "measured (MEASURED_PEAKS.json hbm_gbs, copy read+write)") if "hbm_gbs" in peaks else (6650.0, "fallback (B200_PROFILING.md)")
    avg_launch_ms = sum(sum(p) for p in launch_ms) / (len(launch_ms) * max(n_launch, 1))
    # algorithmic HBM bytes of this rank per launch: source read once + pool writes landing in THIS GPU's HBM
    alg_per_step = local_src + part["out_bytes"] * (1 if mode == gpupool.MODE_SCATTER else world) if mode != gpupool.MODE_SINGLE else local_src + part["out_bytes"]
    if raw_order:  # stage 1: read own part + incoming peers' parts written; stage 2: read the whole image + write the whole pool
        alg_per_step = local_src + (file_bytes - local_src) + file_bytes + pool_bytes
    if pull_order:  # stage 1: read own part, write it twice (pool + slice buffer); stage 2: the other ranks' slices written into the pool
        alg_per_step = local_src + 2 * part["out_bytes"] + (pool_bytes - part["out_bytes"])
    alg_per_launch = alg_per_step / max(n_launch, 1)
    achieved = alg_per_launch / (avg_launch_ms / 1e3) / 1e9 if avg_launch_ms > 0 else 0.0
    # DRAM traffic of the dominant kernel from the committed `ncu --set full` capture of THIS kernel build (profiles/traffic.json names the capture and
    # the build it was taken from): dram__bytes_read.sum + dram__bytes_write.sum of one launch as a ratio to that launch's algorithmic bytes, scaled to
    # this run's launch.  Never measured inside a timed run (nothing here runs under a profiler).
    traffic = traffic_src = None
    tf = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tf) and world == 1:
        try:
            key = args.workload if (args.workload != "mixtral-q4k" or args.qtype == "Q4_K") else None  # the capture is of the Q4_K kernel only
            ent = json.load(open(tf)).get(key, {}) if key else {}
            if ent.get("ratio"):
                traffic, traffic_src = ent["ratio"] * alg_per_launch, ent.get("source")
        except Exception:  # noqa: BLE001
            traffic = None
    # HBM-write roofline (SURVEY.md §8(d)): bytes WRITTEN per launch against what a store-only kernel sustains on this box, measured now.
    # A probe failure must never fail the bench: the keys are null then.
    write_peak = copy_probe = None
    if world == 1 and not args.kernel_only:
        try:
            write_peak = max(pool.probe_hbm(local, gpupool.PROBE_WRITE, 4 << 30) for _ in range(3))
            copy_probe = max(pool.probe_hbm(local, gpupool.PROBE_COPY, 2 << 30) for _ in range(3))
        except Exception as e:  # noqa: BLE001
            print(f"[bench] HBM probe failed: {e}", file=sys.stderr)
    hbm_roofline = {"bound": "hbm", "kernel": "kk_convert_kernel", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                    "write_peak_GBps": write_peak, "ldst_copy_probe_GBps": copy_probe,
                    "hbm_write_frac": ((part["out_bytes"] / max(n_launch, 1)) / (avg_launch_ms / 1e3) / 1e9 / write_peak) if write_peak and avg_launch_ms > 0 else None,
                    "hbm_write_note": "a device-resident bf16 copy reads what it writes: half its traffic is reads, so its write fraction is capped near 0.5 and the "
                                      ">= 0.70 HBM-write target only applies to expanding conversions (see `secondary`)" if spec["kind"] == "llama" else None,
                    "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src, "algorithmic_bytes_per_launch": alg_per_launch, "avg_launch_ms": avg_launch_ms,
                    "launches_per_step": n_launch,
                    "write_only_frac_of_peak": (part["out_bytes"] / max(n_launch, 1)) / (avg_launch_ms / 1e3) / 1e9 / peak if avg_launch_ms > 0 else 0.0}
    roofline = hbm_roofline
    nvlink = None
    if world > 1 and mode == gpupool.MODE_BROADCAST:
        # peer-copy peak measured NOW: every rank reads from its ring neighbour's attached buffer at the same moment (copy engine, CUDA events)
        probes = []
        try:
            for _ in range(3):
                barrier()
                probes.append(m.probe_peer((rank + 1) % world, which, 1 << 30))
        except Exception as e:  # noqa: BLE001
            print(f"[bench] peer probe failed: {e}", file=sys.stderr)
        mine = max(probes) if probes else 0.0
        probe_mean = allsum(mine) / world
        probe_min = -allmax(-mine)
        step = sum(step_ms) / len(step_ms)
        if pull_order:
            moved = pool_bytes - part["out_bytes"]  # ingress: every other rank's slice
            stage_ms = sum(b for _, b in raw_ms) / len(raw_ms)
            form = "all-gather by P2P bulk LOADS from the peers' slice buffers (stage 2; bytes are NVLink ingress per GPU)"
        elif raw_order:
            moved = local_src * (world - 1)
            stage_ms = sum(a for a, _ in raw_ms) / len(raw_ms)
            form = "all-gather of the file bytes by P2P bulk stores (stage 1; bytes are NVLink egress per GPU)"
        else:
            moved = part["out_bytes"] * (world - 1)
            stage_ms = step
            form = "sharded ingest + fused P2P all-gather stores (bytes are NVLink egress per GPU)"
        gbps = moved / (stage_ms / 1e3) / 1e9 if stage_ms > 0 else 0.0
        pk_meas = probe_mean if probe_mean > 0 else None
        nvlink = {"bytes_per_step_per_gpu": moved, "stage_ms": stage_ms, "achieved_GBps_per_gpu": gbps, "peak_measured": pk_meas, "peak_measured_min_over_ranks": probe_min or None,
                  "peak_measured_how": "cudaMemcpyAsync D2D of 1 GiB from the ring neighbour's attached buffer, all ranks at once, best of 3, mean over ranks",
                  "peak_nominal": 900.0, "frac_of_measured": gbps / pk_meas if pk_meas else None, "frac_of_nominal": gbps / 900.0, "form": form}
        roofline = {"bound": "nvlink", "kernel": "kk_convert_kernel", "achieved": gbps, "peak": pk_meas or 900.0, "unit": "GB/s",
                    "frac": gbps / (pk_meas or 900.0), "peak_source": "peer-copy probe measured in this run (see nvlink.peak_measured_how)" if pk_meas else "nominal 900 GB/s per direction (probe failed)",
                    "peak_nominal": 900.0, "frac_of_nominal": gbps / 900.0, "traffic": None, "bytes_per_step_per_gpu": moved, "stage_ms": stage_ms, "form": form,
                    "hbm_side": {k: hbm_roofline[k] for k in ("achieved", "peak", "frac", "algorithmic_bytes_per_launch", "avg_launch_ms", "launches_per_step")}}

    # ---- optional NCCL comparison collective ----------------------------------------------------------------
    nccl = None
    if args.nccl_compare and world > 1 and mode == gpupool.MODE_BROADCAST:
        nccl = nccl_compare(torch, dist, file_bytes, world, local, args)

    # ---- CPU baseline beside it (rank 0, N == 1) ------------------------------------------------------------
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        try:
            m.unstage_resident()
            ctx = cpu_port_setup(path, None if file_bytes <= (40 << 30) else 40 << 30)
            cpu_port_step(ctx)  # untimed: parallel first touch of the output buffer
            cpu_port_step(ctx)
            ts = [cpu_port_step(ctx) for _ in range(args.steps)]
            cpu = {"value": ctx[3] / statistics.median(ts) / 1e9, "unit": UNIT, "cores": os.cpu_count() or 1, "kind": "port",
                   "sample": (("the whole checkpoint" if ctx[3] == file_bytes else f"first {ctx[3] / 1e9:.2f} GB of the checkpoint") +
                              f" ({ctx[3] / 1e9:.2f} GB), median of {len(ts)} passes after 2 untimed ones, pread + convert into host memory, all OpenMP threads"),
                   "best": ctx[3] / min(ts) / 1e9, "worst": ctx[3] / max(ts) / 1e9}
        except Exception as e:  # noqa: BLE001
            cpu = {"value": None, "unit": UNIT, "cores": 0, "kind": "port", "sample": f"failed: {e}"}

    # ---- secondary record (N = 1, default workload): an EXPANDING conversion, where the HBM-write fraction means something ------------------
    secondary = secondary_g = None
    if rank == 0 and world == 1 and args.workload == "llama3-8b" and not args.layers and not args.no_secondary and not args.kernel_only:
        try:
            m.unstage_resident()
            secondary = secondary_q4k(args, pool, gpupool, modelhub, peak, write_peak)
        except Exception as e:  # noqa: BLE001
            secondary = {"error": str(e)}
        try:
            secondary_g = secondary_gpt2(args, pool, gpupool, modelhub, peak, write_peak)
        except Exception as e:  # noqa: BLE001
            secondary_g = {"error": str(e)}

    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": N, "steps": args.steps, "warmup": max(args.warmup, 3),
        "ms_per_step": dev_ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16" if spec["kind"] != "gpt2" else "f32->bf16",
        "data": "synthetic",
        "config": {"workload": spec["name"], "file_bytes": file_bytes, "tensors": len(ref.tensors), "shards": len(ref.shards),
                   "mode": {0: "single", 1: "broadcast (sharded ingest + fused P2P fan-out)",
                            2: "scatter" + (" (row-parallel tensors exchanged over NVLink: KK_LOAD_SCATTER_EXCHANGE)" if exchange else "")}[mode], "pool_bytes_per_gpu": pool_bytes,
                   "l2": "inputs (>= 2 GB per GPU) far larger than the 126 MB L2; no flush needed", "files": f"warm in {os.path.dirname(d) or d}: written, then read twice by the ranks before anything is timed" + (", pages interleaved over the host's NUMA nodes (set_mempolicy while writing)" if _INTERLEAVED else ""),
                   "staging": "zero-copy pinned reads" if args.zerocopy else "pinned ring + H2D copy engine", "read_mode": os.environ.get("KUKEON_GPULOAD_READ", "auto (tmpfs shards: mapping + streaming stores + per-range MADV_DONTNEED; other file systems: pread)"), "verified_vs_files": verified,
                   **({"transpose_tiles": "8 source rows x <= 4 KiB, thread = column, 16-byte stores"} if spec["kind"] == "gpt2" else {})},
        "clocks": ck,
        "e2e": {"value": e2e_val, "unit": UNIT, "h2d_bytes_per_step": int(allsum(float(local_src))), "d2h_bytes_per_step": 8 * world,
                "ms_per_step": e2e_time / args.steps * 1e3, "ms_each": [t * 1e3 for t in e2e_ts], "steps_detail_rank0": step_detail[-args.steps:], "python_gc": "collected and frozen before, disabled during the e2e steps",
                "file_GBps": file_read * args.steps / e2e_time / 1e9 if e2e_time == e2e_time else None,
                "what": "kk_load_part (page cache->pinned->H2D->kernels) + kk_export + checksum word D2H; `value` counts the bytes made resident in all N pools "
                        "(N x checkpoint for a broadcast), `file_GBps` the checkpoint bytes read from the files once per step"},
        "gpu_launches": n_launch * args.steps,
        "roofline": roofline,
        "cpu_baseline": cpu,
        "time_to_agent_ready_s": t_ready,
        "time_to_agent_ready_incl_kk_open_s": t_ready_incl_open,
        "time_to_agent_ready_breakdown_rank0": brk,
        "time_to_agent_ready_breakdown_max_over_ranks": brk_max,
        "wall_ms_per_step": wall / args.steps * 1e3,
        "setup": {"synth_s": t_gen, "page_cache_warm_s": t_warm, "kk_open_s": t_open, "index_s": st0["index_s"], "plan_s": st0["plan_s"], "alloc_s": st0["alloc_s"],
                  "first_load_s": st0["load_s"], "chunks_per_load": chunks_per_load, "h2d_probe_GBps": h2d_probe},
    }
    if pull_order:
        line["config"]["mode"] = "broadcast, PULL order: convert into own pool + slice buffer (stage 1), pull the peers' slices over NVLink (stage 2)"
        line["pull_stages_ms_rank0"] = {"convert_ms": sum(a for a, _ in raw_ms) / len(raw_ms), "pull_ms": sum(b for _, b in raw_ms) / len(raw_ms)}
    if raw_order:
        line["config"]["mode"] = "broadcast, RAW order: all-gather file bytes over NVLink (stage 1) + local convert (stage 2)"
        line["raw_stages_ms_rank0"] = {"fanout_ms": sum(a for a, _ in raw_ms) / len(raw_ms), "convert_ms": sum(b for _, b in raw_ms) / len(raw_ms)}
    if world > 1 and mode == gpupool.MODE_BROADCAST:
        line["scaling_note"] = ("value(N) / (N x value(1)) is not a parallel efficiency here: at N = 1 a step is a copy inside one GPU's HBM, at N > 1 it is a "
                                "broadcast whose floor is NVLink ingress, (N-1)/N x checkpoint bytes per GPU at the link rate — at most ~0.28 of N x value(1) "
                                "for N = 8.  The per-N figure is roofline.frac (bound nvlink); end to end it is e2e.file_GBps and time_to_agent_ready_s.")
    if secondary is not None:
        line["secondary"] = secondary
    if secondary_g is not None:
        line["secondary_gpt2"] = secondary_g
    if nvlink:
        line["nvlink"] = nvlink
    if nccl:
        line["nccl_compare"] = nccl
    try:  # the measurements are complete: a teardown error is reported, never allowed to swallow the line
        m.release()
        pool.close()
    except Exception as e:  # noqa: BLE001
        line["teardown_error"] = str(e)
    barrier()
    # ---- time-to-agent-ready in kukeond's real shape: ONE process owning all N GPUs (no CUDA IPC between ranks) ------
    if world > 1 and not args.no_single_process:
        if rank == 0:
            try:
                t0 = time.time()
                sp = gpupool.Pool(list(range(world)), n_staging_buffers=args.slots, staging_buffer_bytes=args.slot_mb << 20, n_reader_threads=args.readers)
                sp_open = time.time() - t0
                t0 = time.time()
                ref2 = modelhub.Pull(path)
                spf = (gpupool.LOAD_GPT2_CONV1D_T if spec["kind"] == "gpt2" else 0) | (gpupool.LOAD_SCATTER_EXCHANGE if exchange else 0)
                m2 = modelhub.Load(sp, ref2, mode=mode, fanout=gpupool.FANOUT_RAW if raw_order else gpupool.FANOUT_P2P, flags=spf)
                for dev in range(world):
                    m2.export(dev)
                sp_ready = time.time() - t0
                t0 = time.time()
                m2.release()
                m3 = modelhub.Load(sp, ref2, mode=mode, fanout=gpupool.FANOUT_RAW if raw_order else gpupool.FANOUT_P2P, flags=spf)
                for dev in range(world):
                    m3.export(dev)
                sp_ready2 = time.time() - t0
                st2 = m3.stats()
                m3.release()
                if args.nvls_compare and mode == gpupool.MODE_BROADCAST:
                    cmpres = {}
                    for label, fo in (("p2p", gpupool.FANOUT_P2P), ("nvls", gpupool.FANOUT_NVLS)):
                        try:
                            mc = modelhub.Load(sp, ref2, mode=mode, fanout=fo, flags=spf | gpupool.LOAD_DEFER)
                            try:
                                mc.stage_resident()
                                for _ in range(max(args.warmup, 3)):
                                    mc.convert_resident()
                                ts = [mc.convert_resident()[0] for _ in range(args.steps)]
                                sums = {mc.checksum(dev, 0, mc.info()["pool_bytes"] // 8 * 8) for dev in range(world)}
                                cmpres[label] = {"ms_per_step": sum(ts) / len(ts), "ms_min": min(ts), "pools_identical": len(sums) == 1}
                            finally:
                                mc.release()
                        except Exception as e:  # noqa: BLE001
                            cmpres[label] = {"error": str(e)}
                    line["nvls_compare"] = cmpres
                sp.close()
                line["time_to_agent_ready_single_process_s"] = min(sp_ready, sp_ready2)
                line["time_to_agent_ready_single_process_incl_kk_open_s"] = sp_open + sp_ready  # a daemon that opens the pool only when the first model arrives
                line["single_process"] = {"what": "one process, one kk_ctx over all N GPUs (kukeond's shape): Pull + kk_load(mode) + kk_export x N; pinned ring and peer access are "
                                                  "set up in kk_open, once per daemon lifetime — reported both without it (a running daemon) and with it (cold daemon, first model)",
                                          "kk_open_s": sp_open, "first_s": sp_ready, "second_s": sp_ready2, "load_s": st2["load_s"], "alloc_s": st2["alloc_s"]}
            except Exception as e:  # noqa: BLE001
                line["single_process"] = {"error": str(e)}
        barrier()
    if rank == 0:
        emit(line)
        if not args.keep_data:
            shutil.rmtree(d, ignore_errors=True)
    if world > 1:
        dist.destroy_process_group()


def args_for_secondary(args, workload="mixtral-q4k", layers=4):
    import copy
    a = copy.copy(args)
    a.workload, a.qtype, a.layers = workload, "Q4_K", layers
    return a


def secondary_kernel_stage(args, pool, gpupool, modelhub, peak, write_peak, workload, layers, load_flags, what):
    """Kernel stage of a second BASELINE workload from the HBM-resident image, same timing rules as `value`: >= 3 warm-ups, CUDA events on the
    launching stream inside the library, inputs larger than L2."""
    from tools import synth
    t0 = time.time()
    a2 = args_for_secondary(args, workload, layers)
    spec = workload_spec(a2)
    base = os.path.dirname(pick_data_dir(args, synth.total_bytes(spec["tensors"])))
    d = os.path.join(base, f"kk_bench_secondary_{workload}_{layers}")
    path = make_files(spec, d, a2)
    synth_s = time.time() - t0
    try:
        ref = modelhub.Pull(path)
        m = modelhub.Load(pool, ref, mode=gpupool.MODE_SINGLE, fanout=gpupool.FANOUT_P2P, flags=gpupool.LOAD_DEFER | load_flags)
        try:
            m.stage_resident()
            for _ in range(3):
                m.convert_resident()
            steps = args.steps
            runs = [m.convert_resident() for _ in range(steps)]
            part = m.stats()["parts"][0]
        finally:
            m.release()
    finally:
        if not args.keep_data:
            shutil.rmtree(d, ignore_errors=True)
    ms = sum(t for t, _ in runs) / steps
    n_launch = len(runs[0][1])
    alg = part["src_bytes"] + part["out_bytes"]
    ach = alg / (ms / 1e3) / 1e9
    wr = part["out_bytes"] / (ms / 1e3) / 1e9
    return {"workload": spec["name"], "what": what, "steps": steps, "warmup": 3,
            "ms_per_step": ms, "launches_per_step": n_launch, "src_bytes": part["src_bytes"], "out_bytes": part["out_bytes"], "synth_s": synth_s,
            "value": part["out_bytes"] / (ms / 1e3) / 1e9, "unit": "GB/s of pool bytes made resident",
            "roofline": {"bound": "hbm", "kernel": "kk_convert_kernel", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                         "algorithmic_bytes_per_step": alg, "write_GBps": wr, "write_peak_GBps": write_peak,
                         "hbm_write_frac": wr / write_peak if write_peak else None}}


def secondary_q4k(args, pool, gpupool, modelhub, peak, write_peak):
    """4-layer Mixtral-8x7B q4_K GGUF (3.4 GB of blocks -> 12.1 GB of bf16): the expanding conversion of BASELINE config 4 at reduced depth."""
    return secondary_kernel_stage(args, pool, gpupool, modelhub, peak, write_peak, "mixtral-q4k", 4, 0,
                                  "kernel stage only (resident image), the expanding conversion of BASELINE config 4 at reduced depth")


def secondary_gpt2(args, pool, gpupool, modelhub, peak, write_peak):
    """GPT-2-small f32 -> bf16 with the Conv1D weights transposed (BASELINE config 1's checkpoint, 0.5 GB; small: ~105 tiles per SM, so launch
    ramp-up and tail are a visible part of its 0.15 ms)."""
    return secondary_kernel_stage(args, pool, gpupool, modelhub, peak, write_peak, "gpt2", 0, gpupool.LOAD_GPT2_CONV1D_T,
                                  "kernel stage only (resident image): BASELINE config 1's checkpoint, f32 -> bf16 casts + Conv1D transposes")


def nccl_compare(torch, dist, file_bytes, world, local, args):
    """Comparison collective only (north_star): all-gather of equal 1/N slices with NCCL, timed with CUDA events."""
    per = (file_bytes // world + 255) // 256 * 256
    src = torch.empty(per, dtype=torch.uint8, device=f"cuda:{local}")
    dst = torch.empty(per * world, dtype=torch.uint8, device=f"cuda:{local}")
    for _ in range(3):
        dist.all_gather_into_tensor(dst, src)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    dist.barrier()
    e0.record()
    for _ in range(args.steps):
        dist.all_gather_into_tensor(dst, src)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / args.steps
    t = torch.tensor([ms], dtype=torch.float64, device=f"cuda:{local}")
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item())
    return {"collective": "ncclAllGather", "ms": ms, "GBps_delivered_total": per * world * world / (ms / 1e3) / 1e9,
            "egress_GBps_per_gpu": per * (world - 1) / (ms / 1e3) / 1e9}


if __name__ == "__main__":
    main()
