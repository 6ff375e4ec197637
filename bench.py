#!/usr/bin/env python
"""bench.py -- compress+decompress throughput of the blocked shuffle->LZ hot path on B200.

Headline (`value`, `e2e`, `roofline`): BASELINE.json configs[1] -- LZ4 + byte-shuffle, clevel 5,
typesize 4, one 256 MiB bench.c-shaped buffer per GPU (bench/bench.c:141-170).  A step = one
blosc_compress_ctx + one blosc_decompress_ctx of that buffer.  `value` = (bytes compressed + bytes
decompressed) / time with the buffers resident in HBM; `e2e` = the same through the C ABI with
pinned HOST buffers (H2D/D2H inside the timed region).  N>1: one process per GPU, each rank owns
its own chunk (chunks are independent: no data-path collective, weak scaling), max over ranks.

The same JSON line also carries
  cfg3  BASELINE.json configs[2]: BloscLZ + bitshuffle, typesize 8 (N=1 only);
  cfg5  BASELINE.json configs[4]: 8 GiB = 32 chunks of 256 MiB sharded over the N GPUs
        (c-blosc_b200/sharding.py), typesize sweep {1,2,4,8,16}, without and with the NCCL
        scatter / gather-v legs from rank 0 (pipelined chunk by chunk);
  fast_parse  the opt-in segment-parallel parse on the headline workload (when built);
  cpu_baseline  the unmodified reference (oracle/_ref) on this box's host cores at its best
        thread count / API / placement (scripts/cpu_ref.py), N=1 only.
`--impl reference` prints the reference arm: the same sweep, best configuration as `value`.
`--workload NAME` restricts the run to one of the parts (faster iteration).
`--dump-outputs DIR` writes what the timed calls returned in their last step (compressed bytes, decoded
bytes, sizes) as DIR/<workload>.<name>.npy in float32 -- a fixed, seeded sample of each large buffer -- so that
two builds can be compared output for output on identical inputs.

Prints ONE JSON line on rank 0.
"""
from __future__ import annotations

import argparse
import csv
import io
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))

WORKLOADS = {
    # name: (compressor, doshuffle, typesize, clevel, nbytes)
    "lz4-shuffle-ts4-cl5-256MiB": ("lz4", 1, 4, 5, 256 << 20),
    "blosclz-bitshuffle-ts8-cl5-256MiB": ("blosclz", 2, 8, 5, 256 << 20),
}
CFG2, CFG3 = "lz4-shuffle-ts4-cl5-256MiB", "blosclz-bitshuffle-ts8-cl5-256MiB"
# BASELINE.json configs[4]: 8 GiB = 32 independent 256 MiB chunks sharded over the GPUs of one box
SHARDED = {
    # name: (compressor, doshuffle, clevel, total bytes, chunk bytes, typesizes, headline typesize)
    "lz4-shuffle-cl5-8GiB-sharded": ("lz4", 1, 5, 8 << 30, 256 << 20, (1, 2, 4, 8, 16), 4),
}
CFG5 = "lz4-shuffle-cl5-8GiB-sharded"
METRIC = "compress+decompress GB/s"
DUMP_SAMPLES = 1 << 20        # elements kept per dumped buffer: 4 MiB of float32 each, well under 64 MB per run
NVLINK_GBS = 770.0            # measured peer copy per direction per GPU (B200_PROFILING.md)


def bench_words(nbytes, np):
    i = np.arange(nbytes // 4, dtype=np.uint32)
    w = ((i << np.uint32(26)) ^ (i << np.uint32(18)) ^ (i << np.uint32(11)) ^ (i << np.uint32(3)) ^ i) & np.uint32((1 << 19) - 1)
    return w.view(np.uint8)


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured"
        except Exception:
            pass
    return 6650.0, "fallback"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING a timed region."""

    def __init__(self, index):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "20",
                                          "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
            t0 = time.time()
            while not self.rows and time.time() - t0 < 1.0:      # the first sample is there before the timed region starts
                time.sleep(0.01)
        except Exception:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"], "samples": 0}
        time.sleep(0.05)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 6:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for k, nme in enumerate(names):
                if f[2 + k].lower().startswith("active"):
                    reasons.add(nme)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def gpu_local_cpus(torch, index):
    """CPUs of the NUMA node the GPU hangs off (sysfs), or None.  Page-locked staging buffers are
    allocated while the process is confined to them, so that H2D / D2H DMA does not cross the
    socket interconnect -- what any host application that cares about PCIe throughput does."""
    try:
        p = torch.cuda.get_device_properties(index)
        bdf = "%04x:%02x:%02x.0" % (p.pci_domain_id, p.pci_bus_id, p.pci_device_id)
        node = int(open(f"/sys/bus/pci/devices/{bdf}/numa_node").read())
        if node < 0:
            return None
        cpus = set()
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            lo, _, hi = part.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
        cpus &= os.sched_getaffinity(0)
        return cpus or None
    except Exception:
        return None


class near_gpu:
    """with near_gpu(torch, index): ... -- run (and allocate) on the GPU's NUMA node."""

    def __init__(self, torch, index):
        self.cpus = gpu_local_cpus(torch, index)
        self.saved = None

    def __enter__(self):
        if self.cpus:
            self.saved = os.sched_getaffinity(0)
            os.sched_setaffinity(0, self.cpus)
        return self

    def __exit__(self, *a):
        if self.saved:
            os.sched_setaffinity(0, self.saved)


def dump_outputs(dump_dir, workload, arrays):
    """arrays: name -> uint8 tensor or int.  Buffers longer than DUMP_SAMPLES are sampled at sorted positions drawn
    from a fixed seed (the same positions for the same length), so that equal outputs give equal files.  Bytes are
    written as float32; sizes as float64, which holds them exactly (float32 would round sizes above 2^24)."""
    if not dump_dir or int(os.environ.get("RANK", "0")) != 0:
        return
    import numpy as np
    import torch
    os.makedirs(dump_dir, exist_ok=True)
    for name, t in arrays.items():
        path = os.path.join(dump_dir, f"{workload}.{name}.npy")
        if not torch.is_tensor(t):
            np.save(path, np.array([t], np.float64))
            continue
        if t.numel() > DUMP_SAMPLES:
            idx = np.sort(np.random.default_rng(0).integers(0, t.numel(), DUMP_SAMPLES))
            t = t.reshape(-1)[torch.from_numpy(idx).to(t.device)]
        np.save(path, t.reshape(-1).cpu().numpy().astype(np.float32))


# ------------------------------------------------------------------------------------------------
# reference CPU arm (scripts/cpu_ref.py does the work)
# ------------------------------------------------------------------------------------------------
def cpu_best(np, workload, budget_s):
    import cpu_ref
    r = cpu_ref.sweep(np, WORKLOADS[workload], budget_s=budget_s, reps=10)
    b = r["best"]
    table = [{k: (round(v, 3) if isinstance(v, float) else v) for k, v in row.items() if k in
              ("api", "threads", "placement", "value", "compress_gbs", "decompress_gbs", "reps", "final")} for row in r["sweep"]]
    nbytes = WORKLOADS[workload][4]
    return {"value": b["value"], "unit": "GB/s", "cores": b["threads"], "kind": r["kind"],
            "sample": f"{b['reps']} x (compress+decompress) of the full {nbytes >> 20} MiB buffer, median; best cell of the sweep",
            "compress_gbs": b["compress_gbs"], "decompress_gbs": b["decompress_gbs"], "api": b["api"],
            "placement": b.get("placement_note", b["placement"]), "cbytes": b["cbytes"],
            "cpu_model": r["cpu_model"], "physical_cores": r["physical_cores"], "hw_threads": r["hw_threads"],
            "numa_nodes": r["numa_nodes"], "sweep_seconds": round(r["seconds"], 1), "sweep": table,
            "api_note": "global = blosc_compress/blosc_decompress with a persistent pool (bench/bench.c:195,257,286); "
                        "ctx = blosc_*_ctx, which creates and joins its pool on every call (blosc.c:1302-1305)"}


def reference_arm(args, np):
    base = cpu_best(np, CFG2, 30.0)
    comp_name, shuf, ts, clevel, nbytes = WORKLOADS[CFG2]
    t_ms = 2 * nbytes / base["value"] / 1e6
    line = {"impl": "reference", "metric": METRIC, "value": base["value"], "unit": "GB/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": t_ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "u8", "data": "synthetic", "config": chunk_config(CFG2),
            "compress_gbs": base["compress_gbs"], "decompress_gbs": base["decompress_gbs"], "ratio": nbytes / base["cbytes"],
            "cpu_baseline": base,
            "e2e": {"value": base["value"], "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    if args.workload in ("all", CFG3):
        c3 = cpu_best(np, CFG3, 20.0)
        line["cfg3"] = {"workload": CFG3, "value": c3["value"], "unit": "GB/s", "compress_gbs": c3["compress_gbs"],
                        "decompress_gbs": c3["decompress_gbs"], "ratio": WORKLOADS[CFG3][4] / c3["cbytes"], "cpu_baseline": c3}
    if args.workload in ("all", CFG5):
        total, chunk = SHARDED[CFG5][3], SHARDED[CFG5][4]
        line["cfg5"] = {"workload": CFG5, "value": base["value"], "unit": "GB/s",
                        "note": f"the {total // chunk} chunks of the ts=4 row are {total // chunk} repetitions of the cfg 2 chunk "
                                "(per-chunk restart of the generator), compressed one after another by the whole pool: same GB/s"}
    print(json.dumps(line), flush=True)


def chunk_config(workload):
    comp_name, shuf, ts, clevel, nbytes = WORKLOADS[workload]
    return {"workload": workload, "codec": comp_name, "filter": ["none", "shuffle", "bitshuffle"][shuf], "typesize": ts,
            "clevel": clevel, "chunk_bytes": nbytes, "chunks_per_gpu": 1, "sharding": "one independent chunk per GPU",
            "l2": "input (256 MiB) larger than the 126 MB L2, no explicit flush"}


# ------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------
class Env:
    pass


def setup(world, local_rank):
    if world > 1:
        os.environ["CUDA_VISIBLE_DEVICES"] = os.environ.get("CUDA_VISIBLE_DEVICES", ",".join(str(i) for i in range(world))).split(",")[local_rank]
    import torch
    import __graft_entry__ as g
    e = Env()
    e.torch = torch
    e.pkg = g.load_package()
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback)"
    e.dev = torch.device("cuda", 0 if world > 1 else local_rank)
    torch.cuda.set_device(e.dev)
    e.world, e.dist = world, None
    e.smi_index = local_rank if world > 1 else torch.cuda.current_device()
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=e.dev)
        e.dist = dist
    return e


def barrier(e):
    e.torch.cuda.synchronize()
    if e.world > 1:
        e.dist.barrier()
    e.torch.cuda.synchronize()


def reduce_max(e, vals):
    if e.world == 1:
        return list(vals)
    t = e.torch.tensor(list(vals), device=e.dev, dtype=e.torch.float64)
    e.dist.all_reduce(t, op=e.dist.ReduceOp.MAX)
    return t.tolist()


def timed_steps(e, comp_args, dec_args, steps):
    """CUDA events around the whole region (the API calls are synchronous: each returns after its own
    stream has drained, so the events bracket all device work of the steps); max over ranks."""
    torch, pkg = e.torch, e.pkg
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier(e)
    e0.record()
    tc = td = 0.0
    cb = nb = 0
    for _ in range(steps):
        t0 = time.perf_counter()
        cb = pkg.compress_ctx(*comp_args)
        t1 = time.perf_counter()
        nb = pkg.decompress_ctx(*dec_args)
        t2 = time.perf_counter()
        tc += t1 - t0; td += t2 - t1
    e1.record()
    torch.cuda.synchronize()
    ms, tc, td = reduce_max(e, [e0.elapsed_time(e1), tc, td])
    barrier(e)
    return ms, tc, td, cb, nb


def bench_chunk(e, np, workload, steps, warmup, concurrent=False, env=None, dump_dir=None, dump_name=None):
    """One 256 MiB chunk per rank: device-resident value, host-pinned e2e, per-kernel times, clocks."""
    torch, pkg, dev, world = e.torch, e.pkg, e.dev, e.world
    comp_name, shuf, ts, clevel, nbytes = WORKLOADS[workload]
    saved_env = {}
    for k, v in (env or {}).items():
        saved_env[k] = os.environ.get(k); os.environ[k] = v
    try:
        numa = near_gpu(torch, dev.index)
        with numa:
            src_h = torch.from_numpy(bench_words(nbytes, np).copy()).pin_memory()
            chunk_h = torch.zeros(nbytes + 16, dtype=torch.uint8).pin_memory()
            out_h = torch.zeros(nbytes, dtype=torch.uint8).pin_memory()
        d_src = src_h.to(dev)
        d_chunk = torch.zeros(nbytes + 16, dtype=torch.uint8, device=dev)
        d_out = torch.zeros(nbytes, dtype=torch.uint8, device=dev)
        dev_args = ((clevel, shuf, ts, nbytes, d_src, d_chunk, nbytes + 16, comp_name), (d_chunk, d_out, nbytes))
        host_args = ((clevel, shuf, ts, nbytes, src_h, chunk_h, nbytes + 16, comp_name), (chunk_h, out_h, nbytes))
        for _ in range(max(3, warmup)):
            cb = pkg.compress_ctx(*dev_args[0]); nb = pkg.decompress_ctx(*dev_args[1])
            assert cb > 0 and nb == nbytes
        assert torch.equal(d_out, d_src), "round trip mismatch"
        pkg.compress_ctx(*host_args[0]); pkg.decompress_ctx(*host_args[1])
        assert torch.equal(out_h, src_h), "host round trip mismatch"

        # timed region 1: device-resident (`value`), kernel events on, clocks sampled
        sampler = ClockSampler(e.smi_index).start()
        pkg.set_profiling(True); pkg.prof_reset()
        launches0 = pkg.launch_count()
        ms, tc, td, cb, nb = timed_steps(e, dev_args[0], dev_args[1], steps)
        launches = pkg.launch_count() - launches0
        prof = pkg.prof_get(); pkg.set_profiling(False)
        assert cb > 0 and nb == nbytes
        dump_outputs(dump_dir, dump_name or workload, {"compressed": d_chunk[:cb], "decompressed": d_out, "cbytes": cb})
        # timed region 2: end to end from/to pinned host memory through the C ABI
        ms_h, tc_h, td_h, cb_h, nb_h = timed_steps(e, host_args[0], host_args[1], steps)
        clocks = sampler.stop()                  # sampled over both timed regions
        assert cb_h == cb and nb_h == nbytes and torch.equal(out_h, src_h)

        conc = None
        if concurrent and world == 1:
            # supplementary: 4 independent chunks in flight from 4 host threads (the _ctx API is re-entrant)
            K = 4
            bufs = [(d_src.clone(), torch.zeros_like(d_chunk), torch.zeros_like(d_out)) for _ in range(K)]

            def worker(i):
                s_, c_, o_ = bufs[i]
                pkg.compress_ctx(clevel, shuf, ts, nbytes, s_, c_, nbytes + 16, comp_name)
                pkg.decompress_ctx(c_, o_, nbytes)
            dt = None
            for rep in range(3):
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                th = [threading.Thread(target=worker, args=(i,)) for i in range(K)]
                [t.start() for t in th]
                [t.join() for t in th]
                torch.cuda.synchronize()
                dt = time.perf_counter() - t0
            assert all(torch.equal(b[2], d_src) for b in bufs)
            conc = {"chunks_in_flight": K, "value": K * 2 * nbytes / dt / 1e9, "unit": "GB/s",
                    "note": "4 x (compress+decompress) of 256 MiB issued concurrently from 4 host threads, device resident"}
            del bufs
    finally:
        for k, v in saved_env.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v

    hbm, hbm_src = peaks()
    per_step = ms / steps / 1e3
    kernels = {k: {"ms_avg": (v[0] / v[1] if v[1] else 0.0), "launches": v[1]} for k, v in prof.items() if v[1]}
    enc_ms, enc_n = prof["encode"]
    enc_name = "encode_kernel"
    if enc_n == 0 and prof.get("parse", (0, 0))[1]:          # fast parse: index_kernel + parse_kernel + fscan_kernel per compress
        enc_n = prof["parse"][1]
        enc_ms = prof["index"][0] + prof["parse"][0] + prof["scan"][0]
        enc_name = "index_kernel + parse_kernel + fscan_kernel"
    dec_ms, dec_n = prof["decode"]
    enc_avg = enc_ms / max(enc_n, 1) / 1e3
    dec_avg = dec_ms / max(dec_n, 1) / 1e3
    res = {"workload": workload, "value": world * 2 * nbytes / per_step / 1e9, "unit": "GB/s", "ms_per_step": per_step * 1e3,
           "compress_gbs": world * nbytes / (tc / steps) / 1e9, "decompress_gbs": world * nbytes / (td / steps) / 1e9,
           "ratio": nbytes / cb, "cbytes": cb,
           "e2e": {"value": world * 2 * nbytes / (ms_h / steps / 1e3) / 1e9, "unit": "GB/s", "h2d_bytes_per_step": nbytes + cb,
                   "d2h_bytes_per_step": cb + nbytes, "compress_gbs": world * nbytes / (tc_h / steps) / 1e9,
                   "decompress_gbs": world * nbytes / (td_h / steps) / 1e9,
                   "host_buffers": "page-locked, allocated on the GPU's NUMA node" if numa.cpus else "page-locked"},
           "gpu_launches": launches, "clocks": clocks,
           "roofline": {"bound": "hbm", "kernel": enc_name, "achieved": (nbytes + cb) / enc_avg / 1e9 if enc_avg > 0 else 0.0,
                        "peak": hbm, "unit": "GB/s", "frac": ((nbytes + cb) / enc_avg / 1e9 / hbm) if enc_avg > 0 else 0.0,
                        "traffic": None, "peak_source": hbm_src, "algorithmic_bytes_per_launch": nbytes + cb,
                        "avg_launch_ms": enc_avg * 1e3,
                        "decode_kernel": {"achieved": (nbytes + cb) / dec_avg / 1e9 if dec_avg > 0 else 0.0,
                                          "frac": ((nbytes + cb) / dec_avg / 1e9 / hbm) if dec_avg > 0 else 0.0,
                                          "avg_launch_ms": dec_avg * 1e3},
                        "whole_step": {"achieved": 2 * (nbytes + cb) / per_step / 1e9, "frac": 2 * (nbytes + cb) / per_step / 1e9 / hbm,
                                       "note": "algorithmic bytes of compress + decompress (2 x (U + C)) / step time, per GPU"}},
           "kernels": kernels}
    for kname in ("filter", "unfilter"):
        if kname in kernels and kernels[kname]["ms_avg"] > 0:
            res["roofline"][kname + "_kernel"] = {"achieved": 2 * nbytes / (kernels[kname]["ms_avg"] / 1e3) / 1e9,
                                                  "frac": 2 * nbytes / (kernels[kname]["ms_avg"] / 1e3) / 1e9 / hbm}
    if conc:
        res["concurrent"] = conc
    return res


def measure_traffic(workload):
    """dram__bytes_read.sum + dram__bytes_write.sum of ONE encode_kernel and ONE decode_kernel launch of this
    workload: a separate short `ncu` run of scripts/kbench.py (counters only -- nothing timed under the profiler)."""
    comp_name, shuf, ts, clevel, nbytes = WORKLOADS[workload]
    cmd = ["ncu", "--metrics", "dram__bytes_read.sum,dram__bytes_write.sum", "--clock-control", "none", "-k",
           "regex:encode_kernel|encode_team_kernel|decode_kernel|decode_pair_kernel", "-s", "6", "-c", "2", "--csv", sys.executable,
           os.path.join(ROOT, "scripts", "kbench.py"), "ncu", f"{comp_name}:{shuf}:{ts}"]
    try:
        env = dict(os.environ, KBENCH_STEPS="1")
        out = subprocess.run(cmd, capture_output=True, text=True, timeout=240, env=env).stdout
        start = out.find('"ID"')
        if start < 0:
            return None
        rows = list(csv.DictReader(io.StringIO(out[start:])))
        acc = {}
        for r in rows:
            kname = "encode" if "encode" in r.get("Kernel Name", "") else "decode"
            v = float(r["Metric Value"].replace(",", ""))
            u = r.get("Metric Unit", "byte").lower()
            v *= {"byte": 1, "kbyte": 1e3, "mbyte": 1e6, "gbyte": 1e9}.get(u, 1)
            acc[kname] = acc.get(kname, 0) + v
        return {k: int(v) for k, v in acc.items()} or None
    except Exception:
        return None


def bench_sharded(e, np, name, steps, warmup, dump_dir=None):
    """8 GiB as 32 chunks of 256 MiB, 32/N per GPU.  Leg 1: every rank's run is resident on its GPU and is
    compressed as one frame (blosc_b200_frame_*: 4 chunks in flight per GPU), no collective.  Leg 2 (N>1): rank 0's
    GPU holds the whole buffer, scatters it chunk by chunk over NCCL while the ranks compress, gathers the frames,
    sends them back and gathers the decoded slices (c-blosc_b200/sharding.py, pipelined variants)."""
    torch, pkg, dev, world, dist = e.torch, e.pkg, e.dev, e.world, e.dist
    from cblosc_b200 import sharding
    comp_name, shuf, clevel, total, chunk, sweep, head_ts = SHARDED[name]
    nchunks = total // chunk
    assert nchunks % world == 0, "32 chunks must divide over the ranks"
    k = nchunks // world
    mine = k * chunk
    rank = int(os.environ.get("RANK", "0"))
    one_h = torch.from_numpy(bench_words(chunk, np).copy())
    d_src = one_h.to(dev).repeat(k)
    bound = pkg.frame_bound(mine, 1, chunk)
    d_frame = torch.empty(bound, dtype=torch.uint8, device=dev)
    d_out = torch.empty(mine, dtype=torch.uint8, device=dev)

    def timed(ts, nsteps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier(e)
        e0.record()
        tc = td = 0.0
        fb = 0
        for _ in range(nsteps):
            t0 = time.perf_counter()
            fb = pkg.frame_compress(clevel, shuf, ts, mine, d_src, d_frame, bound, comp_name, 0, chunk)
            t1 = time.perf_counter()
            nb = pkg.frame_decompress(d_frame, fb, d_out, mine)
            tc += t1 - t0; td += time.perf_counter() - t1
            assert fb > 0 and nb == mine
        e1.record()
        torch.cuda.synchronize()
        ms, tc, td = reduce_max(e, [e0.elapsed_time(e1), tc, td])
        barrier(e)
        return ms, tc, td, fb

    sweep_out, head, clocks, prof, launches = {}, None, None, None, 0
    nst = steps
    for ts in sweep:
        timed(ts, 1)
        assert torch.equal(d_out, d_src), f"round trip mismatch at typesize {ts}"
        if ts == head_ts:
            timed(ts, 2)
            sampler = ClockSampler(e.smi_index).start()
            pkg.set_profiling(True); pkg.prof_reset(); launches0 = pkg.launch_count()
        ms, tc, td, fb = timed(ts, nst)
        if ts == head_ts:
            clocks = sampler.stop(); launches = pkg.launch_count() - launches0; prof = pkg.prof_get(); pkg.set_profiling(False)
            head = (ms, tc, td, fb)
        cb_chunk = (fb - 32 - 8 * k) // k
        sweep_out[str(ts)] = {"value": 2 * total / (ms / nst / 1e3) / 1e9, "compress_gbs": total / (tc / nst) / 1e9,
                              "decompress_gbs": total / (td / nst) / 1e9, "ratio": chunk / cb_chunk, "cbytes_per_chunk": cb_chunk}
    dump_outputs(dump_dir, name, {f"frame_ts{sweep[-1]}": d_frame[:fb], f"decompressed_ts{sweep[-1]}": d_out, "frame_bytes": fb})
    del d_frame, d_out

    sg = None
    if world > 1:
        full = one_h.to(dev).repeat(nchunks) if rank == 0 else None
        del d_src
        kw = dict(clevel=clevel, doshuffle=shuf, typesize=head_ts, compressor=comp_name)
        sampler = ClockSampler(e.smi_index).start()
        best = None
        for rep in range(3):                                   # rep 0 warms NCCL's P2P channels
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            barrier(e); e0.record()
            t0 = time.perf_counter()
            frames, sizes = sharding.compress_sharded_pipelined(pkg, dist, full, total, chunk, rank, world, dev, **kw)
            t1 = time.perf_counter()
            back = sharding.decompress_sharded_pipelined(pkg, dist, frames, sizes, total, chunk, rank, world, dev)
            t2 = time.perf_counter()
            e1.record(); torch.cuda.synchronize()
            ms_sg, tcs, tds = reduce_max(e, [e0.elapsed_time(e1), t1 - t0, t2 - t1])
            barrier(e)
            if rep and (best is None or ms_sg < best[0]):
                best = (ms_sg, tcs, tds)
        sg_clocks = sampler.stop()
        if rank == 0:
            assert torch.equal(back, full)
            moved = total - mine                                # bytes that leave rank 0 (and come back decoded)
            cfr = sum(sizes) - sizes[0]
            bound_ms = 2 * (moved + cfr) / NVLINK_GBS / 1e6     # out + back, each direction once, at the measured link rate
            sg = {"value": 2 * total / (best[0] / 1e3) / 1e9, "unit": "GB/s", "ms": best[0], "compress_ms": best[1] * 1e3,
                  "decompress_ms": best[2] * 1e3, "clocks": sg_clocks,
                  "nvlink": {"bytes_out_of_root": moved + cfr, "bytes_into_root": cfr + moved, "link_gbs": NVLINK_GBS,
                             "bound_ms": bound_ms, "frac_of_bound": bound_ms / best[0],
                             "note": "lower bound = the bytes that must cross rank 0's NVLink ports in each phase / 770 GB/s "
                                     "(scatter of the input + return of the frames, then frames out + decoded slices back)"},
                  "note": "rank 0 scatters 8 GiB chunk by chunk over NCCL/NVLink while the ranks compress, gathers the frames, "
                          "sends them back and gathers the decoded slices as they finish (best of 2 after a warm-up pass)"}
        del full, back, frames
    if rank != 0:
        return None
    hbm, hbm_src = peaks()
    ms, tc, td, fb = head
    per_step = ms / nst / 1e3
    cb_chunk = (fb - 32 - 8 * k) // k
    enc_ms, enc_n = prof["encode"]
    enc_avg = enc_ms / max(enc_n, 1) / 1e3
    agg = 2 * (total + nchunks * cb_chunk) / per_step / 1e9
    res = {"workload": name, "value": 2 * total / per_step / 1e9, "unit": "GB/s", "n_gpus": world, "scaling": "strong",
           "steps": nst, "ms_per_step": per_step * 1e3, "chunks_per_gpu": k, "typesize": head_ts,
           "compress_gbs": total / (tc / nst) / 1e9, "decompress_gbs": total / (td / nst) / 1e9,
           "ratio": chunk / cb_chunk, "cbytes": nchunks * cb_chunk, "typesize_sweep": sweep_out, "gpu_launches": launches, "clocks": clocks,
           "roofline": {"bound": "hbm", "kernel": "encode_kernel", "achieved": (chunk + cb_chunk) / enc_avg / 1e9 if enc_avg else 0.0,
                        "peak": hbm, "unit": "GB/s", "frac": ((chunk + cb_chunk) / enc_avg / 1e9 / hbm) if enc_avg else 0.0,
                        "peak_source": hbm_src, "avg_launch_ms": enc_avg * 1e3,
                        "note": "per launch, while up to 4 chunks per GPU are in flight",
                        "whole_step": {"achieved": agg / world, "frac": agg / world / hbm,
                                       "note": "algorithmic bytes of the whole step (both directions) / step time, per GPU"}},
           "kernels": {kk: {"ms_avg": (v[0] / v[1] if v[1] else 0.0), "launches": v[1]} for kk, v in prof.items() if v[1]},
           "sharding": "whole chunks per GPU (contiguous runs); per-chunk restart of the bench.c generator; inputs (>= 1 GiB per GPU) "
                       "larger than the 126 MB L2"}
    if sg:
        res["with_scatter_gather"] = sg
        res["scatter_gather_share"] = 1.0 - sg["value"] / res["value"] if res["value"] else None
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="all", choices=["all"] + sorted(WORKLOADS) + sorted(SHARDED))
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-traffic", action="store_true", help="skip the ncu DRAM-traffic subprocess")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's outputs to DIR/*.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    import numpy as np

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        if rank == 0:
            reference_arm(args, np)
        return

    e = setup(world, local_rank)
    want = lambda w: args.workload in ("all", w)
    head_wl = CFG3 if args.workload == CFG3 else CFG2
    dump = args.dump_outputs
    head = bench_chunk(e, np, head_wl, args.steps, args.warmup, concurrent=True, dump_dir=dump) if (want(CFG2) or want(CFG3)) else None
    cfg3 = bench_chunk(e, np, CFG3, args.steps, args.warmup, dump_dir=dump) if (args.workload == "all" and world == 1) else None
    fast = None
    if args.workload == "all" and getattr(e.pkg, "HAS_FAST_PARSE", False):
        fast = bench_chunk(e, np, CFG2, args.steps, args.warmup, env={"BLOSC_B200_PARSE": "fast"}, dump_dir=dump,
                           dump_name=CFG2 + "-fast-parse")
    cfg5 = bench_sharded(e, np, CFG5, args.steps, args.warmup, dump_dir=dump) if want(CFG5) else None
    if rank != 0:
        if world > 1:
            e.dist.destroy_process_group()
        return

    if head is None:                                            # --workload <sharded>: that workload is the line
        line = {"metric": METRIC, "value": cfg5["value"], "unit": "GB/s", "n_gpus": world, "steps": cfg5["steps"], "warmup": 1,
                "ms_per_step": cfg5["ms_per_step"], "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "u8",
                "data": "synthetic", "config": {"workload": CFG5}, "gpu_launches": cfg5["gpu_launches"], "clocks": cfg5["clocks"],
                "roofline": cfg5["roofline"], "e2e": None, "cfg5": cfg5}
        print(json.dumps(line), flush=True)
        if world > 1:
            e.dist.destroy_process_group()
        return

    config = chunk_config(head_wl)              # identical in both arms (the driver compares them); host placement is under e2e
    line = {"metric": METRIC, "value": head["value"], "unit": "GB/s", "n_gpus": world, "steps": args.steps, "warmup": max(3, args.warmup),
            "ms_per_step": head["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8",
            "data": "synthetic", "config": config, "compress_gbs": head["compress_gbs"], "decompress_gbs": head["decompress_gbs"],
            "ratio": head["ratio"], "cbytes": head["cbytes"], "e2e": head["e2e"], "gpu_launches": head["gpu_launches"],
            "clocks": head["clocks"], "roofline": head["roofline"], "kernels": head["kernels"]}
    if "concurrent" in head:
        line["concurrent"] = head["concurrent"]
    if world == 1 and not args.no_traffic:
        tr = measure_traffic(head_wl)
        if tr:
            line["roofline"]["traffic"] = tr.get("encode")
            line["roofline"]["decode_kernel"]["traffic"] = tr.get("decode")
            line["roofline"]["traffic_source"] = "ncu dram__bytes_read.sum + dram__bytes_write.sum, one launch, measured in this run (separate process)"
    if cfg3:
        cfg3["e2e"].pop("host_buffers", None)
        line["cfg3"] = cfg3
    if fast:
        fast["e2e"].pop("host_buffers", None)
        fast["note"] = ("BLOSC_B200_PARSE=fast (opt-in, NOT the default): hash-chain index + one thread per 256-byte segment "
                        "(csrc/dev_lz4fast.cuh); chunks are valid Blosc-1 / LZ4 that the reference decodes, but not byte-identical to its output")
        line["fast_parse"] = fast
    if cfg5:
        line["cfg5"] = cfg5
    if world == 1 and not args.no_cpu:
        line["cpu_baseline"] = cpu_best(np, head_wl, 25.0)
        if cfg3:
            line["cfg3"]["cpu_baseline"] = cpu_best(np, CFG3, 15.0)
        if cfg5:
            line["cfg5"]["cpu_baseline"] = {"value": line["cpu_baseline"]["value"], "unit": "GB/s", "cores": line["cpu_baseline"]["cores"],
                                            "kind": line["cpu_baseline"]["kind"],
                                            "sample": "the ts=4 chunks are repetitions of the cfg 2 chunk: the reference compresses them one "
                                                      "after another with its whole pool, i.e. at the cfg 2 rate above"}
    print(json.dumps(line), flush=True)
    if world > 1:
        e.dist.destroy_process_group()


if __name__ == "__main__":
    main()
