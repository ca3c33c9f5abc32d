#!/usr/bin/env python
"""bench.py -- vGPU worker hot-path benchmark (BASELINE.json metric, config[1]).

One "step" = one replay of the synthetic cudaMemcpy+launch stream of SURVEY.md 8d C2:
64 MALLOCs of 64 MiB, 256 x 64 MiB H2D copies (16 GiB of payload), one noop launch, one
SYNC.  Reported on ONE JSON line:

  value     payload GB/s with the trace resident in HBM when the timed region starts
            (tfw_trace_replay: only kernels are launched; inputs 16 GiB >> 126 MB L2)
  e2e       the same stream fed through the C-ABI (tfw_submit) from pinned HOST memory:
            deserialize + H2D DMA + unpack kernel + a D2H read of the result, all timed
  roofline  the byte-mover kernel: algorithmic bytes (2N per staged payload byte, N per
            filled byte) / CUDA-event time, against MEASURED_PEAKS.json hbm_gbs
  cpu_baseline  the oracle's sequential CPU replay of a bounded sample of the same stream
  overhead_vs_native  wall-clock of the worker path vs the identical calls issued straight
            to the CUDA runtime (bulk leg and 4 KiB latency leg)

`--impl reference` times the CPU side only (the reference worker is closed source, so this
is the oracle port of the path on the host cores; see DESIGN.md).
Multi-GPU (torchrun, --gpus N): the path does not shard -- one independent vGPU worker
per GPU ("replicas only", weak scaling), plus the peer-HBM swap leg of the tiering path.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "vgpu_replay_payload_GBps_into_HBM"
UNIT = "GB/s"
MIB = 1 << 20


def bind_to_gpu_numa(index):
    """Pin this process (and the threads it spawns) to the CPUs of the NUMA node its GPU hangs off, so that the
    pinned trace buffer is first-touched on that node: on a 2-socket HGX box half of the GPUs otherwise DMA their
    input across the socket interconnect (8-rank e2e 249 vs 425 GB/s).  Best effort; returns the node or None."""
    try:
        bus = subprocess.run(["nvidia-smi", f"--id={index}", "--query-gpu=pci.bus_id", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=10).stdout.strip().lower()
        if not bus:
            return None
        dom, rest = bus.split(":", 1)
        dev = f"{dom[-4:]}:{rest}"
        node = int(open(f"/sys/bus/pci/devices/{dev}/numa_node").read())
        if node < 0:
            return None
        cpus = set()
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            lo, _, hi = part.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
        os.sched_setaffinity(0, cpus & os.sched_getaffinity(0) or cpus)
        return node
    except Exception:
        return None


def peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            p = json.load(f)
        return float(p["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs, read+write copy)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def ncu_traffic():
    """dram__bytes_read+write of one mover launch from the committed ncu capture (profiles/), or None."""
    import glob
    files = sorted(glob.glob(os.path.join(ROOT, "profiles", "*_mover_traffic.json")))
    if not files:
        return None, None
    try:
        with open(files[-1]) as f:
            t = json.load(f)
        return int(t["dram_bytes"]), {"launch": f"copy batch, grid {t['grid']}", "algorithmic_bytes": t["algorithmic_bytes_if_copy"],
                                      "source": t["source"]}
    except Exception:
        return None, None


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons while the timed region runs."""

    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self.stop_flag = index, [], threading.Event()

    def run(self):
        while not self.stop_flag.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([x.strip() for x in out.split(",")])
            except Exception:
                pass
            self.stop_flag.wait(0.2)

    def summary(self):
        self.stop_flag.set()
        self.join(timeout=6)
        sm = sorted(float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit())
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows if len(r) >= 7 for i in range(4) if r[3 + i].lower().startswith("active")})
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(self.rows)}


def _numpy_bulk_stream(nbuf, ncopies, each):
    """The C2 bulk stream built with numpy + struct only (the reference arm maps no product library):
    nbuf MALLOCs, ncopies H2D frames of `each` bytes round-robin, one noop LAUNCH, one SYNC."""
    import struct
    import numpy as np
    hdr = struct.Struct("<IHHIIIIQQQIIII")

    def frame(op, call, h0=0, length=0, arg1=0, arg2=0):
        return hdr.pack(0x53434654, 1, op, call, 0, h0, 0, 0, 0, length, 0, arg1, arg2, 0)

    per = 64 + ((each + 15) & ~15)
    total = 64 * nbuf + per * ncopies + 128
    out = np.empty(total, dtype=np.uint8)
    pos = call = 0
    for h in range(1, nbuf + 1):
        out[pos:pos + 64] = np.frombuffer(frame(1, call, h, each), dtype=np.uint8)
        pos += 64
        call += 1
    payload = np.random.default_rng(7).integers(0, 256, each, dtype=np.uint8)
    for i in range(ncopies):
        out[pos:pos + 64] = np.frombuffer(frame(3, call, 1 + i % nbuf, each), dtype=np.uint8)
        np.copyto(out[pos + 64:pos + 64 + each], payload)       # (also the first touch of the stream's pages)
        out[pos + 64 + each:pos + per] = 0
        pos += per
        call += 1
    out[pos:pos + 64] = np.frombuffer(frame(7, call, 0, 0, 1, 32), dtype=np.uint8)
    out[pos + 64:pos + 128] = np.frombuffer(frame(8, call + 1), dtype=np.uint8)
    return out


def cpu_replay_baseline(stream, payload_bytes, threads, budget_s=20.0, max_passes=6):
    """The reference side of the path on the host cores: the oracle's CPU replay of the SAME stream (the reference
    worker itself is closed source, README.md:131).  The engine a CPU implementation meant to be fast would have:
    a persistent thread pool for copies and zero-fills, freed buffers kept for the next MALLOC (no first-touch page
    faults after the warm-up pass).  Returns GB/s of payload for `threads` threads and for one."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle

    def timed(nthreads, budget):
        oracle.lib.tfo_set_threads(nthreads)
        oracle.lib.tfo_set_buffer_cache(1)
        r = oracle.Replay(stream)      # warm-up: pool start, page faults of the destination buffers
        assert r.rc == 0
        r.close()
        t0, passes = time.perf_counter(), 0
        while True:
            r = oracle.Replay(stream)
            assert r.rc == 0
            r.close()
            passes += 1
            if time.perf_counter() - t0 > budget or passes >= max_passes:
                break
        dt = time.perf_counter() - t0
        oracle.lib.tfo_set_buffer_cache(0)
        oracle.lib.tfo_set_threads(1)
        return payload_bytes * passes / dt / 1e9, passes, dt

    # more threads are not more memcpy: try a few pool sizes briefly and keep the best (the reported `cores`)
    cands = sorted({t for t in (threads, 64, 32, 16, 8) if 1 < t <= threads}, reverse=True) or [1]
    probe = {t: timed(t, 2.0)[0] for t in cands} if len(cands) > 1 else {cands[0]: 0.0}
    best_t = max(probe, key=probe.get)
    multi, passes, dt = timed(best_t, budget_s)
    single, p1, dt1 = timed(1, min(budget_s, 8.0)) if threads > 1 else (multi, passes, dt)
    threads_available, threads = threads, best_t
    return {"value": round(multi, 3), "unit": UNIT, "cores": threads, "kind": "port", "single_thread_value": round(single, 3),
            "same_config": True, "host_cores_available": threads_available, "pool_sizes_tried_GBps": {str(k): round(v, 1) for k, v in probe.items()},
            "sample": f"{passes} x oracle replay of the whole stream ({payload_bytes / 2**30:.0f} GiB payload per pass, {dt:.1f} s; 1 thread: {p1} pass(es), "
                      f"{dt1:.1f} s) with a persistent thread pool and re-used (pre-faulted, zero-filled) destinations; "
                      "reference worker is closed source (README.md:131)"}


DUMP_CHUNKS, DUMP_CHUNK_BYTES, DUMP_SEED = 4, 16 << 10, 20240601


def save_output(d, name, arr):
    """One output array as DIR/<name>.npy, in float32 (bytes are 0..255: exact) or float64."""
    import numpy as np
    os.makedirs(d, exist_ok=True)
    arr = np.asarray(arr)
    np.save(os.path.join(d, name + ".npy"), arr.astype(np.float64 if arr.dtype.itemsize > 2 else np.float32))


def dump_replay_outputs(d, w, t, nbuf, resp, replays):
    """What the last replay of the resident trace left for its caller: the response stream of that replay, a
    digest of every buffer (tfw_dev_digest, as two 32-bit halves) and a fixed, seeded sample of their bytes
    (DUMP_CHUNKS x DUMP_CHUNK_BYTES per buffer: 64 x 64 KiB = 16 MB as float32 for the default 4 GiB)."""
    import numpy as np
    assert len(resp) % replays == 0, (len(resp), replays)
    per = len(resp) // replays
    save_output(d, "replay_responses", np.frombuffer(resp[len(resp) - per:], dtype=np.uint8))
    rng = np.random.default_rng(DUMP_SEED)
    digests, sample, offsets = [], [], []
    for h in range(1, nbuf + 1):
        size, ptr = t.buffer_info(h)
        dg = w.dev_digest(ptr, size)
        digests.append((dg >> 32, dg & 0xFFFFFFFF))
        n = min(DUMP_CHUNK_BYTES, size)
        offs = np.sort(rng.integers(0, size - n + 1, DUMP_CHUNKS))
        offsets.append(offs)
        sample.append(np.concatenate([w.dev_read(ptr + int(o), n) for o in offs]))
    save_output(d, "replay_buffer_digests", np.array(digests, dtype=np.uint64))
    save_output(d, "replay_buffer_sample_offsets", np.array(offsets, dtype=np.int64))
    save_output(d, "replay_buffer_sample", np.stack(sample))


def bench_config(args, world):
    """The `config` object of the JSON line -- the same for both arms (the reference arm runs `your arm's config`)."""
    payload = args.copies * args.payload_mib * MIB
    return {"workload": f"C2 bulk stream: 1 vGPU @100%, {args.buffers} MALLOC + {args.copies} x {args.payload_mib} MiB H2D "
                        f"({payload / 2**30:.0f} GiB payload) + noop launch + SYNC per step",
            "parallelism": "replicas only: one vGPU worker per GPU, each bound to its GPU's NUMA node" if world > 1 else "1 worker, 1 GPU",
            "staging_chunk_mib": args.chunk_mib or 32, "l2": "inputs (16 GiB) far larger than the 126 MB L2; no flush needed",
            "value_leg": "trace resident in HBM, tfw_trace_replay", "e2e_leg": "tfw_submit from pinned host memory"}


def run_reference(args):
    """--impl reference: CPU implementation of the path on the host cores, on the same config."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    threads = os.cpu_count() or 1
    steps, warm = max(1, args.steps), max(0, args.warmup)
    each = args.payload_mib * MIB
    stream = _numpy_bulk_stream(args.buffers, args.copies, each)
    payload = args.copies * each
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle
    oracle.lib.tfo_set_buffer_cache(1)
    # more threads are not more memcpy: one untimed pass per pool size (the first is the page-fault warm-up), keep the fastest
    available, probe = threads, {}
    for tcount in [t for t in (16, 32, 64, available) if t <= available] or [1]:
        oracle.lib.tfo_set_threads(tcount)
        for rep in range(2 if not probe else 1):
            t0 = time.perf_counter()
            r = oracle.Replay(stream)
            assert r.rc == 0
            r.close()
        probe[tcount] = payload / (time.perf_counter() - t0) / 1e9
    threads = max(probe, key=probe.get)
    oracle.lib.tfo_set_threads(threads)
    times = []
    budget_end = time.perf_counter() + 150.0
    for i in range(warm + steps):
        t0 = time.perf_counter()
        r = oracle.Replay(stream)
        assert r.rc == 0
        r.close()
        if i >= warm:
            times.append(time.perf_counter() - t0)
        if time.perf_counter() > budget_end and times:
            break
    oracle.lib.tfo_set_buffer_cache(0)
    oracle.lib.tfo_set_threads(1)
    ms = sum(times) / len(times) * 1e3
    v = payload / (ms * 1e-3) / 1e9
    line = {"impl": "reference", "metric": METRIC, "value": round(v, 3), "unit": UNIT, "n_gpus": args.gpus, "steps": len(times),
            "warmup": warm, "ms_per_step": round(ms, 2), "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "config": bench_config(args, max(1, args.gpus)),
            "cpu_baseline": {"value": round(v, 3), "unit": UNIT, "cores": threads, "kind": "port", "same_config": True,
                             "host_cores_available": available, "pool_sizes_tried_GBps": {str(k): round(x, 1) for k, x in probe.items()},
                             "engine": "oracle/replay_oracle.c: persistent thread pool, freed buffers re-used (pre-faulted), MALLOC zero-fills",
                             "sample": f"{len(times)} timed replays of the whole stream ({payload / 2**30:.0f} GiB payload each), {warm} warm-up"},
            "e2e": {"value": round(v, 3), "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--buffers", type=int, default=64)
    ap.add_argument("--copies", type=int, default=256)
    ap.add_argument("--payload-mib", type=int, default=64)
    ap.add_argument("--chunk-mib", type=int, default=0, help="staging slot size (0 = library default)")
    ap.add_argument("--latency-calls", type=int, default=20000)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-swap", action="store_true")
    ap.add_argument("--no-boundary", action="store_true", help="skip the legs through tensor-fusion-worker + libtfc_client")
    ap.add_argument("--no-c3", action="store_true", help="skip the 4 x 25 %% limiter leg")
    ap.add_argument("--no-c4", action="store_true", help="skip the 256 GiB-on-one-GPU policy sweep")
    ap.add_argument("--c5-gib", type=int, default=0, help="size of the C5 vGPU address space (0 = 1 TiB at 8 GPUs, scaled down with fewer)")
    ap.add_argument("--swap-regions", type=int, default=8, help="1 GiB regions evicted/prefetched per GPU in the swap leg")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the timed legs computed in their last step to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        return run_reference(args)
    args.warmup = max(3, args.warmup)

    import numpy as np
    import torch
    import torch.distributed as dist
    from tensor_fusion_b200 import _native as N
    from tensor_fusion_b200 import multi, trace, wire
    from tensor_fusion_b200.worker import PinnedBuffer, Worker

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    cpu_group = None
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
        cpu_group = dist.new_group(backend="gloo")   # host-side barrier: an NCCL barrier parks a spinning kernel on every waiting GPU
    torch.cuda.set_device(local)
    numa = bind_to_gpu_numa(local) if world > 1 else None

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    each = args.payload_mib * MIB
    payload_per_step = args.copies * each
    size = trace.bulk_size(args.buffers, args.copies, each)
    pin = PinnedBuffer(size + 4096)
    raw = trace.gen_bulk(args.buffers, args.copies, each, seed=trace.SEED_C1 + rank, nthreads=min(32, os.cpu_count() or 8), into=pin)

    w = Worker(device=local, chunk_bytes=args.chunk_mib * MIB)
    stream = torch.cuda.ExternalStream(N.lib.tfw_exec_stream(w.h), device=torch.device("cuda", local))

    # ---------------- leg 1: trace resident in HBM (value + roofline) ----------------
    t = w.load_trace(raw)
    info = t.info()
    sampler = ClockSampler(local)   # samples across warm-up, the resident leg and the e2e leg
    sampler.start()
    for _ in range(args.warmup):
        t.replay()
    w.flush()
    s0 = w.stats()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(args.steps):
        t.replay()
    e1.record(stream)
    e1.synchronize()
    barrier()
    dev_ms = e0.elapsed_time(e1)
    s1 = w.stats()
    replay_resp = w.poll()   # the responses of every replay since the trace was loaded, each the same length
    launches = sum(s1[k] - s0[k] for k in ("mover_launches", "client_launches", "gate_launches"))
    mover_launches = s1["mover_launches"] - s0["mover_launches"]
    if world > 1:
        tt = torch.tensor([dev_ms], device="cuda")
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        dev_ms_max = float(tt.item())
    else:
        dev_ms_max = dev_ms
    value = world * payload_per_step * args.steps / (dev_ms_max * 1e-3) / 1e9
    # roofline of the mover: the timed region is mover launches back to back (+1 noop launch per step)
    peak, peak_src = peaks()
    algo_per_launch = info["algorithmic_bytes"] / info["mover_launches"]
    avg_launch_ms = dev_ms / max(1, mover_launches)
    achieved = algo_per_launch / (avg_launch_ms * 1e-3) / 1e9
    traffic, traffic_note = ncu_traffic()
    if args.dump_outputs and rank == 0:
        dump_replay_outputs(args.dump_outputs, w, t, args.buffers, replay_resp, args.warmup + args.steps)
    t.free()

    # ---------------- leg 2: end to end from pinned host memory through the C-ABI ----------------
    e2e_steps = args.steps
    tail = bytes(wire.Builder().d2h(1, 0, 4096).sync())
    tail_arr = np.frombuffer(tail, dtype=np.uint8)
    free_all = wire.Builder()
    for h in range(1, args.buffers + 1):
        free_all.free(h)
    free_arr = np.frombuffer(bytes(free_all), dtype=np.uint8)

    def e2e_step():
        n = w.submit(raw)
        assert n == raw.nbytes
        w.submit(tail_arr)          # read 4 KiB of the result back + SYNC
        w.flush()
        resp = w.poll()
        w.submit(free_arr)          # end of session: the next step starts from an empty handle table
        return resp

    for _ in range(2):
        e2e_step()
    w.flush()
    s0 = w.stats()
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        resp = e2e_step()
    barrier()
    e2e_s = time.perf_counter() - t0
    s1 = w.stats()
    if world > 1:
        tt = torch.tensor([e2e_s], device="cuda")
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        e2e_s = float(tt.item())
    e2e_val = world * payload_per_step * e2e_steps / e2e_s / 1e9
    clocks = sampler.summary()
    if args.dump_outputs and rank == 0:
        save_output(args.dump_outputs, "e2e_responses", np.frombuffer(resp, dtype=np.uint8))
    h2d_per_step = (s1["h2d_dma_bytes"] - s0["h2d_dma_bytes"]) // e2e_steps
    d2h_per_step = (s1["d2h_bytes"] - s0["d2h_bytes"]) // e2e_steps
    assert len(resp) >= 4096 and d2h_per_step >= 4096

    # ---------------- native-CUDA comparator (rank 0, N = 1 only) ----------------
    overhead = None
    if rank == 0 and world == 1:
        nat_s, _, _ = trace.native_replay(raw, passes=3, device=local)
        bulk = {"worker_ms": round(e2e_s / e2e_steps * 1e3, 2), "native_ms": round(nat_s * 1e3, 2),
                "added_percent": round((e2e_s / e2e_steps / nat_s - 1) * 100, 2)}
        small = trace.gen_small(args.latency_calls, 4096)
        spin = PinnedBuffer(small.nbytes)
        spin.array[: small.nbytes] = small
        sview = spin.array[: small.nbytes]
        close1 = np.frombuffer(bytes(wire.Builder().free(1)), dtype=np.uint8)
        lat = []
        for _ in range(3):
            t0 = time.perf_counter()
            w.submit(sview)
            w.flush()
            lat.append(time.perf_counter() - t0)
            w.poll()
            w.submit(close1)
        nat_small, _, ncalls = trace.native_replay(sview, passes=3, device=local)
        wk = sorted(lat)[1]
        # the mixed 1k-call trace (C1): many small calls, 25 % unaligned, D2H / D2D / launches
        c1 = trace.gen_c1(error_permille=0)
        cpin = PinnedBuffer(c1.nbytes)
        cpin.array[: c1.nbytes] = c1
        cview = cpin.array[: c1.nbytes]
        handles = sorted({h["h0"] for h, _ in wire.parse_frames(c1) if h["opcode"] == wire.OP_MALLOC})
        fb = wire.Builder()
        for hnd in handles:
            fb.free(hnd)          # frees of already-freed handles only produce error frames
        cfree = np.frombuffer(bytes(fb), dtype=np.uint8)
        c1_t = []
        for _ in range(5):
            t0 = time.perf_counter()
            w.submit(cview)
            w.flush()
            c1_t.append(time.perf_counter() - t0)
            w.poll()
            w.submit(cfree)
            w.flush()
            w.poll()
        nat_c1, _, c1_calls = trace.native_replay(cview, passes=5, device=local)
        c1_w = sorted(c1_t)[len(c1_t) // 2]
        cpin.free()
        overhead = {"bulk_16GiB": bulk,
                    "c1_mixed_trace": {"calls": int(c1_calls), "worker_ms": round(c1_w * 1e3, 3), "native_ms": round(nat_c1 * 1e3, 3),
                                       "added_percent": round((c1_w / nat_c1 - 1) * 100, 2)},
                    "latency_4KiB": {"calls": int(ncalls), "worker_us_per_call": round(wk / ncalls * 1e6, 3),
                                     "native_us_per_call": round(nat_small / ncalls * 1e6, 3),
                                     "added_percent": round((wk / nat_small - 1) * 100, 2)}}
        spin.free()
        # the same stream through the REAL process boundary: libtfc_client.so in this process, tensor-fusion-worker in
        # another, over the page-locked shared rings and over TCP loopback, next to native CUDA (tools/boundary_bench.py)
        if not args.no_boundary:
            try:   # in a process of its own, under a timeout: a wedged transport must not take the bench line with it
                r = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "boundary_bench.py"), "--device", str(local), "--copies", str(args.copies),
                                    "--each-mib", str(args.payload_mib)], capture_output=True, text=True, timeout=900)
                if r.returncode != 0:
                    raise RuntimeError(r.stderr[-300:])
                b = json.loads(r.stdout.strip().splitlines()[-1])
                overhead["native_cuda"] = b["native"]
                overhead["through_worker_shm"] = b["through_worker_shm"]
                overhead["through_worker_loopback_upgraded"] = b.get("through_worker_loopback_upgraded")
                overhead["through_worker_tcp_loopback"] = b["through_worker_tcp_loopback"]
                overhead["boundary_workload"] = b["workload"]
            except Exception as e:   # the boundary legs must not take the headline down with them
                overhead["through_worker_shm"] = {"error": f"{type(e).__name__}: {e}"[:300]}

    # ---------------- VRAM-tier swap legs (north_star c) ----------------
    swap = None
    swap_all = None
    if not args.no_swap:
        from tensor_fusion_b200 import vram as V
        R, K = 1 << 30, args.swap_regions

        def pattern_digests(seeds, nbytes):
            """tfw_digest64 of the test pattern for each seed, computed by the CPU oracle (the checker)."""
            sys.path.insert(0, os.path.join(ROOT, "tests"))
            import oracle
            from concurrent.futures import ThreadPoolExecutor
            with ThreadPoolExecutor(max_workers=min(16, len(seeds))) as ex:   # ctypes releases the GIL: regions in parallel
                return list(ex.map(lambda sd: oracle.digest(oracle.pattern(sd, nbytes)), seeds))

        def swap_leg(home, peers, flags, everyone):
            """Evict K x 1 GiB regions from `home` (striped over `peers`, or to host DRAM) and bring them back."""
            tier = V.PEER if peers else V.HOST
            with V.VSpace(home=home, va_bytes=K * R, region_bytes=R, home_budget=K * R, peer_budget=K * R,
                          host_budget=0 if peers else K * R, peers=peers, flags=flags) as vs:
                for r in range(K):
                    vs.populate(r, V.HOME)
                    vs.fill_pattern(r, 1000 * rank + r)
                want = pattern_digests([1000 * rank + r for r in range(K)], R)   # CPU oracle: independent of every GPU kernel
                slots = multi.stripe_slots(K, len(peers), rank if everyone else 0)
                ev_ms, pf_ms, ev_wall, pf_wall = [], [], [], []
                for rep in range(3):
                    if everyone:
                        barrier()
                    ev = vs.migrate(list(range(K)), [tier] * K, slots)
                    if everyone:
                        barrier()
                    pf = vs.migrate(list(range(K)), [V.HOME] * K)
                    if rep:
                        ev_ms.append(ev["copy_ms"]); pf_ms.append(pf["copy_ms"]); ev_wall.append(ev["total_ms"]); pf_wall.append(pf["total_ms"])
                got = [vs.digest(r) for r in range(K)]
                assert got == want, f"region bytes changed across evict/prefetch: {[r for r in range(K) if got[r] != want[r]]}"
            return [min(ev_ms), min(pf_ms), min(ev_wall), min(pf_wall)]

        def c5_policy_sweep(ngpus, va_gib, extra=()):
            """C4 / C5 as a client sees it (tools/tier_sweep.py): ONE vGPU larger than its GPU, swept sequentially through the
            policy entry point.  In a process of its own under a timeout: the headline must survive whatever happens there."""
            try:
                r = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "tier_sweep.py"), "--gpus", str(ngpus), "--va-gib", str(va_gib),
                                    "--home-device", str(local if ngpus == 1 else 0), *extra], capture_output=True, text=True, timeout=1200)
                if r.returncode != 0:
                    return {"error": (r.stderr or r.stdout)[-400:]}
                return json.loads(r.stdout.strip().splitlines()[-1])
            except Exception as e:
                return {"error": f"{type(e).__name__}: {e}"[:300]}

        def summarize(vals, npeers, homes, what):
            nbytes = K * R
            d = {"what": what, "bytes_per_direction_per_home_gpu": nbytes, "region_mib": R >> 20,
                 "verified": f"all {K} regions against the CPU oracle's pattern digests after 3 evict/prefetch round trips",
                 "evict_GBps_per_home_gpu": round(nbytes / vals[0] / 1e6, 1), "prefetch_GBps_per_home_gpu": round(nbytes / vals[1] / 1e6, 1),
                 "evict_GBps_incl_remap": round(nbytes / vals[2] / 1e6, 1), "prefetch_GBps_incl_remap": round(nbytes / vals[3] / 1e6, 1),
                 "aggregate_evict_GBps": round(homes * nbytes / vals[0] / 1e6, 1)}
            if npeers:
                d["evict_frac_of_nvlink_nominal_900"] = round(nbytes / vals[0] / 1e6 / 900.0, 3)
                d["prefetch_frac_of_nvlink_nominal_900"] = round(nbytes / vals[1] / 1e6 / 900.0, 3)
                d["evict_frac_of_measured_peer_copy_770"] = round(nbytes / vals[0] / 1e6 / 770.0, 3)
            return d

        if world == 1:
            swap = summarize(swap_leg(local, [], 0, False), 0, 1, "C4 tier: 1 vGPU, cold regions in pinned host DRAM over PCIe")
            if not args.no_c4:
                swap["c4_policy_sweep"] = c5_policy_sweep(1, args.c5_gib, ("--laps", "3"))
                swap["c4_policy_sweep_fixed_frames"] = c5_policy_sweep(1, args.c5_gib, ("--fixed-frames", "--laps", "3"))
        else:
            # C5 as specified (SURVEY 8d): ONE vGPU homed on GPU 0, cold regions striped over the other N-1 GPUs;
            # evictions are pulled by the peers, prefetches by the home GPU.  The other ranks stay idle.
            barrier()
            if rank == 0:
                swap = summarize(swap_leg(0, multi.peers_of(0, world), 0, False), world - 1, 1,
                                 f"C5: 1 vGPU homed on GPU0, regions striped over {world - 1} peer GPUs (receiver-driven one-sided P2P)")
                c5 = c5_policy_sweep(world, args.c5_gib)
                if c5:
                    swap["c5_policy_sweep"] = c5
                # the same sweep with TFW_VS_FIXED_FRAMES: frames mapped once at every VA that will use them, direct-mapped
                # replacement (== LRU's choice for a sweep), no VMM call per migration
                swap["c5_policy_sweep_fixed_frames"] = c5_policy_sweep(world, args.c5_gib, ("--fixed-frames", "--laps", "3"))
            dist.barrier(group=cpu_group)   # the other GPUs must be genuinely idle while rank 0 measures: wait on the CPU
            barrier()
            # N vGPUs at once, each homed on its own GPU and spilling to all others: copy kernels stay on the
            # tenant's own GPU (TFW_VS_PUSH_EVICT), every NVLink port carries egress and ingress together.
            vals = multi.max_over_ranks(swap_leg(local, multi.peers_of(local, world), V.PUSH_EVICT, True), "cuda")
            swap_all = summarize(vals, world - 1, world, f"{world} vGPUs at once, each spilling to the {world - 1} other GPUs (home-driven copies)")

    # ---------------- C3: 4 vGPUs @ 25 % under the ERL limiter (north_star b) ----------------
    c3 = None
    if rank == 0 and world == 1 and not args.no_c3:
        c3 = {}
        for fb in ("device", "process"):
            try:
                r = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "limiter_c3.py"), "--seconds", "16", "--workers", "4", "--limit", "25",
                                    "--feedback", fb], capture_output=True, text=True, timeout=300)
                c3[f"feedback_{fb}"] = json.loads(r.stdout.strip().splitlines()[-1]) if r.returncode == 0 else {"error": r.stderr[-300:]}
            except Exception as e:
                c3[f"feedback_{fb}"] = {"error": f"{type(e).__name__}: {e}"[:300]}
        c3["note"] = ("4 worker processes, upLimit 25 each, saturating streams of 200 us kernels, 16 s (steady_* = the second half, after the controller has settled); the parent plays the hypervisor's 2 Hz loop "
                      "(AccelGetDeviceMetrics -> LimiterUpdateERL).  feedback=device is the reference's semantics: whole-device utilisation "
                      "is regulated towards each worker's target (quota_controller.go:388-436), so four tenants share ~25 % in total; "
                      "feedback=process feeds each worker its own SM utilisation instead")

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cpu = cpu_replay_baseline(raw, payload_per_step, os.cpu_count() or 1)

    w.close()
    pin.free()
    if rank == 0:
        line = {
            "metric": METRIC, "value": round(value, 2), "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": round(dev_ms_max / args.steps, 4), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "u8", "data": "synthetic",
            "config": bench_config(args, world),
            "e2e": {"value": round(e2e_val, 3), "unit": UNIT, "h2d_bytes_per_step": int(h2d_per_step), "d2h_bytes_per_step": int(d2h_per_step),
                    "steps": e2e_steps, "bound": "PCIe Gen5 x16 host->device copy"},
            "gpu_launches": int(launches),
            "roofline": {"bound": "hbm", "kernel": "tfw_mover_ldg", "achieved": round(achieved, 1), "peak": peak, "unit": UNIT,
                         "frac": round(achieved / peak, 4), "peak_source": peak_src, "traffic": traffic, "traffic_of": traffic_note,
                         "algorithmic_bytes_per_launch": int(algo_per_launch), "launches_per_step": int(mover_launches // args.steps),
                         "avg_launch_us": round(avg_launch_ms * 1e3, 2)},
            "clocks": clocks,
        }
        if cpu:
            line["cpu_baseline"] = cpu
        if overhead:
            line["overhead_vs_native"] = overhead
        if swap:
            line["swap"] = swap
        if swap_all:
            line["swap_all_vgpus_at_once"] = swap_all
        if c3:
            line["limiter_c3"] = c3
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
