#!/usr/bin/env python3
"""bench.py -- SSE chunks/sec of the streaming-response hot path on B200 (BASELINE.json metric).

A step = one pass of the hot path over one micro-batch of synthetic SSE input: workload C4 of BASELINE.json
(65,536 concurrent mixed cohere/groq/anthropic/ollama streams incl. tool_calls deltas, ~512 B mean chunk,
mode R = MCP reframe + JSON side-band) per GPU, every stream complete in the batch (11 SSE events).

  value      emitted chunks/s with the batch already resident in HBM (all kernels of the step, CUDA events); the timed steps
             rotate over three resident copies of the input, so no step finds its input in L2
  segmented  the same streams cut into k seeded TCP pieces: a step is k launches, the unterminated tails travel through
             the per-connection carry slots (no reset between the pieces)
  c5_strong  (N > 1) ONE population of --streams connections sharded by hash(conn_id) % N (BASELINE configs[4])
  e2e        through the C ABI a caller uses (sse_submit/sse_collect): pinned H2D + kernels + D2H per step
  roofline   algorithmic bytes of the step / its measured duration vs the measured HBM peak
  cpu_baseline  the CPU oracle port (oracle/, test infrastructure) on the host cores, same streams

Multi-GPU (torchrun, one rank per GPU): connections shard by hash(conn_id) % N, no collective on the data path.
`--impl reference` times the reference's CPU path (the oracle port: the reference is Go and cannot be built here).
`--dump-outputs DIR` writes what the last timed step computed as .npy files (dump_outputs): the inputs depend on the
arguments alone, so two builds run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

N_SLOTS = 4      # device-resident copies / batches in flight
N_ROT = 3        # resident input copies the timed steps rotate over
METRIC = "SSE chunks/sec @ 64k concurrent streams"
UNIT = "chunks/s"
WORKLOADS = {
    "C2": "C2: {n} concurrent OpenAI streams, passthrough (identity remap), 256 B mean chunk, mode P",
    "C3": "C3: {n} concurrent Anthropic (OpenAI-compatible) streams, 512 B mean chunk, mode R (MCP reframe + JSON side-band)",
    "C4": "C4: {n} concurrent mixed cohere/groq/anthropic/ollama streams incl. tool_calls deltas, 512 B mean chunk, "
          "mode R (MCP reframe + JSON side-band)",
}


def log(*a):
    print(*a, file=sys.stderr, flush=True)


def env_int(name, default):
    try:
        return int(os.environ.get(name, default))
    except ValueError:
        return default


def cpu_quota():
    """CPUs' worth of time the container may use (cgroup CFS quota / period), None when unlimited. A quota smaller than the
    affinity mask throttles a long multi-threaded run to the quota however many threads it starts: sustained throughput is
    what a server gets, so the CPU arm runs long enough (seconds) to be measured under it and reports it."""
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()[:2]                 # cgroup v2
        return None if q == "max" else float(q) / float(per)
    except (OSError, ValueError):
        pass
    try:
        q = float(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())            # cgroup v1
        per = float(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
        return None if q <= 0 else q / per
    except (OSError, ValueError):
        return None


def host_threads() -> int:
    """Threads for the CPU arm: the cores this process may run on, capped by the container's CPU quota (the GPU boxes of this
    pool show 128 logical cores in the affinity mask and a CFS quota of 16 CPUs)."""
    try:
        n = max(1, len(os.sched_getaffinity(0)))
    except (AttributeError, OSError):
        n = os.cpu_count() or 1
    q = cpu_quota()
    return n if q is None else max(1, min(n, int(np.ceil(q))))     # more threads than the quota only get throttled


def build_workload(n_streams: int, shard: int, workload: str, n_content=None):
    from inference_gateway_b200 import synth
    t0 = time.time()
    streams, mode = synth.make_config(workload, n_streams=n_streams, shard=shard, n_content=n_content)
    bodies = [b for b, _, _ in streams]
    n_events = sum(n for _, n, _ in streams)
    log(f"[bench] rank shard {shard}: generated {len(bodies)} streams, {sum(map(len, bodies)) / 1e6:.1f} MB, "
        f"{n_events} SSE events in {time.time() - t0:.1f}s")
    return bodies, (mode if mode is not None else 3), n_events


def fill_slot(eng, arena, segs, bodies, mode):
    off = 0
    lens = np.fromiter((len(b) for b in bodies), dtype=np.int64, count=len(bodies))
    offs = np.zeros(len(bodies), dtype=np.int64)
    aligned = (lens + 15) & ~15
    offs[1:] = np.cumsum(aligned)[:-1]
    total = int(offs[-1] + aligned[-1]) if len(bodies) else 0
    for b, o in zip(bodies, offs):
        arena[o:o + len(b)] = np.frombuffer(b, dtype=np.uint8)
    segs["conn"][:len(bodies)] = np.arange(len(bodies), dtype=np.uint32)
    segs["in_off"][:len(bodies)] = offs.astype(np.uint32)
    segs["in_len"][:len(bodies)] = lens.astype(np.uint32)
    segs["mode"][:len(bodies)] = mode
    segs["provider"][:len(bodies)] = np.arange(len(bodies), dtype=np.uint8) % 4   # the connection's provider (flavours cycle cohere/groq/anthropic/ollama)
    segs["reserved"][:len(bodies)] = 0
    return len(bodies), total, int(lens.sum())


class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.p = None
        self.idx = gpu_index
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--id={gpu_index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                       "-lms", "50"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except OSError:
            self.p = None

    def stop(self):
        if not self.p:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.p.terminate()
        try:
            out, _ = self.p.communicate(timeout=5)
        except subprocess.TimeoutExpired:
            self.p.kill()
            out, _ = self.p.communicate()
        sm, mx, reasons = [], [], set()
        for line in out.splitlines():
            f = [x.strip() for x in line.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def _oracle_arrays(bodies, mode):
    arena = np.frombuffer(b"".join(bodies), dtype=np.uint8)
    lens = np.fromiter((len(b) for b in bodies), dtype=np.uint32, count=len(bodies))
    offs = np.zeros(len(bodies), dtype=np.uint64)
    offs[1:] = np.cumsum(lens.astype(np.uint64))[:-1]
    return arena, offs, lens, np.full(len(bodies), mode, dtype=np.uint8)


def cpu_baseline(bodies, mode, threads: int, target_s: float = 3.0, with_single: bool = True):
    """Times the oracle port (CPU restatement of the reference path) on the SAME streams as the GPU arm: one pool of
    `threads` threads, enough passes over all streams for >= target_s seconds of wall time."""
    from oracle import orc
    arena, offs, lens, modes = _oracle_arrays(bodies, mode)
    passes = 1
    secs, _, frames, _ = orc.bench_run(arena, offs, lens, modes, threads, passes)        # warm-up pass (page in, allocators)
    while secs < 0.6 * target_s and passes < (1 << 14):      # grow by at most 8x per try: a short run overstates the sustained rate
        passes = int(min(1 << 14, np.ceil(passes * min(8.0, target_s / max(secs, 1e-4)))))
        secs, _, frames, _ = orc.bench_run(arena, offs, lens, modes, threads, passes)
    # (a short run can be far faster per pass than a long one: under a cgroup CPU quota the first tens of milliseconds run on
    #  every core of the affinity mask, then the container is throttled to its quota; the long run is the one reported)
    quota = cpu_quota()
    out = {"value": frames / secs, "unit": UNIT, "cores": threads, "kind": "port", "seconds": secs,
           "cpu_quota_cores": quota,
           "sample": f"all {len(bodies)} streams of the workload x {passes} passes ({arena.size / 1e6:.0f} MB per pass), "
                     f"{secs:.1f} s of wall time, one pool of {threads} threads; oracle/sse_oracle.c (C restatement; the "
                     f"reference is Go and no Go toolchain exists on this box)"}
    if with_single:
        sub = max(1, len(bodies) // 8)
        a1, o1, l1, m1 = _oracle_arrays(bodies[:sub], mode)
        s1, _, f1, _ = orc.bench_run(a1, o1, l1, m1, 1, 1)
        out["value_1_thread"] = f1 / s1
        out["sample"] += f"; 1 thread: the first {sub} streams once, {s1:.1f} s"
    return out


def workload_text(args):
    return WORKLOADS.get(args.workload, args.workload + ": {n} streams").format(n=args.streams)


def run_reference(args, rank, world):
    """--impl reference: the reference's CPU path (oracle port) with all host threads, rank 0 only, on the GPU arm's streams."""
    if rank != 0:
        return
    threads = host_threads()
    bodies, mode, _ = build_workload(args.streams, 0, args.workload)
    if args.mode is not None:
        mode = args.mode
    vals = []
    for _ in range(args.warmup):
        cpu_baseline(bodies, mode, threads, target_s=0.3, with_single=False)
    for _ in range(args.steps):
        vals.append(cpu_baseline(bodies, mode, threads, target_s=1.5, with_single=False))
    v = statistics.mean(x["value"] for x in vals)
    step_ms = 1e3 * statistics.mean(x["seconds"] for x in vals)
    cb = dict(vals[-1]); cb["value"] = v
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": step_ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "u8", "data": "synthetic",
            "config": {"workload": workload_text(args), "streams_per_gpu": args.streams, "threads": threads,
                       "step": "one bounded sample: all streams of the workload, as many passes as fill >= 1.5 s",
                       "parity": "parity unpinned: the arm is the C restatement of the Go path (oracle/), not a Go run"},
            "cpu_baseline": cb,
            "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


def time_steps(torch, fn, steps):
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for i in range(steps):
        fn(i)
    ev1.record()
    torch.cuda.synchronize()
    return ev0.elapsed_time(ev1)


def bind_to_gpu_numa_node(torch, local_rank):
    """Pins this rank to the CPU cores of the NUMA node its GPU hangs off (sysfs local_cpulist of the GPU's PCI function), so
    that the pinned staging buffers the library allocates next are first-touched on that node and the H2D / D2H copies do not
    cross the socket interconnect. Returns a description for the JSON line; None when the topology cannot be read."""
    try:
        bus = torch.cuda.get_device_properties(local_rank).pci_bus_id
        dom = torch.cuda.get_device_properties(local_rank).pci_domain_id
        dev = torch.cuda.get_device_properties(local_rank).pci_device_id
        path = f"/sys/bus/pci/devices/{dom:04x}:{bus:02x}:{dev:02x}.0"
        cpus = open(os.path.join(path, "local_cpulist")).read().strip()
        node = int(open(os.path.join(path, "numa_node")).read().strip())
        want = set()
        for part in cpus.split(","):
            lo, _, hi = part.partition("-")
            want.update(range(int(lo), int(hi or lo) + 1))
        want &= os.sched_getaffinity(0)
        if not want:
            return None
        os.sched_setaffinity(0, want)
        return {"numa_node": node, "cpus": cpus, "bound_threads": len(want)}
    except (OSError, ValueError, AttributeError):
        return None


def per_segment(res):
    """(frames, frame bytes, records) each segment of a batch result delivers: its inline run plus the runs linked from it."""
    cs = np.concatenate([[0], np.cumsum(res.frames["len"].astype(np.int64))])
    ff, frames = res.segs["frame_first"].astype(np.int64), res.segs["frame_count"].astype(np.int64)
    nbytes, recs = cs[ff + frames] - cs[ff], res.segs["rec_count"].astype(np.int64)
    owner, cur = np.arange(len(res.segs)), res.segs["next"].astype(np.int64)
    while True:
        live = cur != 0xFFFFFFFF
        owner, cur = owner[live], cur[live]
        if not cur.size:
            return frames, nbytes, recs
        run = res.runs[cur]
        a, b = run["frame_first"].astype(np.int64), run["frame_count"].astype(np.int64)
        np.add.at(frames, owner, b)
        np.add.at(nbytes, owner, cs[a + b] - cs[a])
        np.add.at(recs, owner, run["rec_count"].astype(np.int64))
        cur = run["next"].astype(np.int64)


def delivered(res):
    """(frames, frame bytes) a batch result delivers: the inline run of every segment plus the runs linked from it."""
    frames, nbytes, _ = per_segment(res)
    return int(frames.sum()), int(nbytes.sum())


DUMP_BYTES = 64_000_000    # --dump-outputs writes at most this much
DUMP_SEED = 0xD0           # seeds the order in which connections are sampled
CONN_COLS = ("conn", "carry_len", "flags", "frames", "frame_bytes", "records")
SAMPLE_COLS = ("conn", "frames", "records")
REC_COLS = ("conn", "frame", "flags", "payload_len", "n_choices", "prompt_tokens", "completion_tokens", "total_tokens",
            "content_len", "tool_calls")
TC_COLS = ("record", "index", "has_id", "has_type", "has_function", "id_len", "type_len", "name_len", "args_len")


def dump_outputs(res, out_dir):
    """Writes what a caller receives from one batch result as <name>.npy under out_dir (at most DUMP_BYTES in all):
      connections   one row per connection (CONN_COLS): its sse_seg_result and what it delivered
      sample        the connections shown in full below, in a seeded order, as many as fit (SAMPLE_COLS)
      frame_len, frame_bytes          their delivered frames in stream order, and the bytes of those frames
      records, content_bytes          their delivered records (REC_COLS; frame = ordinal among the connection's frames,
                                      -1 if not emitted; usage -1 when absent) and the content each carries
      tool_calls, tool_call_bytes     the tool calls of those records (TC_COLS; record = row in records) and their id, type,
                                      name and arguments
    Arena offsets and table indices are resolved to what they point at, and the flag that says which arena a content
    span lives in is cleared: the kernels place frames and records in whatever order their atomic allocations run, so
    positions change from run to run while what a caller reads through them does not. A connections table larger than a
    quarter of the budget keeps the first connections of the seeded order (sorted by id).
    Returns the number of connections written in full."""
    from inference_gateway_b200 import _abi as A
    from tests.util import rec_to_dict
    frames, nbytes, recs = per_segment(res)
    n = len(res.segs)
    order = np.random.default_rng(DUMP_SEED).permutation(n)
    rows = np.sort(order[:min(n, DUMP_BYTES // 4 // (8 * len(CONN_COLS)))])
    out = {"connections": np.stack([rows, res.segs["carry_len"][rows], res.segs["flags"][rows], frames[rows], nbytes[rows],
                                    recs[rows]], axis=1).astype(np.float64)}
    budget = DUMP_BYTES - 4096 - out["connections"].nbytes          # 4096: the .npy headers
    sample, flen, fbytes, rec_rows, content, tc_rows, tc_bytes = [], [], [], [], [], [], []
    for c in map(int, order):
        fidx = [k for ff, fc, _, _ in res.seg_runs(c) for k in range(ff, ff + fc)]
        fb = [res.at(int(res.frames[k]["off"]), int(res.frames[k]["len"])) for k in fidx]
        ordinal = {k: j for j, k in enumerate(fidx)}
        rr, cb, tr, tb = [], [], [], []
        for ri in res.seg_recs(c):
            d = rec_to_dict(res, ri)
            tcs = d.get("tcs", [])
            for t in tcs:
                parts = [t["id"] or b"", t["type"] or b"", t["name"], t["args"]]
                tr.append([len(rec_rows) + len(rr), t["index"], t["id"] is not None, t["type"] is not None, t["function"]]
                          + [len(p) for p in parts])
                tb.extend(parts)
            cb.append(d.get("content", b""))
            rr.append([c, ordinal.get(d["frame"], -1), d["flags"] & ~A.F_CONTENT_TEXT, d["payload_len"], d.get("n_choices", 0),
                       *(d.get("usage") or (-1, -1, -1)), len(cb[-1]), len(tcs)])
        cost = (4 * sum(map(len, fb + cb + tb)) + 8 * (len(SAMPLE_COLS) + len(fb) + len(REC_COLS) * len(rr)
                                                       + len(TC_COLS) * len(tr)))
        if cost > budget:
            break
        budget -= cost
        sample.append([c, len(fb), len(rr)])
        flen += map(len, fb); fbytes += fb; rec_rows += rr; content += cb; tc_rows += tr; tc_bytes += tb
    out["sample"] = np.array(sample, dtype=np.float64).reshape(-1, len(SAMPLE_COLS))
    out["frame_len"] = np.array(flen, dtype=np.float64)
    out["frame_bytes"] = np.frombuffer(b"".join(fbytes), dtype=np.uint8).astype(np.float32)
    out["records"] = np.array(rec_rows, dtype=np.float64).reshape(-1, len(REC_COLS))
    out["content_bytes"] = np.frombuffer(b"".join(content), dtype=np.uint8).astype(np.float32)
    out["tool_calls"] = np.array(tc_rows, dtype=np.float64).reshape(-1, len(TC_COLS))
    out["tool_call_bytes"] = np.frombuffer(b"".join(tc_bytes), dtype=np.uint8).astype(np.float32)
    os.makedirs(out_dir, exist_ok=True)
    for name, arr in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), arr)
    return len(sample)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--streams", type=int, default=None, help="concurrent streams per GPU (default: the workload's)")
    ap.add_argument("--workload", default="C4", choices=sorted(WORKLOADS))
    ap.add_argument("--mode", type=int, default=None, help="override the workload's mode bits (0 P, 2 P+parse, 3 R+parse)")
    ap.add_argument("--flags", type=int, default=0, help="sse_config.flags (4 single-pass tile kernel, 8 copy-out, 16 skeleton-template replay)")
    ap.add_argument("--segments", type=int, default=4, help="TCP pieces per stream of the segmented measurement (0: skip it)")
    ap.add_argument("--n-content", type=int, default=None, help="content deltas per stream (default: the config's 7)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-strong", action="store_true")
    ap.add_argument("--no-numa", action="store_true", help="do not bind the rank to its GPU's NUMA node")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one computed as DIR/<name>.npy (see dump_outputs); "
                         "under torchrun each rank writes to DIR/rank<r>")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the results of the GPU path (--impl b200)")
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup
    if args.streams is None:
        args.streams = {"C2": 4096, "C3": 16384, "C4": 65536}[args.workload]
    args.segments = max(0, min(args.segments, N_SLOTS))

    rank, world, local_rank = env_int("RANK", 0), env_int("WORLD_SIZE", 1), env_int("LOCAL_RANK", 0)
    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    import torch.distributed as dist
    if not torch.cuda.is_available():
        sys.exit("bench.py: no CUDA device; the product path has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    all_cpus = os.sched_getaffinity(0)
    numa = None if args.no_numa else bind_to_gpu_numa_node(torch, local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        # stdout carries exactly one JSON line: NCCL printf()s its version banner to stdout when the communicator is created
        # (NCCL_DEBUG=VERSION/INFO), so fd 1 points at stderr until the first collective has run
        sys.stdout.flush()
        saved_stdout = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
            dist.barrier()
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved_stdout, 1)
            os.close(saved_stdout)

    from inference_gateway_b200 import SseEngine, shard as sh, synth
    # weak scaling: every rank owns its own population of --streams connections (seeded by the rank)
    bodies, mode, n_events = build_workload(args.streams, rank, args.workload, args.n_content)
    if args.mode is not None:
        mode = args.mode
    in_payload = sum(map(len, bodies))
    eng = SseEngine(device=local_rank, max_conns=len(bodies), bytes_per_batch=in_payload, n_slots=N_SLOTS, carry_slot_bytes=16384, flags=args.flags)
    # a non-default torch stream: its handle is passed to the library so that the kernels, the resets and the
    # CUDA events of the timed region all live on the same stream (handle 0 would mean "library stream")
    tstream = torch.cuda.Stream()
    torch.cuda.set_stream(tstream)
    stream = tstream.cuda_stream
    assert stream != 0

    def sync_all():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- resident input: N_ROT copies, the timed steps rotate over them (no step finds its input in L2)
    slots = []
    for _ in range(N_SLOTS):
        sl, arena, segs = eng.acquire()
        slots.append((sl, arena, segs))
    n_segs = in_bytes = 0
    for sl, arena, segs in slots[:N_ROT]:
        n_segs, in_bytes, _ = fill_slot(eng, arena, segs, bodies, mode)
        eng.upload(sl, n_segs, in_bytes, stream)
    torch.cuda.synchronize()

    def step(i):
        eng.reset_all(stream)          # a step = a fresh population of connections
        eng.launch(slots[i % N_ROT][0], n_segs, stream)

    for i in range(args.warmup):
        step(i)
    torch.cuda.synchronize()
    res = eng.download(slots[(args.warmup - 1) % N_ROT][0], stream)   # untimed: counts for the report + sanity
    counts = dict(frames=int(res.raw.n_frames), recs=int(res.raw.n_recs), tcs=int(res.raw.n_tcs), usages=int(res.raw.n_usages),
                  out_bytes=int(res.raw.out_bytes), text_bytes=int(res.raw.text_bytes), runs=int(res.raw.n_runs),
                  in_bytes=in_payload, segs=n_segs, events=n_events)
    # frames of lines after a terminating chunk are allocated but cut from the result (their runs are unlinked): count what
    # is delivered, and its bytes (b_out of SURVEY 8(d)) wherever they live -- the out arena or spans of the input
    counts["frames"], counts["frame_bytes"] = delivered(res)
    counts["zero_copy_frames"] = int(np.count_nonzero(res.frames["off"] >= res.in_base))
    terminated = int(np.count_nonzero(res.segs["flags"] & 1))
    ok_recs = int(np.count_nonzero(res.recs["flags"] & 1))

    sync_all()
    sampler = ClockSampler(local_rank)
    # nvidia-smi needs a few hundred ms before its first sample: keep the GPU under the same load (untimed) meanwhile,
    # so that the clock samples bracket the timed region and are all taken under load
    t_pre = time.perf_counter()
    i = 0
    while time.perf_counter() - t_pre < 1.2:
        step(i); i += 1
        torch.cuda.synchronize()
    sync_all()
    launches0 = eng.launch_count()
    dev_ms = time_steps(torch, step, args.steps)
    sync_all()
    launches = eng.launch_count() - launches0
    clocks = sampler.stop()
    if args.dump_outputs:
        out_dir = args.dump_outputs if world == 1 else os.path.join(args.dump_outputs, f"rank{rank}")
        n_full = dump_outputs(eng.download(slots[(args.steps - 1) % N_ROT][0], stream), out_dir)
        log(f"[bench] outputs of the last timed step -> {out_dir} ({n_full} of {n_segs} connections in full)")

    # ---- the same streams in k seeded TCP pieces: a step is k launches, tails go through the carry slots
    segmented = None
    if args.segments >= 2:
        k = args.segments
        rng = np.random.default_rng(0xB200)
        pieces = [synth.random_cuts(rng, b, k) for b in bodies]
        piece_meta = []
        for b_i, (sl, arena, segs) in enumerate(slots[:k]):
            part = [p[b_i] if b_i < len(p) else b"" for p in pieces]
            ns, nb, _ = fill_slot(eng, arena, segs, part, mode)
            eng.upload(sl, ns, nb, stream)
            piece_meta.append((sl, ns))
        torch.cuda.synchronize()

        def seg_step(_i):
            eng.reset_all(stream)
            for sl, ns in piece_meta:
                eng.launch(sl, ns, stream)

        for i in range(3):
            seg_step(i)
        torch.cuda.synchronize()
        seg_frames = 0
        for sl, ns in piece_meta:      # frames of the last warm-up step (sanity: the same chunks come out)
            seg_frames += delivered(eng.download(sl, stream))[0]
        sync_all()
        seg_ms = sh.max_over_ranks(time_steps(torch, seg_step, args.steps), world)
        seg_tot = sh.reduce_counters({"f": seg_frames}, world)["f"]
        segmented = {"pieces_per_stream": k, "launches_per_step": (2 if args.flags & 4 else 6) * k, "value": seg_tot * args.steps / (seg_ms / 1e3), "unit": UNIT,
                     "ms_per_step": seg_ms / args.steps, "chunks_emitted_per_step": seg_tot,
                     "note": "seeded random TCP cuts; every piece is its own micro-batch, unterminated tails are carried on the device"}
        if seg_frames != counts["frames"]:
            segmented["warning"] = f"emitted {seg_frames} chunks, the one-shot batch emitted {counts['frames']}"

    # ---- BASELINE configs[4]: ONE population of --streams connections sharded over the ranks by hash(conn_id) % N
    strong = None
    if world > 1 and not args.no_strong:
        g_bodies, _, _ = build_workload(args.streams, 0, args.workload, args.n_content)
        mine = np.nonzero(sh.shard_of(np.arange(len(g_bodies), dtype=np.uint64), world) == rank)[0]
        my = [g_bodies[int(c)] for c in mine]
        s_meta = []
        for sl, arena, segs in slots[:N_ROT]:
            ns, nb, _ = fill_slot(eng, arena, segs, my, mode)
            eng.upload(sl, ns, nb, stream)
            s_meta.append((sl, ns))
        torch.cuda.synchronize()

        def strong_step(i):
            eng.reset_all(stream)
            eng.launch(s_meta[i % N_ROT][0], s_meta[i % N_ROT][1], stream)

        for i in range(3):
            strong_step(i)
        torch.cuda.synchronize()
        s_frames = delivered(eng.download(s_meta[2][0], stream))[0]
        sync_all()
        s_ms = sh.max_over_ranks(time_steps(torch, strong_step, args.steps), world)
        s_tot = sh.reduce_counters({"f": s_frames, "n": len(my)}, world)
        strong = {"scaling": "strong", "total_streams": s_tot["n"], "value": s_tot["f"] * args.steps / (s_ms / 1e3), "unit": UNIT,
                  "ms_per_step": s_ms / args.steps, "sharding": "shard_of(conn_id) = fibonacci hash % n_gpus (inference_gateway_b200/shard.py)"}

    # ---- end to end through the public C ABI: pinned H2D + kernels + D2H every step, three slots in flight
    e2e = None
    if not args.no_e2e:
        for sl, arena, segs in slots:
            fill_slot(eng, arena, segs, bodies, mode)
        for sl, _, _ in slots:
            eng.release(sl)
        h2d = in_bytes + n_segs * 16
        d2h = (counts["out_bytes"] + 8 * counts["frames"] + 32 * counts["recs"] + 48 * counts["tcs"] + 24 * counts["usages"]
               + counts["text_bytes"] + 20 * counts["runs"] + 32 * n_segs + 64)
        depth = 3

        def e2e_steps(k):
            inflight = []
            frames = 0
            for i in range(k):
                s2, _, _ = eng.acquire()      # pinned staging already holds the step's input
                eng.reset_all(0)
                eng.submit(s2, n_segs, in_bytes)
                inflight.append(s2)
                if len(inflight) == depth:
                    s_old = inflight.pop(0)
                    r = eng.collect(s_old)
                    frames += int(r.raw.n_frames)
                    eng.release(s_old)
            for s_old in inflight:
                r = eng.collect(s_old)
                frames += int(r.raw.n_frames)
                eng.release(s_old)
            return frames

        e2e_steps(depth)
        sync_all()
        k_e2e = args.steps
        t0 = time.perf_counter()
        fr = e2e_steps(k_e2e)
        torch.cuda.synchronize()
        e2e_s = time.perf_counter() - t0
        e2e_s = sh.max_over_ranks(e2e_s, world)
        fr_all = sh.reduce_counters({"f": fr}, world)["f"]
        e2e = {"value": fr_all / e2e_s, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
               "steps": k_e2e, "ms_per_step": 1e3 * e2e_s / k_e2e, "h2d_gbs_per_rank": h2d / (e2e_s / k_e2e) / 1e9,
               "path": f"sse_acquire/sse_submit/sse_collect/sse_release, {depth} slots in flight, host buffers pinned"}

    dev_ms = sh.max_over_ranks(dev_ms, world)
    tot = sh.reduce_counters(counts, world)
    chunks_per_step = tot["frames"]
    value = chunks_per_step * args.steps / (dev_ms / 1e3)

    # ---- roofline of the step (rank 0's launches): algorithmic bytes / measured duration
    # SURVEY 8(d): b_in read once + b_out delivered once + frame table + records (+ per-segment descriptors and state).
    # moved_bytes is what the zero-copy path really has to touch: frames that are spans of the input are never written.
    side = (8 * counts["frames"] + 32 * counts["recs"] + 48 * counts["tcs"] + 24 * counts["usages"] + counts["text_bytes"]
            + (16 + 32 + 16) * n_segs)
    alg_bytes = counts["in_bytes"] + counts["frame_bytes"] + side
    moved_bytes = counts["in_bytes"] + counts["out_bytes"] + side
    kern_s = (dev_ms / 1e3) / args.steps
    peak, peak_src = 6650.0, "fallback"
    try:
        mp = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        peak, peak_src = float(mp["hbm_gbs"]), "measured"
    except (OSError, KeyError, ValueError):
        pass
    achieved = alg_bytes / kern_s / 1e9
    traffic = None
    try:
        tj = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
        if tj.get("workload") == args.workload and tj.get("streams") == args.streams and args.mode in (None, 3) and not args.flags:
            traffic = tj.get("dram_bytes_per_launch")
    except (OSError, ValueError):
        pass
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": traffic, "peak_source": peak_src,
                "kernel": ("sse_fused_kernel (+ sse_plan_kernel: 2 launches per step; the whole step is timed)" if args.flags & 4 else
                           "sse_stream_kernel<produce> + sse_decode_kernel (+ bucket hist/scan/scatter and finalize: 6 launches per step; "
                           "the whole step is timed)"),
                "alg_bytes_per_launch": alg_bytes, "moved_bytes_per_launch": moved_bytes,
                "zero_copy_frames": counts["zero_copy_frames"], "kernel_ms": 1e3 * kern_s,
                "hbm_read_frac": counts["in_bytes"] / kern_s / 1e9 / peak}

    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": dev_ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "u8", "data": "synthetic",
        "config": {"workload": workload_text(args), "streams_per_gpu": args.streams, "total_streams": args.streams * world,
                   "batch": "every stream complete in one micro-batch (11 SSE events per stream and step)",
                   "sse_events_per_step": tot["events"], "chunks_emitted_per_step": tot["frames"],
                   "records_decoded_per_step": tot["recs"], "mean_event_bytes": tot["in_bytes"] / max(1, tot["events"]),
                   "input_bytes_per_step": tot["in_bytes"], "sharding": "hash(conn_id) % n_gpus, no collective",
                   "l2": f"the timed steps rotate over {N_ROT} resident copies of the input ({in_payload / 1e6:.0f} MB each; L2 is 126 MB)",
                   "streams_terminated": terminated, "records_json_ok": ok_recs,
                   "parity": "bit-exact against oracle/ (C restatement of the Go path); parity unpinned against a Go run"},
        "roofline": roofline, "gpu_launches": int(launches), "clocks": clocks,
    }
    if segmented:
        line["segmented"] = segmented
    if strong:
        line["c5_strong"] = strong
    if e2e:
        line["e2e"] = e2e
    line["config"]["numa"] = numa or "not bound"
    if rank == 0 and not args.no_cpu_baseline and world == 1:
        os.sched_setaffinity(0, all_cpus)          # the CPU arm gets every core the process may use, not just the GPU's node
        try:
            line["cpu_baseline"] = cpu_baseline(bodies, mode, host_threads())
        except Exception as ex:  # the checker library is test infrastructure; report, do not hide
            line["cpu_baseline"] = {"value": None, "unit": UNIT, "cores": 0, "kind": "port", "sample": f"unavailable: {ex}"}
    if rank == 0:
        print(json.dumps(line), flush=True)
    eng.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
