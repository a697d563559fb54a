#!/usr/bin/env python
"""bench.py -- Mpoints/s segmented on SemanticKITTI-shaped synthetic 64-beam streams.

Workload (BASELINE.json configs[1], batched so that it can be HBM-bound at all): B independent
synthetic streams per GPU, ~120 k points per scan, 300 x 300 cells @ 0.33 m (99 m map).  One
"step" = one scan of every stream: GroundGrid::update (map roll to the new ego pose) followed by
GroundSegmentation::filter_cloud (rasterise -> patch detection -> spiral interpolation ->
labelling).  Streams are independent (own map, own rolling terrain prior); scans of one stream
are processed in order because scan t+1 reads the prior written by scan t.

  value : whole-job Mpoints/s with the clouds already resident in HBM (CUDA events on the
          handle's stream, max over ranks)
  e2e   : same metric through the reference-facing C-ABI call with HOST buffers: pinned host
          clouds are copied H2D and the labels D2H inside the timed region, every step
  roofline : dominant kernel, algorithmic bytes (DESIGN.md) / its own CUDA-event duration
  cpu_baseline : the CPU oracle (reference semantics) on this host, bounded sample

  sub-results keyed in the same JSON line: cfg3 (128 beams, 600 x 600), cfg4 (four LiDARs, 364 x 364), the literal
  drop-in call (gg_filter_cloud, pageable host memory, one stream), per-kernel roofline of a serialised step, and --
  with more than one rank -- the NCCL broadcast of the rolling terrain prior with a label check on the receivers.

`--impl reference` times the reference's own CPU implementation on all host cores, one independent stream per core:
oracle/_ref (the unmodified reference sources compiled on CPU stand-ins, cpu_baseline.kind = "reference") when the
prebuilt library is there, else the oracle port.

`--dump-outputs DIR` writes what the last timed step computed for a fixed sample of streams (dump_outputs) as .npy files;
the inputs depend only on the arguments, so two builds run with the same arguments can be compared output for output.
"""
import argparse
import json
import math
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

DIM_M, RES, N_CELLS = 99.0, 0.33, 300
PCAP = 131072
METRIC = "Mpoints/sec segmented (64-beam scan)"
UNIT = "Mpoints/s"


def pingpong(t, s):
    """0,1,..,s-1,s-2,..,1,0,1,...: the ego drives 1 m per scan forth and back over s poses."""
    if s == 1:
        return 0
    period = 2 * (s - 1)
    k = t % period
    return k if k < s else period - k


SENSORS = {"64": ("scan_64", PCAP), "128": ("scan_128", 262144), "4x64": ("scan_4lidar", 524288)}


def _gen_task(args):
    from groundgrid_b200 import synth

    seed, pose, n_pose, sensor = args
    fn, cap = SENSORS[sensor]
    scene = synth.make_scene(seed=seed, stream_len=float(n_pose))
    pts, org = getattr(synth, fn)(scene, ego_xy=(float(pose), 0.0), yaw=0.0, seed=seed * 31 + pose)
    return pts[:cap], org


def generate_streams(first_seed, n_streams, n_pose, procs, sensor="64"):
    """[(points, origin)] indexed [stream][pose]; numpy ray casting in worker processes (before CUDA init)."""
    tasks = [(first_seed + b, s, n_pose, sensor) for b in range(n_streams) for s in range(n_pose)]
    if procs > 1:
        import multiprocessing as mp

        with mp.get_context("fork").Pool(procs) as pool:
            res = pool.map(_gen_task, tasks, chunksize=1)
    else:
        res = [_gen_task(t) for t in tasks]
    return [[res[b * n_pose + s] for s in range(n_pose)] for b in range(n_streams)]


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during a timed region (B200_PROFILING.md recipe)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu_index = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "20",
                                          "-i", str(self.gpu_index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.12)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons, power = [], [], set(), []
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
                power.append(float(f[3]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons), "samples": len(sm),
                "power_w_max": float(max(power))}


def P_mean_single(npts):
    return float(npts[0].mean())


def host_cores():
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


# algorithmic bytes per scan of each kernel (DESIGN.md section "Roofline accounting"; SURVEY.md 8d):
#   A scatter 20 P + 16 N^2 | B classify 36 N^2 | C spiral 16 N^2 | D label 25 P + 4 N^2  => 45 P + 72 N^2
def algorithmic_bytes(kernel, P, N2):
    table = {
        "k_rasterize": 20.0 * P,            # points (16 B packed x,y,z,ring) + prior-G gather (4 B)
        "k_cell_stats": 16.0 * N2,          # write count, mean, M2, min
        "k_detect": 36.0 * N2,              # read count, M2, min, E, G, C; write var, G, C
        "k_spiral": 16.0 * N2,              # read + write G, C
        "k_label": 25.0 * P + 4.0 * N2,     # points 16 B, gather G + var 8 B, label 1 B; obstacle layer
        "k_roll_gather": 8.0 * N2,
        "k_roll_commit": 8.0 * N2,
    }
    return table.get(kernel, 0.0)             # sort / scan kernels: ordering overhead, no algorithmic bytes


def pose_T(s):
    """base_link <- map of pose s of a stream, as (quaternion, translation) and as the 3x4 matrix tf2 derives from it."""
    from groundgrid_b200 import synth

    q, t = synth.base_from_map_qt(float(s), 0.0)
    return q, t, synth.tf2_matrix(q, t)


def make_cpu_impl(threads):
    """The reference's CPU implementation of the path: oracle/_ref (the reference's own sources) if the prebuilt library
    is there, else the oracle port.  Returns (object, kind)."""
    from oracle import ref as refmod

    if refmod.available():
        r = refmod.Reference(DIM_M, RES)
        r.set_config(thread_count=threads)
        return r, "reference"
    from oracle import Oracle

    return Oracle(DIM_M, RES), "port"


def cpu_scan(impl, kind, t, s, pts, org, threads):
    q, tt, T = pose_T(s)
    if t:
        if kind == "reference":
            impl.update(float(s), 0.0, q, tt)
        else:
            impl.update(float(s), 0.0, T)
    if kind == "reference":
        return impl.filter_cloud(pts, org, 0.0)[0]
    return impl.filter_cloud(pts, org, 0.0, threads=threads)[0]


def run_cpu_stream(scans, n_scans, threads, labels_out=None):
    """Replays one stream on the CPU (update + filter_cloud per scan); returns (seconds, points, kind)."""
    impl, kind = make_cpu_impl(threads)
    impl.init_map(0.0, 0.0, 0.0)
    S = len(scans)
    spent = 0.0
    pts_total = 0
    for t in range(n_scans):
        s = pingpong(t, S)
        pts, org = scans[s]
        t0 = time.perf_counter()
        lab = cpu_scan(impl, kind, t, s, pts, org, threads)
        spent += time.perf_counter() - t0
        pts_total += len(pts)
        if labels_out is not None:
            labels_out[t] = lab
    return spent, pts_total, kind


def reference_arm(args, rank, world):
    """The reference's CPU implementation, one independent stream per host core (thread_count = 1 per stream: with one
    stream per core the shipped 8 insert + 4 detect threads would only oversubscribe; cpu_baseline of the GPU arm reports
    the shipped threading on one stream beside it)."""
    if rank != 0:
        return
    cores = host_cores()
    workers = max(1, cores)
    S = min(args.pool, 2)
    streams = generate_streams(5000, workers, S, min(workers, 32))
    impls, kind = [], "port"
    for w in range(workers):
        impl, kind = make_cpu_impl(1)
        impl.init_map(0.0, 0.0, 0.0)
        impls.append(impl)
    pts_per_step = sum(len(streams[w][0][0]) for w in range(workers))

    def one(w, t):
        s = pingpong(t, S)
        pts, org = streams[w][s]
        cpu_scan(impls[w], kind, t, s, pts, org, 1)

    def step(t):
        ths = [threading.Thread(target=one, args=(w, t)) for w in range(workers)]
        for th in ths:
            th.start()
        for th in ths:
            th.join()

    steps = args.steps               # every step is one scan on every core
    for t in range(args.warmup):
        step(t)
    t0 = time.perf_counter()
    for t in range(args.warmup, args.warmup + steps):
        step(t)
    dt = time.perf_counter() - t0
    value = pts_per_step * steps / dt / 1e6
    what = ("oracle/_ref: the unmodified reference sources (GroundSegmentation.cpp, GroundGrid.cpp) on CPU stand-ins" if kind == "reference"
            else "oracle port of the reference")
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": steps,
        "warmup": args.warmup, "ms_per_step": dt / steps * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32/f64", "data": "synthetic",
        "config": {"workload": f"{workers} independent SemanticKITTI-shaped synthetic 64-beam streams (one per host core), "
                               f"~120k pts/scan, {N_CELLS}x{N_CELLS} @ {RES} m; step = one scan of every stream (update + filter_cloud) "
                               f"on {what} (thread_count=1 per stream); the GPU arm runs {args.streams} streams of the same shape per GPU",
                   "streams": workers, "points_per_step": pts_per_step},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": workers, "kind": kind,
                         "sample": f"{steps} steps x {workers} scans after {args.warmup} warm-up steps"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


DUMP_STREAMS = 32   # 32 streams x (labels and output order of <= 131072 points + two 300 x 300 layers) in float32: <= 57 MB


def dump_outputs(g, out_dir, npts):
    """What the last timed step handed back, for a fixed seeded sample of the streams: per input point the label, the
    output order (input index of each output point, gg_get_output) and, per cell, the ground height and confidence
    that the next scan of the stream reads.  Per-stream arrays are concatenated in the order of streams.npy."""
    os.makedirs(out_dir, exist_ok=True)
    sample = np.sort(np.random.default_rng(0).choice(g.n_slots, min(DUMP_STREAMS, g.n_slots), replace=False))
    labels = [g.download_labels(int(npts[b]), slot=int(b)) for b in sample]
    g.synchronize()
    order = [g.get_output(slot=int(b))[0] for b in sample]
    out = {"streams": sample.astype(np.float64),
           "points_per_stream": np.array([len(v) for v in labels], np.float64),
           "labels": np.concatenate(labels).astype(np.float32),
           "output_points_per_stream": np.array([len(v) for v in order], np.float64),
           "output_order": np.concatenate(order).astype(np.float32),   # indices < 2^24: exact in float32
           "ground": np.stack([g.layer("ground", int(b)) for b in sample]),
           "groundpatch": np.stack([g.layer("groundpatch", int(b)) for b in sample])}
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def bind_to_gpu_numa_node(torch, local_rank):
    """numactl --cpunodebind equivalent: keep this rank (and the pinned host buffers it allocates next) on
    the CPUs of the socket its GPU hangs off.  Returns a description for the JSON line."""
    try:
        pr = torch.cuda.get_device_properties(local_rank)
        bdf = "%04x:%02x:%02x.0" % (pr.pci_domain_id, pr.pci_bus_id, pr.pci_device_id)
        with open("/sys/bus/pci/devices/%s/local_cpulist" % bdf) as f:
            text = f.read().strip()
        cpus = set()
        for part in text.split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        cpus &= os.sched_getaffinity(0)
        if not cpus:
            return "unchanged"
        os.sched_setaffinity(0, cpus)
        return "cpus %s (NUMA node of GPU %s)" % (text, bdf)
    except (OSError, ValueError, AttributeError):
        return "unchanged"


def device_bench(capi, torch, local_rank, name, dim, res, streams, pcap, steps, warmup):
    """Device-resident throughput + one-stream latency of a (sub-)workload: `streams` = [stream][pose] -> (points, origin).
    Returns a dict for the JSON line.  Used for BASELINE configs[2] (cfg3) and configs[3] (cfg4)."""
    B, S = len(streams), len(streams[0])
    npts = np.array([[len(streams[b][s][0]) for s in range(S)] for b in range(B)], np.int64)
    total = int(npts.sum()) * 32
    pool = torch.empty(total, dtype=torch.uint8)
    hp = pool.numpy()
    offs = np.zeros((B, S), np.int64)
    o = 0
    for b in range(B):
        for s in range(S):
            raw = np.ascontiguousarray(streams[b][s][0]).view(np.uint8).reshape(-1)
            hp[o:o + raw.size] = raw
            offs[b, s] = o
            o += raw.size
    dev = pool.cuda()
    g = capi.GroundGridB200(dim, res, device=local_rank, n_slots=B, max_points=pcap, full_layers=False)
    for b in range(B):
        g.init_map(0.0, 0.0, 0.0, slot=b)
    slots = np.arange(B, dtype=np.int32)
    descs, ptrs, xy, Ts = [], [], [], []
    for s in range(S):
        descs.append(g.make_descs(list(range(B)), [int(npts[b, s]) for b in range(B)], [streams[b][s][1] for b in range(B)], [0.0] * B))
        ptrs.append([dev.data_ptr() + int(offs[b, s]) for b in range(B)])
        xy.append(np.tile(np.array([float(s), 0.0]), (B, 1)))
        Ts.append(np.tile(pose_T(s)[2].reshape(1, 12), (B, 1)))
    ext = torch.cuda.ExternalStream(g.stream, device=local_rank)
    t = [0]

    def step():
        s = pingpong(t[0], S)
        if t[0]:
            g.update_pose_batch(slots, xy[s], Ts[s])
        g.run_scans_device(descs[s], ptrs[s])
        t[0] += 1
        return s

    for _ in range(warmup):
        step()
    g.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    pts = 0
    e0.record(ext)
    g.fork_streams()
    for _ in range(steps):
        pts += int(npts[:, step()].sum())
    g.join_streams()
    e1.record(ext)
    g.synchronize()
    ms = e0.elapsed_time(e1)
    # one stream, scans strictly in sequence
    d1 = [g.make_descs([0], [int(npts[0, s])], [streams[0][s][1]], [0.0]) for s in range(S)]
    p1 = [[dev.data_ptr() + int(offs[0, s])] for s in range(S)]
    sl = np.array([0], np.int32)

    def one(tt):
        s = pingpong(tt, S)
        g.update_pose_batch(sl, xy[s][:1], Ts[s][:1])
        g.run_scans_device(d1[s], p1[s])

    for k in range(3):
        one(t[0] + k)
    g.synchronize()
    a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a0.record(ext)
    n1 = 20
    for k in range(n1):
        one(t[0] + 3 + k)
    a1.record(ext)
    g.synchronize()
    ms1 = a0.elapsed_time(a1) / n1
    P = float(npts.mean())
    N = g.n
    out = {"workload": name, "cells": N, "points_per_scan_mean": P, "streams": B, "steps": steps,
           "value": pts / (ms * 1e-3) / 1e6, "unit": UNIT, "ms_per_step": ms / steps,
           "single_stream_ms_per_scan": ms1, "single_stream_value": P / ms1 / 1e3,
           "roofline_path_frac": None, "algorithmic_bytes_per_scan": 45.0 * P + 72.0 * N * N + 16.0 * N * N}
    g.close()
    del dev
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--streams", type=int, default=444, help="independent streams (maps) per GPU (444 = 3 per SM: the spiral kernel runs one CTA per scan, three per SM)")
    ap.add_argument("--pool", type=int, default=8, help="distinct ego poses / clouds per stream")
    ap.add_argument("--cpu-scans", type=int, default=200, help="scans of the bounded CPU-baseline sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip cfg3 / cfg4 / drop-in latency / serialised per-kernel roofline / prior broadcast")
    ap.add_argument("--no-bind", action="store_true", help="do not bind the process to the NUMA node of its GPU")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write what the last of them computed "
                    "(labels, output order, ground / groundpatch of a fixed sample of streams) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of the GPU path (--impl ours)")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))

    if args.impl == "reference":
        reference_arm(args, rank, world)
        return

    B, S = args.streams, args.pool
    # ---- synthetic input, generated before CUDA is initialised (fork-based worker pool)
    procs = max(1, min(32, host_cores() // max(1, world)))
    streams = generate_streams(2000 + rank * B, B, S, procs)
    extras = not args.no_extras
    streams3 = streams4 = None
    if extras and rank == 0:
        streams3 = generate_streams(7000, 16, 2, procs, sensor="128")     # cfg3: 128 beams, ~240 k points
        streams4 = generate_streams(8000, 16, 2, procs, sensor="4x64")    # cfg4: four LiDARs, ~480 k points

    import torch
    import torch.distributed as dist

    from groundgrid_b200 import capi

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: groundgrid_b200 has no CPU fallback")
    torch.cuda.set_device(local_rank)
    affinity = "unchanged" if args.no_bind else bind_to_gpu_numa_node(torch, local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    npts = np.array([[len(streams[b][s][0]) for s in range(S)] for b in range(B)], np.int64)
    offs = np.zeros((B, S), np.int64)
    total = 0
    for b in range(B):
        for s in range(S):
            offs[b, s] = total
            total += int(npts[b, s]) * 32
    # device pool: every cloud of every stream; host pool (pinned, for the end-to-end leg): the first S_E2E poses only
    S_E2E = min(S, 4)
    hoffs = np.zeros((B, S_E2E), np.int64)
    htotal = 0
    for b in range(B):
        for s in range(S_E2E):
            hoffs[b, s] = htotal
            htotal += int(npts[b, s]) * 32
    dev_pool = torch.empty(total, dtype=torch.uint8, device="cuda")
    host_pool = torch.empty(htotal if not args.no_e2e else 1, dtype=torch.uint8)
    if not args.no_e2e:
        host_pool = host_pool.pin_memory()
    hp = host_pool.numpy()
    for b in range(B):
        for s in range(S):
            raw = np.ascontiguousarray(streams[b][s][0]).view(np.uint8).reshape(-1)
            if s < S_E2E and not args.no_e2e:
                hp[hoffs[b, s]:hoffs[b, s] + raw.size] = raw
            dev_pool[int(offs[b, s]):int(offs[b, s]) + raw.size] = torch.from_numpy(raw)
            if b > 0:                                        # only stream 0 is replayed on the CPU later
                streams[b][s] = (None, streams[b][s][1])     # (keeps the duplicate clouds of all other streams out of host memory)
    host_labels = torch.zeros((2, B, PCAP), dtype=torch.uint8).pin_memory()   # two sets: batches overlap in the e2e loop

    g = capi.GroundGridB200(DIM_M, RES, device=local_rank, n_slots=B, max_points=PCAP, full_layers=False)
    for b in range(B):
        g.init_map(0.0, 0.0, 0.0, slot=b)
    slots = np.arange(B, dtype=np.int32)
    descs, dev_ptrs, host_ptrs, lab_ptrs, xy, Ts = [], [], [], [], [], []
    for s in range(S):
        descs.append(g.make_descs(list(range(B)), [int(npts[b, s]) for b in range(B)], [streams[b][s][1] for b in range(B)], [0.0] * B))
        dev_ptrs.append([dev_pool.data_ptr() + int(offs[b, s]) for b in range(B)])
        host_ptrs.append([host_pool.data_ptr() + int(hoffs[b, min(s, S_E2E - 1)]) for b in range(B)])
        xy.append(np.tile(np.array([float(s), 0.0]), (B, 1)))
        Ts.append(np.tile(pose_T(s)[2].reshape(1, 12), (B, 1)))
    lab_ptrs = [[host_labels.data_ptr() + (q * B + b) * PCAP for b in range(B)] for q in range(2)]
    pts_per_pose = npts.sum(axis=0)

    ext = torch.cuda.ExternalStream(g.stream, device=local_rank)
    tstep = [0]

    def step_device(h=None):
        h = h or g
        s = pingpong(tstep[0], S)
        if tstep[0]:
            h.update_pose_batch(slots, xy[s], Ts[s])
        h.run_scans_device(descs[s], dev_ptrs[s])
        tstep[0] += 1
        return s

    in_flight = [None]
    last_label_set = [0]

    def step_e2e(overlap=True):
        """One scan of every stream through the host-buffer call.  overlap: the call is issued in its two halves
        (gg_filter_cloud_batch_begin / _wait), so the clouds of this step cross the bus while the kernels of the
        previous step finish; its labels are complete one step later."""
        s = pingpong(tstep[0], S_E2E)
        if tstep[0]:
            g.update_pose_batch(slots, xy[s], Ts[s])
        q = tstep[0] & 1
        if overlap:
            ticket = g.filter_cloud_batch_begin(descs[s], host_ptrs[s], lab_ptrs[q])
            if in_flight[0] is not None:
                g.filter_cloud_batch_wait(in_flight[0])
            in_flight[0] = ticket
        else:
            g.filter_cloud_batch_ptrs(descs[s], host_ptrs[s], lab_ptrs[q])
        last_label_set[0] = q
        tstep[0] += 1
        return s

    def drain_e2e():
        if in_flight[0] is not None:
            g.filter_cloud_batch_wait(in_flight[0])
            in_flight[0] = None

    def barrier():
        g.synchronize()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()

    def max_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def sum_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return float(t.item())

    # ---- device-resident throughput ("value")
    for _ in range(args.warmup):
        step_device()
    barrier()
    g.profile_enable(True)
    g.profile_read(reset=True)
    launches0 = g.kernel_launches
    clk = ClockSampler(local_rank)
    clk.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    pts_dev = 0
    e0.record(ext)
    g.fork_streams()          # every stream of the handle starts after e0 ...
    for _ in range(args.steps):
        pts_dev += int(pts_per_pose[step_device()])
    g.join_streams()          # ... and e1 is recorded after all of them have drained
    e1.record(ext)
    barrier()
    clocks = clk.stop()
    ms_dev = max_over_ranks(e0.elapsed_time(e1))
    launches = g.kernel_launches - launches0
    prof = g.profile_read(reset=True)
    g.profile_enable(False)
    value = sum_over_ranks(pts_dev) / (ms_dev * 1e-3) / 1e6
    if args.dump_outputs and rank == 0:
        dump_outputs(g, args.dump_outputs, npts[:, pingpong(tstep[0] - 1, S)])

    # ---- end to end through the host-buffer C-ABI call
    e2e = None
    if not args.no_e2e:
        n_e2e = max(10, args.steps // 2)
        for _ in range(max(3, args.warmup)):
            step_e2e(overlap=False)
        barrier()
        n_sync = max(3, n_e2e // 4)          # the plain synchronous call, for comparison
        t0 = time.perf_counter()
        pts_sync = 0
        tail_us = 0
        for _ in range(n_sync):
            pts_sync += int(pts_per_pose[step_e2e(overlap=False)])
            tr = g.last_batch_transfer()
            tail_us += tr[5] - tr[4]
        barrier()
        dt_sync = max_over_ranks(time.perf_counter() - t0)
        for _ in range(2):
            step_e2e()
        drain_e2e()
        barrier()
        t0 = time.perf_counter()
        pts_e2e = 0
        h2d = 0
        n_packed = n_raw = 0
        feed_us = pack_us = wait_us = idle_us = 0
        for _ in range(n_e2e):
            s = step_e2e()
            pts_e2e += int(pts_per_pose[s])
            tr = g.last_batch_transfer()
            n_packed += tr[0]
            n_raw += tr[1]
            h2d += tr[2] + tr[3]
            feed_us += tr[4]
            pack_us += tr[6]
            wait_us += tr[7]
            idle_us += tr[8]
        drain_e2e()
        barrier()
        dt = max_over_ranks(time.perf_counter() - t0)
        e2e = {"value": sum_over_ranks(pts_e2e) / dt / 1e6, "unit": UNIT, "h2d_bytes_per_step": int(sum_over_ranks(h2d) / n_e2e),
               "d2h_bytes_per_step": int(sum_over_ranks(int(pts_per_pose.max()))), "ms_per_step": dt / n_e2e * 1e3, "steps": n_e2e,
               "api": "gg_update_pose_batch + gg_filter_cloud_batch_begin/_wait (pinned host PointXYZIR clouds in, labels out; "
                      "the H2D of step t+1 overlaps the kernels and the label read-back of step t); the reference's filter_cloud also "
                      "returns the re-ordered 32 B/point cloud (GroundSegmentation.cpp:174-189), which this timed region does not copy back "
                      "(gg_get_output / gg_filter_cloud deliver it)",
               "synchronous_call": {"value": sum_over_ranks(pts_sync) / dt_sync / 1e6, "unit": UNIT, "ms_per_step": dt_sync / n_sync * 1e3,
                                    "ms_after_last_cloud_enqueued": tail_us / n_sync / 1e3, "api": "gg_filter_cloud_batch"},
               "host_pack_threads": max(0, g.host_pack_threads),
               "begin_call_ms": feed_us / n_e2e / 1e3,
               "begin_call_breakdown_ms": {"packer_threads_packing_sum": pack_us / n_e2e / 1e3,
                                           "packer_threads_waiting_for_slot_sum": wait_us / n_e2e / 1e3,
                                           "feeder_nothing_to_enqueue": idle_us / n_e2e / 1e3},
               "scans_repacked_14B": n_packed, "scans_raw_32B": n_raw,
               "pcie_bytes_per_point": round(h2d / max(1, pts_e2e), 2)}

    # ---- latency of ONE stream (configs[1] read literally: scan t+1 needs the prior of scan t)
    single = None
    dropin = None
    if rank == 0:
        d1 = [g.make_descs([0], [int(npts[0, s])], [streams[0][s][1]], [0.0]) for s in range(S)]
        p1 = [[dev_pool.data_ptr() + int(offs[0, s])] for s in range(S)]
        sl = np.array([0], np.int32)

        def one_scan(t):
            s = pingpong(t, S)
            g.update_pose_batch(sl, xy[s][:1], Ts[s][:1])
            g.run_scans_device(d1[s], p1[s])

        for t in range(5):
            one_scan(tstep[0] + t)
        g.synchronize()
        a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a0.record(ext)
        n_single = 50
        for t in range(n_single):
            one_scan(tstep[0] + 5 + t)
        a1.record(ext)
        g.synchronize()
        ms = a0.elapsed_time(a1) / n_single
        single = {"ms_per_scan": ms, "scans_per_s": 1e3 / ms, "value": P_mean_single(npts) / ms / 1e3, "unit": UNIT,
                  "note": "one stream, scans strictly in sequence (update + filter_cloud per scan), clouds resident in HBM"}
        if extras:
            # the literal drop-in call: GroundGrid::update + GroundSegmentation::filter_cloud through gg_update_pose +
            # gg_filter_cloud with PAGEABLE host clouds in and labels + the re-ordered output cloud back (what
            # points_callback does at GroundGridNodelet.cpp:196)
            clouds = [np.array(streams[0][s][0], copy=True) for s in range(S)]
            for t in range(3):
                s = pingpong(t, S)
                g.update_pose(float(s), 0.0, Ts[s][0], slot=0)
                g.filter_cloud(clouds[s], streams[0][s][1], 0.0, want_index=False, want_cloud=True)
            n_drop = 30
            t0 = time.perf_counter()
            for t in range(3, 3 + n_drop):
                s = pingpong(t, S)
                g.update_pose(float(s), 0.0, Ts[s][0], slot=0)
                g.filter_cloud(clouds[s], streams[0][s][1], 0.0, want_index=False, want_cloud=True)
            dt = (time.perf_counter() - t0) / n_drop
            t0 = time.perf_counter()
            for t in range(3 + n_drop, 3 + 2 * n_drop):
                s = pingpong(t, S)
                g.update_pose(float(s), 0.0, Ts[s][0], slot=0)
                g.filter_cloud(clouds[s], streams[0][s][1], 0.0)
            dt_lab = (time.perf_counter() - t0) / n_drop
            dropin = {"ms_per_scan": dt * 1e3, "scans_per_s": 1.0 / dt, "value": P_mean_single(npts) / dt / 1e6, "unit": UNIT,
                      "labels_only_ms_per_scan": dt_lab * 1e3,
                      "note": "wall clock of gg_update_pose + gg_filter_cloud per scan, one stream, pageable host cloud in (32 B/pt), labels and "
                              "the re-ordered output cloud (32 B/pt) back to pageable host memory; labels_only: without the output cloud"}

    # ---- per-kernel roofline of a SERIALISED step (one stream: no kernel waits for SMs held by another stream's kernel)
    P_mean = float(npts.mean())
    N2 = float(N_CELLS * N_CELLS)
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(peaks_path):
        peak, peak_src = float(json.load(open(peaks_path))["hbm_gbs"]), "of measured (MEASURED_PEAKS.json hbm_gbs)"
    else:
        peak, peak_src = 6650.0, "of fallback (B200_PROFILING.md 6.65 TB/s)"
    total_ms = sum(v[0] for v in prof.values()) or 1.0
    shares = {k: round(v[0] / total_ms, 4) for k, v in sorted(prof.items(), key=lambda kv: -kv[1][0])}
    serial = None
    if extras:
        old = os.environ.get("GG_STREAMS")
        os.environ["GG_STREAMS"] = "1"
        g1 = capi.GroundGridB200(DIM_M, RES, device=local_rank, n_slots=B, max_points=PCAP, full_layers=False)
        if old is None:
            del os.environ["GG_STREAMS"]
        else:
            os.environ["GG_STREAMS"] = old
        for b in range(B):
            g1.init_map(0.0, 0.0, 0.0, slot=b)
        t_keep = tstep[0]
        tstep[0] = 0
        for _ in range(3):
            step_device(g1)
        g1.synchronize()
        g1.profile_enable(True)
        g1.profile_read(reset=True)
        n_ser = 5
        for _ in range(n_ser):
            step_device(g1)
        serial = g1.profile_read(reset=True)
        g1.profile_enable(False)
        g1.close()
        tstep[0] = t_keep
    traffic_tab = {}
    tpath = os.path.join(ROOT, "profiles", "r02_traffic.json")
    if os.path.exists(tpath):                            # DRAM bytes per scan of every kernel from the committed ncu capture
        traffic_tab = json.load(open(tpath)).get("bytes_per_scan", {})
    roofline = None
    src_prof = serial if serial else prof
    scans_per_launch = float(B) if serial else B / max(1, g.n_streams)
    if src_prof:
        per_kernel = {}
        for kname, (kms, kn) in src_prof.items():
            if not kn:
                continue
            ab = algorithmic_bytes(kname, P_mean, N2) * scans_per_launch
            us = kms / kn * 1e3
            per_kernel[kname] = {"avg_launch_us": round(us, 1), "algorithmic_bytes_per_launch": ab, "achieved_gbs": round(ab / (us * 1e-6) / 1e9, 1),
                                 "frac": round(ab / (us * 1e-6) / 1e9 / peak, 4),
                                 "traffic": (traffic_tab[kname] * scans_per_launch) if kname in traffic_tab else None}
        dom = max(src_prof.items(), key=lambda kv: kv[1][0])[0]
        d = per_kernel[dom]
        roofline = {"bound": "hbm", "kernel": dom, "achieved": d["achieved_gbs"], "peak": peak, "unit": "GB/s", "frac": d["frac"],
                    "traffic": d["traffic"], "traffic_source": "profiles/r02_traffic.json (ncu --set full, per scan, scaled to the scans of one launch)",
                    "peak_source": peak_src, "scans_per_launch": scans_per_launch, "avg_launch_us": d["avg_launch_us"],
                    "algorithmic_bytes_per_launch": d["algorithmic_bytes_per_launch"],
                    "how": ("CUDA events around every launch of an extra SERIALISED pass (GG_STREAMS=1 handle, %d steps of %d scans): "
                            "no launch waits for SMs held by another stream's kernel" % (5, B)) if serial else
                           "CUDA events around every launch inside the timed region (kernels of 4 stream groups overlap)",
                    "per_kernel": per_kernel, "kernel_time_shares_live": shares,
                    "kernel_avg_launch_us_live": {k: round(v[0] / v[1] * 1e3, 1) for k, v in prof.items() if v[1]}}
    path_bytes = (45.0 * P_mean + 72.0 * N2 + 16.0 * N2) * B     # + roll every step
    path_gbs = path_bytes / (ms_dev / args.steps * 1e-3) / 1e9
    roofline_path = {"bound": "hbm", "algorithmic_bytes_per_step": path_bytes, "achieved": path_gbs, "peak": peak, "unit": "GB/s",
                     "frac": path_gbs / peak, "formula": "(45 P + 72 N^2 + 16 N^2 roll) x streams / step time",
                     "fused_lower_bound": {"formula": "(17 P + 20 N^2) x streams (points in, labels out, G/C in+out, E in; SURVEY 8d)",
                                           "bytes_per_step": (17.0 * P_mean + 20.0 * N2) * B,
                                           "frac": (17.0 * P_mean + 20.0 * N2) * B / (ms_dev / args.steps * 1e-3) / 1e9 / peak}}

    # ---- BASELINE configs[2] and [3] on this GPU (rank 0)
    cfg3 = cfg4 = None
    if extras and rank == 0:
        cfg3 = device_bench(capi, torch, local_rank, "dense 128-beam synthetic scans (~240k pts), 600x600 @ 0.2 m (BASELINE configs[2]), 16 streams",
                            120.0, 0.2, streams3, SENSORS["128"][1], 10, 3)
        cfg4 = device_bench(capi, torch, local_rank, "4-LiDAR fused clouds (~480k pts/frame), 364x364 @ 0.33 m (BASELINE configs[3]), 16 streams",
                            120.0, 0.33, streams4, SENSORS["4x64"][1], 10, 3)
        for c in (cfg3, cfg4):
            c["roofline_path_frac"] = c["algorithmic_bytes_per_scan"] * c["streams"] / (c["ms_per_step"] * 1e-3) / 1e9 / peak

    # ---- the one exchange of the path: NCCL broadcast of the rolling terrain prior (scans sharing one ego frame)
    prior_bcast = None
    if extras and world > 1:
        from groundgrid_b200 import prior as prior_mod

        barrier()
        src_slot = 0
        prior_mod.broadcast_prior(g, src=0, slot=src_slot)       # functional pass: every rank now holds rank 0's prior of stream 0
        pt = prior_mod.prior_tensor(g, src_slot)
        torch.cuda.synchronize()
        b0, b1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        n_b = 50
        b0.record()
        for _ in range(n_b):
            dist.broadcast(pt, src=0)
        b1.record()
        torch.cuda.synchronize()
        us = max_over_ranks(b0.elapsed_time(b1) / n_b * 1e3)
        # every rank labels rank 0's next cloud of stream 0 against the received prior; the receivers check against the CPU
        s_chk = pingpong(tstep[0], S)
        n_chk = int(npts[0, s_chk])
        cloud_t = torch.zeros(PCAP * 32, dtype=torch.uint8, device="cuda")
        meta = torch.zeros(4, dtype=torch.float64, device="cuda")
        if rank == 0:
            cloud_t[:n_chk * 32] = dev_pool[int(offs[0, s_chk]):int(offs[0, s_chk]) + n_chk * 32]
            meta[:] = torch.tensor([n_chk] + [float(v) for v in streams[0][s_chk][1]], dtype=torch.float64)
        dist.broadcast(cloud_t, src=0)
        dist.broadcast(meta, src=0)
        n_chk = int(meta[0].item())
        org = np.array([meta[1].item(), meta[2].item(), meta[3].item()], np.float32)
        Gp, Cp = g.layer("ground", src_slot), g.layer("groundpatch", src_slot)
        posxy = g.position(src_slot)
        dchk = g.make_descs([src_slot], [n_chk], [org], [0.0])
        g.run_scans_device(dchk, [cloud_t.data_ptr()])
        lab = g.download_labels(n_chk, src_slot)
        g.synchronize()
        ok = 1.0
        checked_with = "none"
        if rank != 0 and not args.no_cpu_baseline:
            from oracle import Oracle

            o = Oracle(DIM_M, RES)
            o.init_map(float(posxy[0]), float(posxy[1]), 0.0)
            o.set_layer("ground", Gp)
            o.set_layer("groundpatch", Cp)
            from groundgrid_b200 import synth as _synth

            pts_np = np.frombuffer(cloud_t[:n_chk * 32].cpu().numpy().tobytes(), dtype=_synth.POINT_DTYPE)
            want = o.filter_cloud(pts_np, org, 0.0, threads=1)[0]
            ok = 1.0 if np.array_equal(lab, want) else 0.0
            checked_with = "oracle port on the receiving ranks"
        all_ok = sum_over_ranks(ok) == world
        lab_sum = torch.tensor([float(lab.astype(np.int64).sum())], dtype=torch.float64, device="cuda")
        mx, mn = lab_sum.clone(), lab_sum.clone()
        dist.all_reduce(mx, op=dist.ReduceOp.MAX)
        dist.all_reduce(mn, op=dist.ReduceOp.MIN)
        prior_bcast = {"us_per_broadcast": us, "bytes": int(2 * N2 * 4), "gbs": 2 * N2 * 4 / (us * 1e-6) / 1e9, "ranks": world,
                       "what": "dist.broadcast (NCCL) of ground||groundpatch of one map, in place on the handles' device memory, max over ranks",
                       "labels_of_all_ranks_identical": bool(mx.item() == mn.item()), "labels_match_cpu_on_receivers": bool(all_ok),
                       "checked_with": "none (--no-cpu-baseline)" if args.no_cpu_baseline else
                                       "oracle port on every receiving rank: prior (ground, groundpatch, position) read back from the GPU, same cloud"}

    # ---- CPU baseline: the reference's CPU path replaying stream 0 of rank 0 on this host (bounded sample)
    cpu = None
    if rank == 0 and not args.no_cpu_baseline:
        n_cpu = args.cpu_scans
        labs = {}
        # the GPU stream 0 went through every step above; replay the same number of scans only if that is affordable
        spent1, pts1, kind = run_cpu_stream(streams[0], n_cpu, 1)
        spent8, pts8, _ = run_cpu_stream(streams[0], n_cpu, 8)
        v1, v8 = pts1 / spent1 / 1e6, pts8 / spent8 / 1e6
        # label check of the GPU against the CPU on a fresh map: two scans of stream 0 through the drop-in call
        chk = capi.GroundGridB200(DIM_M, RES, device=local_rank, n_slots=1, max_points=PCAP, full_layers=False)
        chk.init_map(0.0, 0.0, 0.0)
        impl, _ = make_cpu_impl(1)
        impl.init_map(0.0, 0.0, 0.0)
        match = True
        for t in range(3):
            s = pingpong(t, S)
            if t:
                chk.update_pose(float(s), 0.0, pose_T(s)[2])
            got = chk.filter_cloud(streams[0][s][0], streams[0][s][1], 0.0)
            want = cpu_scan(impl, kind, t, s, streams[0][s][0], streams[0][s][1], 1)
            match = match and bool(np.array_equal(got, want))
        chk.close()
        best, cores = (v1, 1) if v1 >= v8 else (v8, 8)
        what = ("oracle/_ref = the unmodified reference sources on CPU stand-ins" if kind == "reference" else "oracle port of the reference")
        cpu = {"value": best, "unit": UNIT, "cores": cores, "kind": kind,
               "sample": f"stream 0, {n_cpu} consecutive scans (update + filter_cloud), {what}; "
                         f"thread_count=1: {v1:.2f} Mpts/s, reference threading as shipped (8 insert + 4 detect threads): {v8:.2f} Mpts/s; "
                         f"host has {host_cores()} cores",
               "scans_per_s": best * 1e6 / P_mean, "labels_match_gpu": match}

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_dev / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32/f64", "data": "synthetic",
            "config": {"workload": f"{B} independent SemanticKITTI-shaped synthetic 64-beam streams per GPU, ~120k pts/scan, "
                                   f"{N_CELLS}x{N_CELLS} @ {RES} m grid (BASELINE configs[1], batched); step = one scan of every stream: "
                                   "GroundGrid::update (roll) + GroundSegmentation::filter_cloud",
                       "streams_per_gpu": B, "poses_per_stream": S, "points_per_scan_mean": P_mean, "cells": N_CELLS,
                       "parallelism": f"scans sharded one-stream-set-per-GPU x{world}, no data-path collective",
                       "l2": f"inputs larger than L2: {B * P_mean * 32 / 1e6:.0f} MB of clouds + {B * 6 * N2 * 4 / 1e6:.0f} MB of layers per step vs 126 MB L2",
                       "layers": "live layers only (dead layers of SURVEY f2 off)", "cuda_streams": g.n_streams,
                       "host_affinity": affinity},
            "e2e": e2e, "gpu_launches": int(launches), "clocks": clocks, "roofline": roofline, "roofline_path": roofline_path,
            "cpu_baseline": cpu, "scans_per_s": value * 1e6 / P_mean, "single_stream": single, "drop_in_call": dropin,
            "cfg3_128beam_600": cfg3, "cfg4_4lidar_364": cfg4, "prior_broadcast": prior_bcast,
        }
        print(json.dumps(line), flush=True)
    barrier()
    g.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
