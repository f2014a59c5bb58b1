#!/usr/bin/env python
"""bench.py — LiODOM hot path (extract + register) on B200: scans/s, roofline, CPU baseline.

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --gpus N --steps K ...   # restated CPU path (oracle port)

A step = one pass of the hot path (ring split -> curvature/edge selection -> predict ->
2 x {voxel-hash 5-NN association + line gate, on-device LM} -> window update + hash rebuild)
over one batch of `lanes` independent HDL-64-shaped synthetic scans (config C1 of
BASELINE.json, launch/liodom.launch params).  `value` is scans/s with the scans resident in
HBM; `e2e` is the same metric through the C-ABI call with pinned HOST buffers, H2D copy of the
scans and D2H read of the poses inside the timed region.  Under torchrun every rank runs its
own lanes (no data-path collective; weak scaling) and rank 0 prints one JSON line.
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "hdl64_scans_per_sec_extract_plus_register"
UNIT = "scans/s"
N_SEEDS = 8          # distinct synthetic sequences (seeds 1000..1007, SURVEY.md §8(d) C5)
BYTES_PER_POINT = 16


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, help="timed steps (default 20)")
    ap.add_argument("--warmup", type=int, help="warm-up steps (default 3)")
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--lanes", type=int, default=int(os.environ.get("LIODOM_BENCH_LANES", "128")),
                    help="independent sequences per GPU processed by one step")
    ap.add_argument("--sensor", default="hdl64")
    ap.add_argument("--config", default="c1", choices=["c1", "c2", "c3", "c4"],
                    help="c1: the headline workload (launch/liodom.launch); c2 / c3: the other BASELINE.json shapes "
                         "(OS1-128 organised clouds; scan_regions/edges_per_region doubled, prev_frames=20), for profiles/ only; "
                         "c4: liodom_mapping_node's map build over a 4000-frame loop (Map::updateMap / getLocalMap / getMap)")
    ap.add_argument("--mode", default="sequences", choices=["sequences", "sharded"],
                    help="sequences: independent sequences per GPU (the headline); sharded: ONE 1M-point scan stream, ring-sharded "
                         "extraction + edge-sharded registration across the GPUs with a 29-double NCCL all-reduce per LM evaluation")
    ap.add_argument("--frames", type=int, default=4000, help="frames of the c4 loop")
    ap.add_argument("--no-sharded-block", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-stage-pass", action="store_true")
    ap.add_argument("--no-single-stream", action="store_true")
    ap.add_argument("--no-xyz12", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last timed step returned (rank 0's lanes) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.config == "c4" and (args.steps is not None or args.warmup is not None):
        ap.error("--config c4 times --frames map updates after one warm-up frame; it takes no --steps / --warmup")
    args.steps = 20 if args.steps is None else args.steps
    args.warmup = 3 if args.warmup is None else args.warmup
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "b200" or args.config == "c4" or args.mode != "sequences"):
        ap.error("--dump-outputs applies to the default path (--impl b200 --mode sequences, config c1 / c2 / c3)")
    return args


def dist_env():
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    return rank, world, local


def make_sequences(sensor, rank, nseq, nframes, world=1):
    """This rank's shard of the job's world*nseq independent sequences (float32 [n,4] scans)."""
    from liodom_b200 import sharding, synth
    out = []
    for sid in sharding.shard_sequences(world * nseq, world, rank):
        scans, _ = synth.sequence(sensor, sharding.seed_of(sid), nframes)
        out.append(scans)
    return out


class ClockSampler:
    """nvidia-smi clocks/throttle reasons DURING the timed region (B200_PROFILING.md).  Started before the
    pre-roll (the first sample takes a while) and polled every 20 ms; stop() keeps the samples whose
    timestamps fall inside the marked window."""
    Q = ("timestamp,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.lines = []
        self.proc = None
        self.t0 = self.t1 = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except OSError:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.lines.append((time.time(), ln.strip()))

    def mark_begin(self):
        self.t0 = time.time()

    def mark_end(self):
        self.t1 = time.time()

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"], "samples": 0}
        time.sleep(0.05)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]

        def digest(rows):
            sm, mx, reasons = [], [], set()
            for _, ln in rows:
                f = [x.strip() for x in ln.split(",")]
                if len(f) < 8:
                    continue
                try:
                    sm.append(float(f[1]))
                    mx.append(float(f[2]))
                except ValueError:
                    continue
                for k, nm in enumerate(names):
                    if f[4 + k].lower().startswith("active"):
                        reasons.add(nm)
            return sm, mx, reasons

        # a sample is a snapshot taken shortly before its line arrives: keep a margin on both sides
        inside = [r for r in self.lines if self.t0 is not None and self.t0 - 0.03 <= r[0] <= (self.t1 or r[0]) + 0.03]
        sm, mx, reasons = digest(inside)
        sm_all, mx_all, reasons_all = digest(self.lines)
        return {"sm_mhz": float(np.median(sm)) if sm else (float(np.median(sm_all)) if sm_all else None),
                "sm_max_mhz": max(mx_all) if mx_all else None,
                "reasons": sorted(reasons), "samples": len(sm),
                "samples_whole_run": len(sm_all), "sm_mhz_whole_run": float(np.median(sm_all)) if sm_all else None,
                "reasons_whole_run": sorted(reasons_all), "period_ms": 20}


def bind_to_gpu_numa_node(local):
    """Run this rank (and hence first-touch its pinned staging buffers) on the CPUs next to its GPU, so that
    the H2D transfers of the ranks of a node do not all cross the same socket link."""
    try:
        import torch
        prop = torch.cuda.get_device_properties(local)
        bdf = "%04x:%02x:%02x.0" % (prop.pci_domain_id, prop.pci_bus_id, prop.pci_device_id)
        cpus = open("/sys/bus/pci/devices/%s/local_cpulist" % bdf).read().strip()
        ids = set()
        for part in cpus.split(","):
            a, _, b = part.partition("-")
            ids.update(range(int(a), int(b or a) + 1))
        ids &= os.sched_getaffinity(0)
        if ids:
            os.sched_setaffinity(0, ids)
        return "%s cpus %s" % (bdf, cpus)
    except Exception as e:   # best effort: containers may hide sysfs or the affinity call
        return "unbound (%s)" % e


def pose_err(A, B):
    dt = float(np.linalg.norm(A[:3, 3] - B[:3, 3]))
    dR = A[:3, :3] @ B[:3, :3].T
    v = np.array([dR[2, 1] - dR[1, 2], dR[0, 2] - dR[2, 0], dR[1, 0] - dR[0, 1]])
    return dt, float(np.arctan2(0.5 * np.linalg.norm(v), (np.trace(dR) - 1.0) / 2.0))


def run_b200(args):
    import torch
    import torch.distributed as dist
    from liodom_b200 import api

    rank, world, local = dist_env()
    numa = bind_to_gpu_numa_node(local)
    sys.stderr.write("[bench] rank %d: %s\n" % (rank, numa))
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    sampler = ClockSampler(local)
    sampler.start()
    B, K, W = args.lanes, args.steps, args.warmup
    nseq = min(B, N_SEEDS)
    t0 = time.time()
    width = height = 0
    kw_cfg = {}
    workload = ("C1: HDL-64-shaped ray-cast urban sequences (~118k pts/scan), launch/liodom.launch params "
                "(scan_regions=8, edges_per_region=10, prev_frames=15, range 3-75 m), extract+register")
    if args.config == "c2":
        from liodom_b200 import synth
        args.sensor = "os1_128"
        width, height = synth.sensor_shape("os1_128")
        kw_cfg = dict(lidar_type=1, scan_lines=128)
        workload = ("C2: OS1-128-shaped organised clouds (128 x 2048 slots), launch/liodom_ouster.launch params with "
                    "scan_lines=128, extract+register")
    elif args.config == "c3":
        kw_cfg = dict(scan_regions=16, edges_per_region=20, prev_frames=20)
        workload = ("C3: C1 scans with scan_regions=16, edges_per_region=20, prev_frames=20 (large local map), extract+register")
    max_points = 131072 if args.sensor == "hdl64" else (262144 if args.sensor == "os1_128" else 1 << 20)
    kw = dict(prev_frames=15, max_points=max_points)   # launch/liodom.launch:17-31
    kw.update(kw_cfg)
    # Pre-roll: prev_frames + 1 untimed steps before the warm-up, so that the sliding window is FULL (steady state:
    # one frame enters, one is evicted, M = prev_frames * E map points) in every warm-up and timed step.
    P = kw["prev_frames"] + 1
    nframes = P + W + K
    seqs = make_sequences(args.sensor, rank, nseq, nframes, world)
    gen_s = time.time() - t0
    npts = np.array([[len(seqs[s][f]) for f in range(nframes)] for s in range(nseq)])

    # inputs resident in HBM: one tensor per (lane, frame).  Lanes that replay the same synthetic sequence
    # still get their own copy, so that no lane finds its scan in L2 because another lane just read it.
    dev_scans = [[torch.from_numpy(seqs[l % nseq][f]).to(dev) for f in range(nframes)] for l in range(B)]
    # pinned host buffers for the end-to-end leg (warm-up and timed frames only; the pre-roll is fed from HBM):
    # the B scans of a step back to back (what a batching front-end hands over), so that the library can move a
    # step over PCIe as one copy
    host_steps, host_ptrs = {}, {}
    for f in range(P, nframes):
        cnt = [int(npts[l % nseq][f]) for l in range(B)]
        buf = torch.empty((sum(cnt), 4), dtype=torch.float32).pin_memory()
        off, ptrs = 0, []
        for l in range(B):
            buf[off:off + cnt[l]] = torch.from_numpy(seqs[l % nseq][f])
            ptrs.append(buf.data_ptr() + off * BYTES_PER_POINT)
            off += cnt[l]
        host_steps[f] = buf
        host_ptrs[f] = ptrs
    torch.cuda.synchronize()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    from liodom_b200.sharding import max_over_ranks

    # ---------------- device-resident leg (value) -------------------------------------------
    ctx = api.Context(batch=B, device=local, **kw)
    stream = torch.cuda.ExternalStream(ctx.stream, device=dev)

    def step_dev(c, f):
        ptrs = [dev_scans[l][f].data_ptr() for l in range(B)]
        cnts = [int(npts[l % nseq][f]) for l in range(B)]
        c.scan_batch_ptrs(ptrs, cnts, BYTES_PER_POINT, width=width, height=height, on_device=True)

    for f in range(P + W):
        step_dev(ctx, f)
    ctx.sync()
    barrier()
    launches0 = ctx.launch_count
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sampler.mark_begin()
    ev0.record(stream)
    for f in range(P + W, nframes):
        step_dev(ctx, f)
    ev1.record(stream)
    ctx.sync()
    sampler.mark_end()
    barrier()
    ms_total = max_over_ranks(ev0.elapsed_time(ev1))
    launches = ctx.launch_count - launches0
    poses_dev, nedges = ctx.results()
    value = world * B * K / (ms_total * 1e-3)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, ctx, poses_dev, nedges)

    # ---------------- per-stage pass (roofline of the dominant kernel) ----------------------
    roof = None
    stages = None
    if not args.no_stage_pass:
        for l in range(B):
            ctx.reset(l)
        E_sum = M_sum = Ev_sum = pass_sum = 0.0
        nd = 0
        for f in range(nframes):
            if f == P + W:
                ctx.stage_timing(True)
            step_dev(ctx, f)
            if f >= P + W:
                ctx.sync()
                for l in range(min(B, nseq)):
                    d = ctx.scan_diag(l)
                    E_sum += d.n_edges
                    M_sum += 0.5 * (d.n_map[0] + d.n_map[1])
                    Ev_sum += 0.5 * (d.n_matches[0] + d.n_matches[1])
                    pass_sum += 0.5 * sum(d.solve[i].jac_evals + d.solve[i].cost_evals for i in range(2))
                    nd += 1
        ms, calls = ctx.stage_times()
        ctx.stage_timing(False)
        per_call = ms / max(calls, 1)
        E, M, Ev, passes = E_sum / nd, M_sum / nd, Ev_sum / nd, pass_sum / nd
        Npts = float(npts[:, P + W:].mean())
        # algorithmic bytes per launch (SURVEY.md §8(d)), all lanes of one step
        alg = {
            "split": B * (BYTES_PER_POINT * Npts * 2),                     # read scan, write ring-major copy
            "extract": B * (BYTES_PER_POINT * Npts + BYTES_PER_POINT * E),
            "associate": B * (16 * E + 16 * M + 56 * E),
            "solve": B * (passes * 40 * E + 224),
            "window+hash": B * (16 * E + 2 * 16 * M),
        }
        groups = {"split": per_call[0], "extract": per_call[1], "associate": 0.5 * (per_call[2] + per_call[4]),
                  "solve": 0.5 * (per_call[3] + per_call[5]), "window+hash": per_call[6]}
        share = {"split": per_call[0], "extract": per_call[1], "associate": per_call[2] + per_call[4],
                 "solve": per_call[3] + per_call[5], "window+hash": per_call[6]}
        tot = sum(share.values())
        dom = max(share, key=share.get)
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except (OSError, ValueError):
            pass
        peak = float(peaks.get("hbm_gbs", 6650.0))
        achieved = alg[dom] / (groups[dom] * 1e-3) / 1e9
        traffic = traffic_m = traffic_src = None
        try:   # measured DRAM bytes per launch of this kernel from the committed ncu capture (same lane count)
            tr = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json")))
            ent = tr.get("k_" + dom, {}).get(str(B), {})
            traffic, traffic_m, traffic_src = ent.get("dram_bytes_per_launch"), ent.get("map_points_per_lane"), ent.get("capture")
        except (OSError, ValueError):
            pass
        roof = {"bound": "hbm", "kernel": dom, "achieved": round(achieved, 2), "peak": peak, "unit": "GB/s",
                "frac": round(achieved / peak, 5), "traffic": traffic,
                "traffic_source": {"capture": traffic_src, "map_points_per_lane_in_capture": traffic_m, "map_points_per_lane_in_this_run": round(M, 1)},
                "peak_source": "MEASURED_PEAKS.json hbm_gbs (burst copy)" if "hbm_gbs" in peaks else "fallback 6650 GB/s",
                "algorithmic_bytes_per_launch": int(alg[dom]), "launch_ms": round(groups[dom], 4),
                "whole_step": {"algorithmic_bytes": int(sum(alg[k] * (2 if k in ("associate", "solve") else 1) for k in alg)),
                               "gbps": round(sum(alg[k] * (2 if k in ("associate", "solve") else 1) for k in alg) / (ms_total / K * 1e-3) / 1e9, 1)}}
        stages = {"ms_per_step": {k: round(v, 4) for k, v in share.items()},
                  "share": {k: round(v / tot, 4) for k, v in share.items()},
                  "gbps": {k: round(alg[k] / (groups[k] * 1e-3) / 1e9, 2) for k in alg},
                  "per_scan": {"points": round(Npts, 1), "edges": round(E, 1), "map_points": round(M, 1),
                               "matches": round(Ev, 1), "lm_passes_per_solve": round(passes, 2)}}
    ctx.close()

    # ---------------- end-to-end leg (host buffers through the C ABI) -----------------------
    ctx = api.Context(batch=B, device=local, **kw)
    stream = torch.cuda.ExternalStream(ctx.stream, device=dev)

    def enqueue_e2e(f):
        cnts = [int(npts[l % nseq][f]) for l in range(B)]
        ctx.scan_batch_ptrs(host_ptrs[f], cnts, BYTES_PER_POINT, width=width, height=height, on_device=False)

    for f in range(P):          # pre-roll from HBM (untimed): fills the window
        step_dev(ctx, f)
    ctx.results()
    for f in range(P, P + W):   # warm-up through the host path
        enqueue_e2e(f)
        ctx.results()
    barrier()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record(stream)
    t_wall = time.perf_counter()
    h2d = d2h = 0
    # two scans in flight: the H2D copy of step k+1 overlaps the kernels of step k; every step's
    # poses are read back on the host inside the timed region
    for f in range(P + W, nframes):
        enqueue_e2e(f)
        if f > P + W:
            poses_e2e, ne = ctx.results(age=1)
            d2h += poses_e2e.nbytes + ne.nbytes
        h2d += sum(int(npts[l % nseq][f]) for l in range(B)) * BYTES_PER_POINT
    poses_e2e, ne = ctx.results(age=0)
    d2h += poses_e2e.nbytes + ne.nbytes
    ev1.record(stream)
    ctx.sync()
    barrier()
    wall_ms = (time.perf_counter() - t_wall) * 1e3
    e2e_ms = max_over_ranks(max(ev0.elapsed_time(ev1), wall_ms))
    e2e_value = world * B * K / (e2e_ms * 1e-3)
    # what the PCIe link alone would allow: the same pinned step buffers copied back to back, nothing else running
    probe_frames = list(range(P + W, P + W + min(K, 8)))
    probe = torch.empty((max(len(host_steps[f]) for f in probe_frames), 4), dtype=torch.float32, device=dev)
    pe0, pe1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    pe0.record()
    for f in probe_frames:
        probe[:len(host_steps[f])].copy_(host_steps[f], non_blocking=True)
    pe1.record()
    torch.cuda.synchronize()
    h2d_alone_gbps = sum(host_steps[f].numel() * 4 for f in probe_frames) / (pe0.elapsed_time(pe1) * 1e-3) / 1e9
    h2d_in_run_gbps = h2d / (e2e_ms * 1e-3) / 1e9
    # the two legs must agree on the answer: same scans, same start state
    same = bool(np.array_equal(poses_e2e, poses_dev))
    ctx.close()
    clocks = sampler.stop()

    # ---------------- end to end with 12-byte points (x, y, z only) --------------------------------------------
    # The odometry never reads intensity (include/liodom/factors.hpp:71-105; it is only carried into the published
    # edge cloud), and the e2e leg is bound by the PCIe transfer of the scans: a front-end that hands over xyz
    # records moves 25 % fewer bytes.  Same frames, same C ABI call (liodom_scan_batch_layout: point_step 12, no
    # intensity field); poses must equal the 16-byte leg's.
    xyz12 = None
    if args.config == "c1" and not args.no_xyz12:
        lay = api.CloudLayout(12, 0, 0, 4, 8, -1, 0)
        h12, p12 = {}, {}
        for f in range(P, nframes):
            cnt = [int(npts[l % nseq][f]) for l in range(B)]
            buf = torch.empty((sum(cnt), 3), dtype=torch.float32).pin_memory()
            off, ptrs = 0, []
            for l in range(B):
                buf[off:off + cnt[l]] = torch.from_numpy(seqs[l % nseq][f][:, :3])
                ptrs.append(buf.data_ptr() + off * 12)
                off += cnt[l]
            h12[f], p12[f] = buf, ptrs
        ctx = api.Context(batch=B, device=local, **kw)
        stream = torch.cuda.ExternalStream(ctx.stream, device=dev)
        for f in range(P):
            step_dev(ctx, f)
        ctx.results()
        for f in range(P, P + W):
            ctx.scan_batch_layout_ptrs(p12[f], [int(npts[l % nseq][f]) for l in range(B)], lay)
            ctx.results()
        barrier()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record(stream)
        t_wall = time.perf_counter()
        for f in range(P + W, nframes):
            ctx.scan_batch_layout_ptrs(p12[f], [int(npts[l % nseq][f]) for l in range(B)], lay)
            if f > P + W:
                ctx.results(age=1)
        poses12, _ = ctx.results(age=0)
        ev1.record(stream)
        ctx.sync()
        barrier()
        ms12 = max_over_ranks(max(ev0.elapsed_time(ev1), (time.perf_counter() - t_wall) * 1e3))
        xyz12 = {"value": round(world * B * K / (ms12 * 1e-3), 2), "unit": UNIT, "ms_per_step": round(ms12 / K, 4),
                 "h2d_bytes_per_step": int(h2d / K * 12 / 16), "same_poses_as_16_byte_leg": bool(np.array_equal(poses12, poses_e2e)),
                 "layout": "point_step 12: float32 x, y, z (no intensity), liodom_scan_batch_layout"}
        ctx.close()
        del h12, p12

    # ---------------- what the host fabric gives when every rank copies at once -------------------------------
    barrier()
    pe0, pe1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    pe0.record()
    for f in probe_frames:
        probe[:len(host_steps[f])].copy_(host_steps[f], non_blocking=True)
    pe1.record()
    torch.cuda.synchronize()
    h2d_concurrent_gbps = sum(host_steps[f].numel() * 4 for f in probe_frames) / (max_over_ranks(pe0.elapsed_time(pe1)) * 1e-3) / 1e9

    # ---------------- the drop-in facade, single stream (what src/liodom_node.cc drives) -----------------------
    facade = None
    if rank == 0 and world == 1 and not args.no_single_stream:
        try:
            from liodom_b200 import host_api
            nfac = len(seqs[0])
            fk = dict(prev_frames=kw["prev_frames"], width=width, height=height)
            host_api.run_sequence(seqs[0][:3], lockstep=False, **fk)   # warm-up: contexts, first kernels
            skip = min(kw["prev_frames"] + 1, nfac // 2)               # frames while the window is still filling

            def marks(lockstep):
                # per-frame wall-clock marks taken inside the harness (cloud pushed, pose out); the reference's own Stats
                # keeps whole milliseconds.  Start-up and allocation of the call lie before the first mark used.
                _, _, produced = host_api.run_sequence(seqs[0][:nfac], lockstep=lockstep, **fk)
                push, pose = host_api.last_run_times(nfac)
                return produced, push, pose
            produced, _, pose_free = marks(False)
            _, push_lock, pose_lock = marks(True)
            per = float(pose_free[-1] - pose_free[skip]) / max(nfac - 1 - skip, 1)   # ms between poses, free running
            facade = {"value": round(1e3 / per, 1), "unit": UNIT, "ms_per_scan": round(per, 3),
                      "latency_ms_per_scan_lockstep": round(float((pose_lock - push_lock)[skip:].mean()), 3),
                      "frames": [int(skip), int(produced)],
                      "note": "liodom::FeatureExtractor / LaserOdometer worker threads over the SharedData queues, pageable host clouds in, "
                              "poses out; wall-clock marks inside the harness over the full-window frames: ms between consecutive poses with "
                              "all clouds queued (the two workers overlap), and push -> pose latency when the next cloud is pushed only "
                              "after the previous pose.  The workers wait on the queues (condition variable, <= 2 ms) where the reference "
                              "sleeps 2 ms per turn (src/feature_extractor.cc:80, src/laser_odometry.cc:270)"}
        except Exception as e:   # the facade is optional for the headline
            facade = {"error": str(e)}

    # ---------------- point-sharded 1M-point stream (BASELINE config 5, second half; short, outside the headline) -----
    sharded = None
    if not args.no_sharded_block and args.config == "c1":
        del dev_scans, host_steps
        torch.cuda.empty_cache()
        sharded = point_sharded_run(api, torch, dist, rank, world, local, nframes=7, warm=3)
        sharded["note"] = "7 frames (3 warm-up): the 15-frame window is still filling; `bench.py --mode sharded` runs the full-window version"

    # ---------------- single stream (the reference's own shape: one sequence through liodom_node) -------------
    single = None
    if rank == 0 and not args.no_single_stream:
        single = single_stream_block(api, torch, dev, local, seqs[0], npts[0], kw, P, W, K, width, height)

    # ---------------- parity of the benchmarked run against the oracle + CPU baseline ------------------------
    # The oracle replays the same sequences on the host (outside every timed region): its wall time is the CPU
    # baseline (rank 0, N=1), its final poses are compared with the final poses of the lanes of the device leg.
    cpu = None
    parity = None
    if not args.no_cpu_baseline:
        n_or = nseq if world == 1 else min(nseq, 2)
        okw = dict(dict(prev_frames=15), **kw_cfg)
        cpu_run = cpu_baseline_single_stream(seqs[:n_or], okw=okw, width=width, height=height, name=args.config.upper())
        checked = 0
        worst = [0.0, 0.0]
        ok = True
        for l in range(B):
            sidx = l % nseq
            if sidx >= n_or:
                continue
            dt, dr = pose_err(poses_dev[l], cpu_run["final_poses"][sidx])
            e_ok = int(nedges[l]) == int(cpu_run["final_edges"][sidx])
            worst = [max(worst[0], dt), max(worst[1], dr)]
            ok = ok and dt < 1e-4 and dr < 1e-5 and e_ok
            checked += 1
        if world > 1:
            t = torch.tensor([float(checked), 0.0 if ok else 1.0, worst[0], worst[1]], dtype=torch.float64, device=dev)
            tmax = t.clone()
            dist.all_reduce(t, op=dist.ReduceOp.SUM)
            dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
            checked, ok, worst = int(t[0].item()), t[1].item() == 0.0, [tmax[2].item(), tmax[3].item()]
        parity = {"parity_checked_lanes": checked, "parity_ok": bool(ok), "frames_per_lane": nframes,
                  "worst_pose_error_m": worst[0], "worst_pose_error_rad": worst[1], "tolerance": "1e-4 m / 1e-5 rad, edge counts exact",
                  "against": "oracle free run of the same sequences (final frame of the device-resident leg)"}
        if rank == 0 and world == 1:
            cpu = {k: v for k, v in cpu_run.items() if k not in ("final_poses", "final_edges")}

    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if rank != 0:
        return
    out = {
        "metric": METRIC, "value": round(value, 2), "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
        "ms_per_step": round(ms_total / K, 4), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32 selection/kNN, f64 gates+LM", "data": "synthetic",
        "config": {"workload": workload,
                   "lanes_per_gpu": B, "distinct_sequences_per_gpu": nseq, "points_per_scan": int(npts.mean()),
                   "sharding": "independent sequences per GPU, no collective",
                   "pre_roll_steps": P,
                   "window": "full (prev_frames=%d frames) in every warm-up and timed step: %d untimed pre-roll steps come first" % (kw["prev_frames"], P),
                   "l2": "every step reads a distinct scan batch at distinct addresses per lane (%d MB/step/GPU; %d MB over the run; L2 is 126 MB), uploaded before timing"
                         % (int(B * npts.mean() * 16 / 1e6), int(B * npts.sum(axis=1).mean() * 16 / 1e6))},
        "ms_per_scan_amortised": round(ms_total / K / B, 5),
        "latency_ms_per_scan": round(ms_total / K, 4),
        "e2e": {"value": round(e2e_value, 2), "unit": UNIT, "h2d_bytes_per_step": int(h2d / K), "d2h_bytes_per_step": int(d2h / K),
                "ms_per_step": round(e2e_ms / K, 4), "latency_ms_per_scan": round(e2e_ms / K, 4), "same_poses_as_device_leg": same,
                "h2d_gbps_in_run": round(h2d_in_run_gbps, 1), "h2d_gbps_link_alone": round(h2d_alone_gbps, 1),
                "h2d_gbps_per_rank_all_ranks_copying": round(h2d_concurrent_gbps, 1),
                "bound": "PCIe H2D of the raw scans (16 B/point)" if h2d_in_run_gbps > 0.85 * h2d_alone_gbps else "kernels"},
        "gpu_launches": int(launches),
        "clocks": clocks,
        "synth_seconds": round(gen_s, 1),
    }
    if parity is not None:
        out.update({"parity_checked_lanes": parity["parity_checked_lanes"], "parity": parity})
    if roof is not None:
        out["roofline"] = roof
        out["stages"] = stages
    if xyz12 is not None:
        out["e2e_xyz12"] = xyz12
    if single is not None:
        out["single_stream"] = single
    if facade is not None:
        out["facade_single_stream"] = facade
    if sharded is not None:
        out["point_sharded"] = sharded
    if cpu is not None:
        out["cpu_baseline"] = cpu
    emit(out)


DUMP_BYTES = 64 << 20


def dump_outputs(out_dir, ctx, poses, nedges):
    """What a caller of the device-resident path receives for the last timed step, so that two builds can be
    compared output for output on the same seeded inputs: poses [lanes,4,4] (f64), edge counts [lanes] (as f64) and
    the edge clouds of all lanes back to back [sum(edges),4] (f32 x, y, z, intensity).  Edge rows beyond the 64 MB
    budget are thinned to a fixed seeded sample (the same rows whenever the edge counts agree)."""
    os.makedirs(out_dir, exist_ok=True)
    edges = np.concatenate([ctx.scan_edges(l) for l in range(ctx.batch)])
    room = max((DUMP_BYTES - poses.nbytes - 8 * nedges.size) // (edges.itemsize * edges.shape[1]), 0)
    if len(edges) > room:
        edges = edges[np.sort(np.random.default_rng(0).choice(len(edges), room, replace=False))]
    np.save(os.path.join(out_dir, "poses.npy"), np.asarray(poses, np.float64))
    np.save(os.path.join(out_dir, "n_edges.npy"), np.asarray(nedges, np.float64))
    np.save(os.path.join(out_dir, "edges.npy"), np.asarray(edges, np.float32))


def single_stream_block(api, torch, dev, local, scans, npts, kw, P, W, K, width, height):
    """One sequence through a batch-1 context (lanes = 1): the reference's own shape, one stream through
    liodom_node (src/liodom_node.cc:85-91).  Device-resident scans/s and end to end from pinned host scans."""
    nframes = len(scans)
    K1 = nframes - P - W
    dscans = [torch.from_numpy(s).to(dev) for s in scans]
    hscans = [torch.from_numpy(s).pin_memory() for s in scans]
    out = {}
    for leg in ("device", "e2e"):
        ctx = api.Context(batch=1, device=local, **kw)
        stream = torch.cuda.ExternalStream(ctx.stream, device=dev)

        def enq(f):
            if leg == "device":
                ctx.scan_batch_ptrs([dscans[f].data_ptr()], [int(npts[f])], BYTES_PER_POINT, width=width, height=height, on_device=True)
            else:
                ctx.scan_batch_ptrs([hscans[f].data_ptr()], [int(npts[f])], BYTES_PER_POINT, width=width, height=height, on_device=False)

        for f in range(P + W):
            enq(f)
            ctx.results()
        torch.cuda.synchronize()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        ev0.record(stream)
        for f in range(P + W, nframes):
            enq(f)
            if leg == "e2e" and f > P + W:
                ctx.results(age=1)     # every frame's pose is read back on the host
        ctx.results(age=0)
        ev1.record(stream)
        ctx.sync()
        wall = (time.perf_counter() - t0) * 1e3
        ms = ev0.elapsed_time(ev1) if leg == "device" else max(ev0.elapsed_time(ev1), wall)
        out[leg] = (K1 / (ms * 1e-3), ms / K1)
        ctx.close()
    return {"lanes": 1, "value": round(out["device"][0], 1), "ms_per_scan": round(out["device"][1], 4),
            "e2e_value": round(out["e2e"][0], 1), "e2e_ms_per_scan": round(out["e2e"][1], 4), "unit": UNIT, "frames_timed": K1,
            "note": "one sequence, full window; the GPU is mostly idle at this shape (latency of ~20 dependent kernels)"}


def point_sharded_run(api, torch, dist, rank, world, local, nframes, warm, sensor="hdl64_1m", scan_regions=64):
    """BASELINE.json config 5, second half: ONE stream of 1M-point scans (64 rings x 15,625 az; scan_regions=64 so that
    E ~ 45k edges, SURVEY.md §8(d) note F5).  world == 1: the ordinary single-GPU path on that shape.  world > 1: every
    rank receives the same scan; extraction shards by ring, association / LM evaluation by edge, one all-gather of the
    edge slots per scan and one 29-double ncclAllReduce per LM evaluation; rank 0 also runs the single-GPU path on the
    same scans (untimed against the others) as the parity reference and the same-shape baseline."""
    from liodom_b200 import synth
    dev = torch.device("cuda", local)
    scans, _ = synth.sequence(sensor, 1000, nframes)
    kw = dict(prev_frames=15, scan_regions=scan_regions, max_points=1 << 20, device=local)
    dscans = [torch.from_numpy(s).to(dev) for s in scans]

    def run(ctx, timed_from):
        stream = torch.cuda.ExternalStream(ctx.stream, device=dev)
        poses, ne = [], []
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        for f in range(nframes):
            if f == timed_from:
                if world > 1:
                    dist.barrier()
                torch.cuda.synchronize()
                ev0.record(stream)
            ctx.scan_batch_ptrs([dscans[f].data_ptr()], [len(scans[f])], 16, on_device=True)
            if f < timed_from:
                ctx.sync()
            if f >= timed_from - 1:
                p, n = ctx.results()      # poses are read back every frame (the stream is sequential anyway)
                poses.append(p[0].copy())
                ne.append(int(n[0]))
        ev1.record(stream)
        ctx.sync()
        return ev0.elapsed_time(ev1) / (nframes - timed_from), poses, ne

    out = {"sensor": sensor, "points_per_scan": int(np.mean([len(s) for s in scans])), "scan_regions": scan_regions,
           "frames_timed": nframes - warm, "world": world}
    single_ms = None
    single_poses = None
    if rank == 0:
        # the ordinary single-GPU path on the same scans: the job's time at world == 1; at world > 1 the parity reference
        # and same-shape baseline (only rank 0 runs it, before the sharded leg; `run` must not hit the barrier then)
        ctx = api.Context(batch=1, **kw)
        stream = torch.cuda.ExternalStream(ctx.stream, device=dev)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        single_poses, ne = [], []
        for f in range(nframes):
            if f == warm:
                torch.cuda.synchronize()
                e0.record(stream)
            ctx.scan_batch_ptrs([dscans[f].data_ptr()], [len(scans[f])], 16, on_device=True)
            p, n = ctx.results()
            if f >= warm - 1:
                single_poses.append(p[0].copy())
                ne.append(int(n[0]))
        e1.record(stream)
        ctx.sync()
        single_ms = e0.elapsed_time(e1) / (nframes - warm)
        d = ctx.scan_diag(0)
        out.update({"edges_per_scan": int(np.mean(ne)), "map_points": int(d.n_map[0]), "single_gpu_ms_per_scan": round(single_ms, 4)})
        # per-stage device times of one more scan (events between the stages; outside the timed span)
        ctx.stage_timing(True)
        ctx.scan_batch_ptrs([dscans[nframes - 1].data_ptr()], [len(scans[nframes - 1])], 16, on_device=True)
        ctx.sync()
        sms, _ = ctx.stage_times()
        ctx.stage_timing(False)
        out["single_gpu_stage_ms"] = {k: round(float(v), 4) for k, v in zip(api.STAGE_NAMES, sms)}
        ctx.close()
    if world > 1:
        uid = [api.shard_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(uid, src=0)
        ctx = api.Context(batch=1, **kw)
        ctx.shard_init(rank, world, uid[0])
        l0 = ctx.launch_count
        ms, poses, ne = run(ctx, warm)
        launches = ctx.launch_count - l0
        ctx.stage_timing(True)   # one more scan with events between the stages (every rank: the collectives need all of them)
        ctx.scan_batch_ptrs([dscans[nframes - 1].data_ptr()], [len(scans[nframes - 1])], 16, on_device=True)
        ctx.sync()
        sms, _ = ctx.stage_times()
        ctx.stage_timing(False)
        out["sharded_stage_ms"] = {k: round(float(v), 4) for k, v in zip(api.STAGE_NAMES, sms)}
        t = torch.tensor([ms], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        # every rank must hold bitwise the same poses (the LM controller is replicated)
        mine = torch.from_numpy(np.stack(poses)).to(dev)
        ref0 = mine.clone()
        dist.broadcast(ref0, src=0)
        same = torch.tensor([1.0 if torch.equal(mine, ref0) else 0.0], device=dev)
        dist.all_reduce(same, op=dist.ReduceOp.MIN)
        ctx.close()
        if rank == 0:
            worst = max(max(pose_err(a, b)) for a, b in zip(poses, single_poses))
            out.update({"sharded_ms_per_scan": round(float(t.item()), 4), "value": round(1e3 / float(t.item()), 2), "unit": "scans/s",
                        "speedup_vs_single_gpu": round(single_ms / float(t.item()), 3),
                        "ranks_bitwise_equal": bool(same.item() == 1.0), "worst_pose_diff_vs_single_gpu": worst,
                        "kernel_launches_per_scan": round(launches / nframes, 1),
                        "collectives": "1 grouped all-gather of the edge slots + up to 10 ncclAllReduce(29 x f64) per scan, on the context's stream"})
    elif rank == 0:
        out.update({"value": round(1e3 / single_ms, 2), "unit": "scans/s"})
    return out


def run_sharded(args):
    """bench.py --mode sharded [--gpus N]: the point-sharded 1M-point stream as its own JSON line (strong scaling)."""
    import torch
    import torch.distributed as dist
    from liodom_b200 import api
    rank, world, local = dist_env()
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    torch.cuda.set_device(local)
    K, W = args.steps, max(args.warmup, 1)
    r = point_sharded_run(api, torch, dist, rank, world, local, 16 + W + K, 16 + W)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if rank != 0:
        return
    ms = r.get("sharded_ms_per_scan", r.get("single_gpu_ms_per_scan"))
    emit({"metric": "scans_per_sec_1m_point_stream_point_sharded", "value": r["value"], "unit": "scans/s", "n_gpus": world, "steps": K, "warmup": W,
          "ms_per_step": ms, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32 selection/kNN, f64 gates+LM",
          "data": "synthetic",
          "config": {"workload": "C5b: one stream of 1M-point scans (64 x 15,625), scan_regions=64, prev_frames=15, full window; "
                                 "ring-sharded extraction, edge-sharded association + LM, replicated window", "pre_roll_steps": 16},
          "point_sharded": r})


def run_c4(args):
    """BASELINE.json config 4: liodom_mapping_node's per-message sequence (src/liodom_mapping_node.cc:45-90) over a
    closed loop: Map::updateMap + Map::getLocalMap every frame, Map::getMap every 100th, both shipped parameter sets,
    GPU (C ABI, host buffers in / out) against the oracle Map on the host, maps compared bit for bit."""
    import oracle
    from liodom_b200 import api, synth
    rank, world, local = dist_env()
    if rank != 0:
        return
    nfr = args.frames
    t0 = time.time()
    ctx = api.Context(max_points=131072, device=local)
    clouds, poses = [], []
    T0 = synth.gt_pose(1000, 0, traj=1)
    for f in range(nfr):      # edge clouds from the GPU extractor (untimed), ground-truth poses of the ~4 km circuit
        clouds.append(ctx.extract(synth.scan("hdl64", 1000, f, traj=1)))
        poses.append(np.linalg.inv(T0) @ synth.gt_pose(1000, f, traj=1))
    ctx.close()
    gen_s = time.time() - t0
    res = {}
    for name, (xy, z, cxy, cz) in {"liodom_mapping.launch": (20.0, 25.0, 2, 1), "liodom.launch": (30.0, 35.0, 3, 2)}.items():
        gm = api.Map(xy, z, 0.4, device=local, max_points=1 << 23)
        gm.update(clouds[0], poses[0])          # warm-up (allocations, first kernels)
        gm.get_local_map(poses[0], cxy, cz)
        gm.close()
        gm = api.Map(xy, z, 0.4, device=local, max_points=1 << 23)
        nloc = nfull = 0
        t_upd = t_loc = t_full = 0.0
        g_samples = {}
        for f, (c, T) in enumerate(zip(clouds, poses)):
            a = time.perf_counter()
            gm.update(c, T)
            b = time.perf_counter()
            loc = gm.get_local_map(T, cxy, cz)
            d = time.perf_counter()
            t_upd += b - a
            t_loc += d - b
            nloc += len(loc)
            if f % 100 == 0:      # the mapping node publishes the full map only when someone listens; BASELINE: every 100th frame
                a = time.perf_counter()
                full = gm.get_map()
                t_full += time.perf_counter() - a
                nfull += 1
                g_samples[f] = (loc.copy(), len(full))
        tg = t_upd + t_loc + t_full
        npts, ncells = gm.size()
        gfull = gm.get_map()
        gk, gc = gm.cells()
        om = oracle.Map(xy, z, 0.4)
        ok_local = True
        t0c = time.perf_counter()
        for f, (c, T) in enumerate(zip(clouds, poses)):
            om.update(c, T)
            ol = om.get_local_map(T, cxy, cz)
            if f % 100 == 0:
                of = om.get_map()
                ok_local = ok_local and np.array_equal(ol.view(np.uint32), g_samples[f][0].view(np.uint32)) and len(of) == g_samples[f][1]
        tc = time.perf_counter() - t0c
        okk, okc = om.cells()
        same = bool(np.array_equal(gfull.view(np.uint32), om.get_map().view(np.uint32)) and np.array_equal(gk, okk) and np.array_equal(gc, okc))
        assert same and ok_local, "C4 %s: GPU map differs from the oracle map" % name
        res[name] = {"voxel_xysize": xy, "voxel_zsize": z, "cells_xy": cxy, "cells_z": cz, "frames": nfr,
                     "edges_per_frame": int(np.mean([len(c) for c in clouds])), "map_points": npts, "cells": ncells,
                     "local_map_points_per_frame": int(nloc / nfr), "getMap_calls": nfull,
                     "gpu_ms_per_frame": round(tg / nfr * 1e3, 4),
                     "gpu_ms": {"updateMap": round(t_upd / nfr * 1e3, 4), "getLocalMap": round(t_loc / nfr * 1e3, 4), "getMap_per_call": round(t_full / max(nfull, 1) * 1e3, 3)},
                     "cpu_oracle_ms_per_frame": round(tc / nfr * 1e3, 4),
                     "map_and_sampled_local_maps_bitwise_equal_to_oracle": True}
        gm.close()
    head = res["liodom_mapping.launch"]
    emit({"metric": "c4_map_build_ms_per_frame", "value": head["gpu_ms_per_frame"], "unit": "ms/frame", "n_gpus": 1, "steps": nfr, "warmup": 1,
          "ms_per_step": head["gpu_ms_per_frame"], "higher_is_better": False, "scaling": "weak", "vs_baseline": None, "dtype": "f32 centroids, f64 keys",
          "data": "synthetic",
          "config": {"workload": "C4: %d-frame closed loop (~4 km rounded square) of HDL-64 edge clouds + ground-truth poses through updateMap -> "
                                 "getLocalMap (every frame) -> getMap (every 100th), launch/liodom_mapping.launch:15-19 and launch/liodom.launch:46-50 params" % nfr},
          "e2e": {"value": head["gpu_ms_per_frame"], "unit": "ms/frame", "note": "the Map C ABI takes and returns HOST buffers: every number here is end to end"},
          "cpu_baseline": {"value": head["cpu_oracle_ms_per_frame"], "unit": "ms/frame", "cores": 1, "kind": "port",
                           "sample": "the same %d frames through the oracle Map (restated src/map.cc + PCL VoxelGrid), one thread as the reference" % nfr},
          "results": res, "synth_seconds": round(gen_s, 1)})


def cpu_baseline_single_stream(seqs, okw=None, width=0, height=0, name="C1"):
    """The oracle port with the reference's own threading (OpenMP curvature loop with
    max(2, nthreads-5) threads, solver threads = nproc), one stream after another.  Also returns the
    final pose / edge count of every sequence (the bench's parity check against the GPU lanes)."""
    import oracle
    op = oracle.make_params(**(okw or dict(prev_frames=15)))
    n = 0
    t0 = time.perf_counter()
    stage = np.zeros(5)
    finals, fedges = [], []
    for scans in seqs:
        poses, st, _ = oracle.run_sequence(op, scans, width, height)
        stage += st
        n += len(scans)
        finals.append(poses[-1])
    dt = time.perf_counter() - t0
    for scans in seqs:   # edge count of the last frame (outside the timed span)
        fedges.append(len(oracle.extract_scan(op, scans[-1], width, height)[0]))
    return {"value": round(n / dt, 3), "unit": UNIT, "cores": os.cpu_count(), "kind": "port",
            "sample": "%d scans (%d %s sequences x %d frames), single stream, reference threading (restated CPU path, pinned against "
                      "the reference's own object code in oracle/_ref; the reference binary needs ROS/PCL/Ceres and cannot be built here)"
                      % (n, len(seqs), name, len(seqs[0])),
            "ms_per_scan": round(dt / n * 1e3, 3),
            "stage_ms_per_scan": {k: round(v / n / 1e3, 3) for k, v in zip(("split", "extract", "associate", "solve", "window"), stage)},
            "final_poses": finals, "final_edges": fedges}


def run_reference(args):
    """Reference arm: the restated CPU path on the host cores, one independent sequence per
    worker thread (the same sharding the GPU arm uses), all cores busy."""
    rank, world, _ = dist_env()
    if rank != 0:
        return
    import oracle
    from concurrent.futures import ThreadPoolExecutor
    K, W = args.steps, args.warmup
    cores = os.cpu_count() or 1
    workers = cores
    P = 15 + 1            # the same pre-roll as the GPU arm: the window is full in every warm-up and timed step
    nframes = P + W + K
    nseq = min(workers, N_SEEDS)
    seqs = make_sequences(args.sensor, 0, nseq, nframes)
    op = oracle.make_params(prev_frames=15, omp_threads=1)
    odos = [oracle.Odometer(op) for _ in range(workers)]

    def one(wf):
        w, f = wf
        s = seqs[w % nseq][f]
        edges, _ = oracle.extract_scan(op, s)
        odos[w].process(edges)
        return len(edges)

    pool = ThreadPoolExecutor(workers)
    for f in range(P + W):
        list(pool.map(one, [(w, f) for w in range(workers)]))
    t0 = time.perf_counter()
    for f in range(P + W, nframes):
        list(pool.map(one, [(w, f) for w in range(workers)]))
    dt = time.perf_counter() - t0
    pool.shutdown()
    value = workers * K / dt
    npts = int(np.mean([len(s) for s in seqs[0]]))
    out = {
        "impl": "reference", "metric": METRIC, "value": round(value, 3), "unit": UNIT, "n_gpus": args.gpus, "steps": K,
        "warmup": W, "ms_per_step": round(dt / K * 1e3, 3), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32 selection/kNN, f64 gates+LM", "data": "synthetic",
        "config": {"workload": "C1: HDL-64-shaped ray-cast urban sequences (~118k pts/scan), launch/liodom.launch params, "
                               "extract+register", "lanes": workers, "points_per_scan": npts, "pre_roll_steps": P},
        "cpu_baseline": {"value": round(value, 3), "unit": UNIT, "cores": cores, "kind": "port",
                         "sample": "%d workers x %d scans, one independent sequence per host thread (restated CPU path: "
                                   "the reference binary needs ROS/PCL/Ceres and cannot be built here)" % (workers, K)},
        "e2e": {"value": round(value, 3), "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(out)


_REAL_STDOUT = None


def emit(obj):
    """The one JSON line of the contract, written to the process's original stdout."""
    line = json.dumps(obj) + "\n"
    if _REAL_STDOUT is None:
        sys.stdout.write(line)
        sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, line.encode())


def main():
    global _REAL_STDOUT
    args = parse()
    # Libraries print to stdout on their own (NCCL's version banner under torchrun): keep fd 1 for the
    # JSON line only and send everything else to stderr.
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    if args.impl == "reference":
        run_reference(args)
    elif args.config == "c4":
        run_c4(args)
    elif args.mode == "sharded":
        run_sharded(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
