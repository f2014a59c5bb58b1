"""Cost of partial steps (liodom_scan_lanes) on a 128-lane C1 context, device-resident scans.

For every k in {1, 8, 32, 64, 128}: a 128-lane context P_k steps a fixed seeded random subset S_k of k lanes (in a
fresh seeded order every step), and a batch-k context Q_k takes full steps whose lane j runs the same sequence as
P_k's lane S_k[j].  Both are pre-rolled with the same 16 full steps (every window full) and advance one frame per
step, so P_k's lane S_k[j] and Q_k's lane j see the same scans in the same order and do the same work; the run
reports the largest pose difference between them.  A further pair of 128-lane contexts with the same history times
liodom_scan_batch against the identity list (liodom_scan_lanes with lanes = 0..127).

Each pair is timed back to back, its order alternating, over --reps rounds; every timed window is --steps steps,
each ended by results() (a synchronise), between two CUDA events on the context's stream.  Prints one JSON line:
median ms per step of each variant, the ratios, the GPU name and its power limit.

After the pre-roll a lane's frame index walks forwards and backwards over the next --frames frames, so consecutive
scans of a lane stay consecutive in the trajectory however many steps the run takes."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from liodom_b200 import api, synth  # noqa: E402

PRE = 16
N_SEEDS = 8


def gpu_info():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    name, power = [s.strip() for s in out.stdout.splitlines()[0].split(",")]
    return name, power


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--batch", type=int, default=128)
    ap.add_argument("--steps", type=int, default=20, help="steps per timed window")
    ap.add_argument("--reps", type=int, default=5, help="alternating rounds")
    ap.add_argument("--frames", type=int, default=24, help="frames after the pre-roll that the lanes walk over")
    ap.add_argument("--ks", default="1,8,32,64,128")
    args = ap.parse_args()
    import torch
    B, ks = args.batch, [int(k) for k in args.ks.split(",")]
    nfr = PRE + args.frames
    seqs = [synth.sequence("hdl64", 1000 + s, nfr)[0] for s in range(N_SEEDS)]
    dev = [[torch.from_numpy(f).cuda() for f in sq] for sq in seqs]
    kw = dict(prev_frames=15, max_points=131072)

    def frame_of(step):   # pre-roll, then back and forth over the next `frames` frames
        if step < PRE:
            return step
        period = 2 * (args.frames - 1)
        u = (step - PRE) % period
        return PRE + (u if u < args.frames else period - u)

    class Ctx:
        """A context whose lane l runs sequence seed[l]; every lane has taken the same number of steps so far, and
        only the lanes stepped advance."""

        def __init__(self, seed):
            self.seed = seed
            self.ctx = api.Context(batch=len(seed), **kw)
            self.taken = [0] * len(seed)
            self.stream = torch.cuda.ExternalStream(self.ctx.stream)

        def _scans(self, lanes):
            out = [dev[self.seed[l]][frame_of(self.taken[l])] for l in lanes]
            for l in lanes:
                self.taken[l] += 1
            return [t.data_ptr() for t in out], [t.shape[0] for t in out]

        def batch(self):
            p, n = self._scans(range(len(self.seed)))
            self.ctx.scan_batch_ptrs(p, n, 16)

        def lanes(self, lanes):
            p, n = self._scans(lanes)
            self.ctx.scan_lanes_ptrs(lanes, p, n, 16)

        def time(self, fn):
            ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            ev0.record(self.stream)
            for _ in range(args.steps):
                fn()
                self.ctx.results()
            ev1.record(self.stream)
            torch.cuda.synchronize()
            return ev0.elapsed_time(ev1) / args.steps

    rng = np.random.default_rng(0)
    seed_of = [l % N_SEEDS for l in range(B)]
    subset = {k: sorted(rng.choice(B, size=k, replace=False).tolist()) for k in ks}
    part = {k: Ctx(seed_of) for k in ks}
    full = {k: Ctx([seed_of[l] for l in subset[k]]) for k in ks}
    sb, il = Ctx(seed_of), Ctx(seed_of)
    everything = list(part.values()) + list(full.values()) + [sb, il]
    for _ in range(PRE):   # pre-roll: every window full
        for c in everything:
            c.batch()
    for c in everything:
        c.ctx.results()

    def partial_step(k):
        part[k].lanes([subset[k][i] for i in rng.permutation(k)])

    res = {"partial": {k: [] for k in ks}, "batch_k": {k: [] for k in ks}, "scan_batch": [], "identity_list": []}
    for r in range(args.reps + 1):   # round 0 warms up every shape the timed windows use
        for k in ks:
            pair = [("partial", part[k], lambda: partial_step(k)), ("batch_k", full[k], full[k].batch)]
            for name, c, fn in (pair if r % 2 == 0 else pair[::-1]):
                t = c.time(fn)
                if r:
                    res[name][k].append(t)
        pair = [("scan_batch", sb, sb.batch), ("identity_list", il, lambda: il.lanes(list(range(B))))]
        for name, c, fn in (pair if r % 2 == 0 else pair[::-1]):
            t = c.time(fn)
            if r:
                res[name].append(t)
    # like for like: the subset's lanes of P_k and the lanes of Q_k took the same scans, so their poses must agree
    diff = {}
    for k in ks:
        pp, _ = part[k].ctx.results()
        pf, _ = full[k].ctx.results()
        assert [part[k].taken[l] for l in subset[k]] == full[k].taken
        diff[str(k)] = float(np.abs(pp[subset[k]] - pf).max())
    med = lambda v: float(np.median(v))
    name, power = gpu_info()
    out = {"gpu": name, "power_limit": power, "batch": B, "steps_per_window": args.steps, "reps": args.reps,
           "ms_per_step": {
               "partial_on_%d_lanes" % B: {str(k): round(med(res["partial"][k]), 4) for k in ks},
               "full_step_batch_k": {str(k): round(med(res["batch_k"][k]), 4) for k in ks},
               "scan_batch": round(med(res["scan_batch"]), 4), "identity_list": round(med(res["identity_list"]), 4)},
           "partial_over_batch_k": {str(k): round(med(res["partial"][k]) / med(res["batch_k"][k]), 4) for k in ks},
           "identity_list_over_scan_batch": round(med(res["identity_list"]) / med(res["scan_batch"]), 4),
           "spread_ms": {"partial": {str(k): [round(min(res["partial"][k]), 4), round(max(res["partial"][k]), 4)] for k in ks},
                         "batch_k": {str(k): [round(min(res["batch_k"][k]), 4), round(max(res["batch_k"][k]), 4)] for k in ks},
                         "scan_batch": [round(min(res["scan_batch"]), 4), round(max(res["scan_batch"]), 4)],
                         "identity_list": [round(min(res["identity_list"]), 4), round(max(res["identity_list"]), 4)]},
           "max_pose_diff_partial_vs_batch_k": diff}
    print(json.dumps(out))


if __name__ == "__main__":
    main()
