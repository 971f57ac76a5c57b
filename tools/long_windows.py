"""Long windows (T = 33..64) with the open-set head: arx_score on the tiled tensor-core route against the fp32 kernels
(force_path = 1), and the per-frame latency of the resident streaming scorer (arx_stream_push).

arx_score is timed on device events around one call (median / min of --reps, the two routes alternated), on structured
inputs resident in HBM, without an L2 flush between calls: the class tiles and the fp16 image of discriminator.fc1
(66 MB at T=64) stay in L2 as they do in steady use.  attn GFLOP/s is the algorithmic attention work 4*W*N^2*D per
window (N = C(T,2) query and support tuples, D = 128) over the whole call time: a whole-call rate, not a kernel's rate.
rel.diff is the largest relative difference of logits / is_true between the two routes on the timed windows.

arx_stream_push is timed on the host clock per call (the call ends in a stream synchronise): T + 8 warm-up frames, then
--frames frames on the replayed per-frame graph.

Usage (GPU): python tools/long_windows.py [--reps 5] [--frames 200] [--out FILE]"""
import argparse
import os
import subprocess
import sys
import time
from math import comb

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

from oracle.synth import Cfg, make_episode
from tests.util import make_model, rel_err

D = 128
# (T, way, windows on the tiled route, windows on the fp32 kernels)
SCORE_SHAPES = [(40, 5, 1024, 32), (40, 20, 256, 8), (48, 5, 512, 16), (48, 20, 128, 4), (64, 5, 256, 8), (64, 20, 64, 2)]
STREAM_SHAPES = [(40, 5), (64, 5)]


def device_line():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return f"# device: {torch.cuda.get_device_name(0)}; nvidia-smi name, power.limit, clocks.max.sm: {q.stdout.strip() or 'n/a'}"


def timed(fn):
    st = torch.cuda.current_stream()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record(st)
    out = fn()
    b.record(st)
    torch.cuda.synchronize()
    return a.elapsed_time(b), out


def score_line(T, way, n_tc, n_fp, reps):
    cfg = Cfg(way=way, seq_len=T)
    support, _, query, _ = make_episode(cfg, n_tc, 3, "structured")
    S, Q = torch.from_numpy(support[0]).cuda(), torch.from_numpy(query).cuda()
    runs = {}
    for force, n in ((0, n_tc), (1, n_fp)):
        m, _ = make_model(cfg, 0, force_path=force)
        m.set_support(poses=S)
        q = Q[:n].contiguous()
        out = m.score(q)                                          # first call: allocations, one-time tables
        runs[force] = (m, q, out, m.last_path())
    times = {0: [], 1: []}
    for _ in range(reps):
        for force in (0, 1):
            m, q, _, _ = runs[force]
            times[force].append(timed(lambda: m.score(q))[0])
    lo_tc, it_tc = runs[0][2]
    lo_fp, it_fp = runs[1][2]
    diff = max(rel_err(lo_tc[:n_fp].cpu(), lo_fp.cpu()).max(), rel_err(it_tc[:n_fp].cpu(), it_fp.cpu()).max())
    N = comb(T, 2)
    flop = 4 * way * N * N * D
    t_tc, t_fp = np.array(times[0]), np.array(times[1])
    ws_tc, ws_fp = n_tc / (np.median(t_tc) * 1e-3), n_fp / (np.median(t_fp) * 1e-3)
    return (f"{T:3d} {way:4d} {N:5d} {n_tc:6d} {runs[0][3]:4d} {np.median(t_tc):9.3f} {t_tc.min():9.3f} {ws_tc:11.1f} "
            f"{ws_tc * flop * 1e-9:10.0f} {n_fp:5d} {runs[1][3]:4d} {np.median(t_fp):9.3f} {ws_fp:9.1f} {ws_tc / ws_fp:7.1f}x {diff:9.2e}")


def stream_line(T, way, frames):
    cfg = Cfg(way=way, seq_len=T)
    m, _ = make_model(cfg, 0)
    rng = np.random.default_rng(5)
    support = (0.17 * rng.standard_normal((way, T, 90))).astype(np.float32)
    m.set_support(poses=torch.from_numpy(support).cuda())
    x = (0.17 * rng.standard_normal((T + 8 + frames, 90))).astype(np.float32)
    for f in x[:T + 8]:
        m.stream_push(f)
    lat = []
    for f in x[T + 8:]:
        t0 = time.perf_counter()
        _, _, valid = m.stream_push(f)
        lat.append((time.perf_counter() - t0) * 1e3)
        assert valid
    lat = np.array(lat)
    return f"{T:3d} {way:4d} {comb(T, 2):5d} {frames:6d} {m.last_path():4d} {np.median(lat):9.3f} {np.percentile(lat, 90):9.3f} {lat.min():9.3f}"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--frames", type=int, default=200)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("long_windows: needs a CUDA device")
    lines = [device_line(),
             f"# arx_score, DISC, pair tuples, structured inputs: ms = device-event time of one call (median / min of {args.reps},",
             "# routes alternated); path 3 = tiled tensor-core kernels, 1 = fp32 kernels (force_path = 1)",
             f"{'T':>3s} {'way':>4s} {'N':>5s} {'n.tc':>6s} {'path':>4s} {'tc ms':>9s} {'min':>9s} {'tc win/s':>11s} {'attn GF/s':>10s} "
             f"{'n.fp':>5s} {'path':>4s} {'fp32 ms':>9s} {'fp32 win/s':>9s} {'speedup':>8s} {'rel.diff':>9s}"]
    print("\n".join(lines), flush=True)
    for shape in SCORE_SHAPES:
        line = score_line(*shape, args.reps)
        print(line, flush=True)
        lines.append(line)
    head = [f"# arx_stream_push, DISC, pair tuples: host-clock latency of one call over {args.frames} frames (graph replay)",
            f"{'T':>3s} {'way':>4s} {'N':>5s} {'frames':>6s} {'path':>4s} {'median ms':>9s} {'p90 ms':>9s} {'min ms':>9s}"]
    print("\n".join(head), flush=True)
    lines += head
    for T, way in STREAM_SHAPES:
        line = stream_line(T, way, args.frames)
        print(line, flush=True)
        lines.append(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
