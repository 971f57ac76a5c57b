"""Per-episode support sets on the tiled tensor-core route: arx_score_episodes (one batched pass per pool of episodes)
against the per-episode sequence it replaced (set_support + a one-window score per episode), on the same handle.

Times both on device events (the host enqueue of the per-episode sequence is part of its time), alternating them,
checks that they give bit-identical outputs, and reports the memory of the batched call: the torch peak
(inputs, outputs) and the drop in free device memory across the first call, which is what the library allocates
with cudaMalloc (support pool, class tiles, workspace).

Usage (GPU): python tools/episodes_tiled.py [--episodes 300] [--reps 5] [--out FILE]"""
import argparse
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

from oracle.synth import Cfg
from tests.util import make_model

SHAPES = [   # name, config (20-way T=32 is the cfg4 shape, temp_set [2, 3])
    ("t32_pairs_w20", Cfg(way=20, seq_len=32, temp_set=[2, 3])),
    ("t8_pairs_w5", Cfg(way=5, seq_len=8)),
    ("t16_triples_w5_nodisc", Cfg(way=5, seq_len=16, temp_set=[3], model="NONE")),
]


def device_line():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    return f"# device: {torch.cuda.get_device_name(0)}; nvidia-smi name, power.limit: {q.stdout.strip() or 'n/a'}"


def timed(fn):
    st = torch.cuda.current_stream()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record(st)
    out = fn()
    b.record(st)
    torch.cuda.synchronize()
    return a.elapsed_time(b), out


def run_shape(name, cfg, n, reps):
    m, _ = make_model(cfg, 0)
    rng = np.random.default_rng(1)
    S = torch.from_numpy((0.17 * rng.standard_normal((n, cfg.way, cfg.seq_len, 90))).astype(np.float32)).cuda()
    Q = (S[torch.arange(n, device="cuda"), torch.from_numpy(rng.integers(0, cfg.way, n)).cuda()]
         + 0.05 * torch.randn((n, cfg.seq_len, 90), generator=torch.Generator().manual_seed(2)).cuda()).contiguous()

    def batched():
        return m.score_episodes(Q, poses=S)

    def loop():
        lg, it = [], []
        for e in range(n):
            m.set_support(poses=S[e])
            a, b = m.score(Q[e:e + 1])
            lg.append(a)
            it.append(b)
        return torch.cat(lg), (torch.cat(it) if it[0] is not None else None)

    m.set_support(poses=S[0])
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    free0 = torch.cuda.mem_get_info()[0]
    base = torch.cuda.memory_allocated()
    l0 = m.launch_count()
    ob = batched()                                                  # first call: allocations, one-time tables
    torch.cuda.synchronize()
    lib_bytes = free0 - torch.cuda.mem_get_info()[0]
    torch_peak = torch.cuda.max_memory_allocated() - base
    launches_b = m.launch_count() - l0
    path = m.last_path()
    l0 = m.launch_count()
    ol = loop()
    launches_l = m.launch_count() - l0
    same = torch.equal(ob[0], ol[0]) and (ob[1] is None or torch.equal(ob[1], ol[1]))
    tb, tl = [], []
    for _ in range(reps):
        tb.append(timed(batched)[0])
        tl.append(timed(loop)[0])
    tb, tl = np.array(tb), np.array(tl)
    return (f"{name:22s} {n:5d} {path:4d} {np.median(tb):9.2f} {tb.min():8.2f} {np.median(tl):9.2f} {tl.min():8.2f} "
            f"{np.median(tl) / np.median(tb):7.1f}x {launches_b:6d} {launches_l:7d} {torch_peak / 2**20:9.1f} {lib_bytes / 2**20:9.1f} "
            f"{'yes' if same else 'NO'}")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--episodes", type=int, default=300)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("episodes_tiled: needs a CUDA device")
    lines = [device_line(),
             f"# {args.episodes} episodes per call; ms = device-event time of one call (median / min of {args.reps}, alternated)",
             "# launches: kernel launches of the first call; torch MiB: torch peak over the call; lib MiB: drop in free device",
             "# memory across the first batched call (library cudaMalloc: pool, class tiles, workspace)",
             f"{'shape':22s} {'eps':>5s} {'path':>4s} {'batch ms':>9s} {'min':>8s} {'loop ms':>9s} {'min':>8s} {'ratio':>8s} "
             f"{'l.batch':>6s} {'l.loop':>7s} {'torch MiB':>9s} {'lib MiB':>9s} bit-equal"]
    print("\n".join(lines), flush=True)
    for name, cfg in SHAPES:
        line = run_shape(name, cfg, args.episodes, args.reps)
        print(line, flush=True)
        lines.append(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
