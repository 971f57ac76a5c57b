"""Accuracy of the tiled tensor-core route at small tuple counts N = C(T, c), against the float64 oracle.

For pairs (with the open-set head) at every T of tests/test_tuple_shapes.py up to 31 and triples up to T = 22, the same
structured and iid windows (3 seeds each, 5-way, 300 // T + 1 windows) are scored on the tiled kernels (force_path = 2,
which takes them at any N) and on the fp32 kernels (force_path = 1); the worst relative logit / is_true error of each
route against TrxOracle in float64 is reported per shape.  ARX_TC_MIN_TUPLES (arx_internal.cuh) is set from this table.

Usage (GPU): python tools/few_tuples_accuracy.py [--out FILE]"""
import argparse
import os
import subprocess
import sys
from math import comb

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

from oracle.synth import Cfg, make_episode
from oracle.trx_oracle import TrxOracle
from tests.util import make_model, rel_err

SHAPES = [(2, T) for T in (2, 3, 4, 5, 6, 7, 8, 9, 12, 15, 17, 20, 23, 25, 31)] + [(3, T) for T in (3, 4, 5, 6, 7, 9, 10, 11, 13, 21, 22)]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    lines = [f"# device: {torch.cuda.get_device_name(0)}; nvidia-smi name, power.limit: {q.stdout.strip() or 'n/a'}",
             "# worst relative error against the float64 oracle over structured + iid windows, 3 seeds each, 5-way",
             f"{'c':>2} {'T':>3} {'N':>5} {'windows':>7} {'tiled logits':>13} {'tiled is_true':>14} {'fp32 logits':>12} {'fp32 is_true':>13}"]
    print("\n".join(lines), flush=True)
    for c, T in SHAPES:
        cfg = Cfg(way=5, seq_len=T, temp_set=[c], model="DISC" if c == 2 else "NONE")
        tiled, sd = make_model(cfg, 0, force_path=2)
        fp32, _ = make_model(cfg, 0, force_path=1)
        o = TrxOracle(cfg, sd, dtype=torch.float64)
        B = 300 // T + 1
        worst = {"tiled": [0.0, 0.0], "fp32": [0.0, 0.0]}
        for kind in ("structured", "iid"):
            for seed in range(3):
                s, l, qr, _ = make_episode(cfg, B, 100 + T + 1000 * seed, kind)
                rl, ri = o.score(s, l, qr, chunk=B)
                for name, m in (("tiled", tiled), ("fp32", fp32)):
                    m.set_support(poses=torch.from_numpy(s[0]).cuda())
                    lo, it = m.score(torch.from_numpy(qr).cuda())
                    assert m.last_path() == (3 if name == "tiled" else 1)
                    worst[name][0] = max(worst[name][0], float(rel_err(lo.cpu(), rl).max()))
                    if it is not None:
                        worst[name][1] = max(worst[name][1], float(rel_err(it.cpu(), ri).max()))
        line = (f"{c:>2} {T:>3} {comb(T, c):>5} {B:>7} {worst['tiled'][0]:>13.2e} {worst['tiled'][1]:>14.2e} "
                f"{worst['fp32'][0]:>12.2e} {worst['fp32'][1]:>13.2e}")
        print(line, flush=True)
        lines.append(line)
        tiled._release()
        fp32._release()
    if args.out:
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
