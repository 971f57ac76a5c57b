"""Logit and is_true error of the tensor-core routes against the float64 oracle, as a function of the static softmax
bound of norm_k's LayerNorm affine.  Sets the accuracy bounds of arx_internal.cuh: ARX_TC_ACCURACY_BOUND is the largest
bound whose worst error stays <= 0.6e-3 on the shapes with >= 120 query tuples, which leaves headroom under the 1e-3
tolerance for inputs the sweep did not draw; ARX_TC_ACCURACY_BOUND_FEW_TUPLES holds T=8 pairs (28 tuples) to 1e-3.

Usage (GPU): python tools/ln_bound_sweep.py [--out FILE]
Every point runs with force_path = 2, so the tensor-core kernels score it whatever the default admission says."""
import argparse
import math
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

from tests.test_layernorm_bound import (KINDS, SHAPES, beta_dominated, episode, ln_state_dict, load_model, reference,
                                        run, softmax_bound, uniform)
from tests.util import rel_err

GAMMAS = [1.0, 1.2, 1.3, 1.4, 1.5, 1.6, 1.7, 1.8, 2.0, 2.2, 2.45]
BETA_BOUNDS = [20.0, 25.0, 30.0, 35.0, 45.0, 55.0, 68.0]


def device_line():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    return f"# device: {torch.cuda.get_device_name(0)}; nvidia-smi name, power.limit: {q.stdout.strip() or 'n/a'}"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--shapes", default=",".join(SHAPES))
    args = ap.parse_args()
    lines = [device_line(), "# max relative error against float64 per query kind (" + " / ".join(KINDS) + ")",
             f"{'route':12s} {'affine':16s} {'bound':>6s} {'path':>4s}  {'logits':>28s}  {'is_true':>28s}  worst"]
    print("\n".join(lines), flush=True)
    affines = [(f"gamma={g:g}", uniform(g * g * math.sqrt(128))) for g in GAMMAS]
    affines += [(f"g0.5,beta@{bb:g}", beta_dominated(bb)) for bb in BETA_BOUNDS]
    for shape in args.shapes.split(","):
        cfg, B, ti = SHAPES[shape]
        B = max(B, 32)
        for name, (g, b) in affines:
            sd = ln_state_dict(cfg, g, b)
            m = load_model(cfg, sd, force_path=2)
            el, ei = [], []
            for kind in KINDS:
                support, labels, query = episode(cfg, B, kind)
                logits, is_true = run(m, ti, support, query)
                lo, it = reference(cfg, sd, ti, support, labels, query)
                el.append(rel_err(logits, lo).max())
                same = logits.argmax(1) == lo.argmax(1)            # a different winner feeds the discriminator another input
                ei.append(rel_err(is_true[same], it[same]).max() if it is not None else 0.0)
            worst = max(el + ei)
            line = (f"{shape:12s} {name:16s} {softmax_bound(g, b):6.1f} {m.last_path():4d}  "
                    f"{' / '.join(f'{e:.2e}' for e in el):>28s}  {' / '.join(f'{e:.2e}' for e in ei):>28s}  {worst:.2e}")
            print(line, flush=True)
            lines.append(line)
            del m
    if args.out:
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
