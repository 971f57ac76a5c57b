#!/usr/bin/env python
"""Benchmark of the AR scoring hot path (BASELINE.json metric: query windows/sec, 5-way 1-shot, T=16).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--config cfg2|cfg3] [--dump-outputs DIR]
  python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 ... bench.py --gpus N ...

Headline workload (default, `--config cfg2`): a step = one pass of the hot path over one batch: BASELINE cfg2, 4096 synthetic
query windows (T=16 x 30 joints x 3) scored against a 5-way 1-shot support set with pair tuples, PER GPU (weak scaling:
windows are independent and shard with no data-path collective; every step re-processes the support set and, with N>1,
all-gathers the scores).  One JSON line (rank 0):

  value        device-timed (CUDA events on the launching stream, max over ranks), inputs resident in HBM, L2 flushed
               between timed steps.  The timed region is EXACTLY K steps, bracketed by barrier + synchronize; value =
               all windows / the summed step times.  At ~0.35 ms a step the default K=50 is ~17 ms of timed work, where
               one scheduling hiccup can move the figure: for a stable number give K >= 3000 (>= 1 s).
  e2e          the same metric through the host-buffer C-ABI entry points, pinned H2D / D2H inside the timed region.
  sustained    >= 2 s of back-to-back steps over a ring of input batches larger than L2 (no flush), clocks sampled
               under load; attention roofline fraction against the SUSTAINED measured bf16 peak.
  roofline     the dominant kernel (cross-attention, tensor bound), burst clocks, as in round 1.
  roofline_per_kernel   every stage of the step (SURVEY 8d k1..k5): bound, algorithmic work, measured ms, fraction.
  other_configs         BASELINE cfg3 / cfg4 / cfg5 and the per-frame streaming latency, measured in the same run (rank 0).
  cfg3         (N >= 1) NTU-shaped 60-way x 65 536 windows split over the N ranks, NCCL broadcast of the support tuple
               embeddings and all-gather of the scores INSIDE every step, cross-rank bit-equality checked.
  cpu_baseline the reference's own TRXOS (oracle/_ref, staged by oracle/build_ref.py; the oracle port if absent) on the
               box's host cores, bounded sample.

`--impl reference` times that same CPU arm on the same config and prints the same line shape.

`--dump-outputs DIR` (rank 0) writes what the last timed step returned to its caller -- the all-gathered logits (B*N, W)
and is_true (B*N, 1) -- as DIR/logits.npy and DIR/is_true.npy (float32).  Inputs and weights come from fixed seeds, so
two builds run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import faulthandler
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "query windows/sec (5-way 1-shot, T=16)"
UNIT = "windows/s"
WINDOWS_PER_GPU = 4096
WAY, T, J3, N_TUP, D, F = 5, 16, 90, 120, 128, 256
# SURVEY.md 8(d): algorithmic work per query window
ATTN_FLOP_PER_WINDOW = 4 * WAY * N_TUP * N_TUP * D          # 36.86 MFLOP
MLP_FLOP_PER_WINDOW = 2 * T * (90 * 180 + 180 * 256)         # 1.993 MFLOP
PROJ_FLOP_PER_WINDOW = 4 * T * F * 2 * D                     # 4.19 MFLOP (factorised per-frame projection)
HEAD_FLOP_PER_WINDOW = 2 * (N_TUP * D * T + N_TUP * T * 256 + 256 * 64 + 64)   # 1.507 MFLOP


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"hbm_gbs": d["hbm_gbs"], "bf16_tflops": d["bf16_tflops"],
                "bf16_tflops_sustained": d.get("bf16_tflops_sustained", d["bf16_tflops"]), "source": "measured"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback (B200_PROFILING.md)"}


class ClockSampler:
    """Samples SM clock, power and throttle reasons during a timed region (NVML; nvidia-smi fields equivalent)."""

    def __init__(self, index):
        self.samples, self.power, self.reasons, self.max_mhz = [], [], set(), None
        self._stop = threading.Event()
        self._t = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def _run(self):
        nv = self.nv
        names = {"hw_slowdown": 0x8, "sw_power_cap": 0x4, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20,
                 "hw_power_brake_slowdown": 0x80}
        while not self._stop.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                self.power.append(nv.nvmlDeviceGetPowerUsage(self.h) / 1000.0)
                r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h) if hasattr(nv, "nvmlDeviceGetCurrentClocksEventReasons") \
                    else nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for k, bit in names.items():
                    if r & bit:
                        self.reasons.add(k)
            except Exception:
                pass
            time.sleep(0.002)

    def start(self):
        if self.nv is not None:
            self._t = threading.Thread(target=self._run, daemon=True)
            self._t.start()
        return self

    def stop(self):
        self._stop.set()
        if self._t:
            self._t.join()
        s = sorted(self.samples)
        med = s[len(s) // 2] if s else None
        return {"sm_mhz": med, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": len(s),
                "power_w_max": max(self.power) if self.power else None}


def ncu_dram_bytes():
    """{kernel substring: DRAM bytes per launch} from the committed ncu --set full captures (profiles/, newest round first)."""
    out = {}
    for name in ("r02_ncu_full_summary.json", "r01_ncu_full_summary.json"):
        p = os.path.join(ROOT, "profiles", name)
        try:
            scale = {"Mbyte": 1e6, "Kbyte": 1e3, "Gbyte": 1e9, "byte": 1.0}
            for d in json.load(open(p)):
                k = d["Kernel Name"]
                if k in out:
                    continue
                rd = float(d["dram__bytes_read.sum"]) * scale[d["units"]["dram__bytes_read.sum"]]
                wr = float(d["dram__bytes_write.sum"]) * scale[d["units"]["dram__bytes_write.sum"]]
                out[k] = rd + wr
        except Exception:
            continue
        if out:
            break          # ONE capture only: the same kernel is spelled differently by different ncu versions and would be counted twice
    return out


def ncu_lookup(table, *subs):
    tot, hit = 0.0, False
    for k, v in table.items():
        if any(s in k for s in subs):
            tot += v
            hit = True
    return tot if hit else None


class CpuArm:
    """The reference's CPU implementation of the path: oracle/_ref (unmodified reference) when staged, else the port."""

    def __init__(self, cfg, sd, threads):
        import torch
        torch.set_num_threads(threads)
        self.threads = threads
        from oracle import ref_runner
        if ref_runner.available():
            self.kind = "reference"
            self.impl = ref_runner.ReferenceScorer(cfg, sd, threads)
            self.what = "unmodified reference TRXOS.forward (oracle/_ref), torch CPU fp32"
        else:
            from oracle.trx_oracle import TrxOracle
            self.kind = "port"
            self.impl = TrxOracle(cfg, sd)
            self.what = "oracle port (torch CPU fp32)"

    def prepare(self, support):
        import torch
        self.ssf = self.impl.embed(torch.from_numpy(support)) if self.kind == "port" else self.impl.embed(support)

    def score(self, labels, q, chunk=512):
        return self.impl.score(None, labels, q, chunk=chunk, ss_features=self.ssf)


def cpu_baseline(cfg, sd, support, labels, query, seconds, threads):
    arm = CpuArm(cfg, sd, threads)
    arm.prepare(support)
    arm.score(labels, query[:64])                                  # warm-up
    chunk = 512
    done, t0 = 0, time.perf_counter()
    while True:
        s = done % query.shape[0]
        q = query[s:s + chunk]
        arm.score(labels, q, chunk=chunk)
        done += q.shape[0]
        el = time.perf_counter() - t0
        if el >= seconds or done >= 4 * query.shape[0]:
            break
    return {"value": done / el, "unit": UNIT, "cores": threads, "kind": arm.kind,
            "sample": f"{done} of the step's windows in {el:.1f} s, {arm.what}, {threads} threads"}


def run_reference(args):
    """--impl reference: the reference's own CPU implementation of the path on the box's host cores."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle.synth import Cfg, make_episode, make_state_dict
    cfg = Cfg()
    sd = make_state_dict(cfg, 0)
    support, labels, query, _ = make_episode(cfg, WINDOWS_PER_GPU, 1, "structured")
    threads = os.cpu_count() or 1
    arm = CpuArm(cfg, sd, threads)
    arm.prepare(support)
    sample = 1024                                                            # windows per step (bounded sample)
    for _ in range(max(1, args.warmup)):
        arm.score(labels, query[:256], chunk=256)
    t0 = time.perf_counter()
    for k in range(args.steps):
        s = (k * sample) % WINDOWS_PER_GPU
        arm.score(labels, query[s:s + sample], chunk=512)
    el = time.perf_counter() - t0
    val = args.steps * sample / el
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * el / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": "cfg2: 5-way 1-shot, T=16, J=30, pair tuples (N=120); each step scores a bounded "
                                   f"sample of {sample} of the {WINDOWS_PER_GPU} query windows on the host CPU"},
            "cpu_baseline": {"value": val, "unit": UNIT, "cores": threads, "kind": arm.kind,
                             "sample": f"{args.steps} steps x {sample} windows, {arm.what}, {threads} threads"},
            "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


def teardown(torch, dist, world, graphs=(), models=()):
    """Ends a run whose result line is printed: destroys the CUDA graphs (before the communicator: they captured NCCL
    kernels) and the library handles (arx_destroy synchronises the device), then the process group, and returns, so the
    process exits normally and its exit handlers run.  A hang must not turn the finished measurement into a timeout:
    - during these steps (seen once: destroy_process_group never returned after graph replays) a timer thread ends the
      process with exit code 0 after 20 s;
    - during interpreter finalization a daemon thread can no longer run, so faulthandler's watchdog (a C thread) covers
      it: after a further 30 s it prints every thread's stack to stderr and ends the process with exit code 1."""
    sys.stdout.flush()
    # (at N=1 too: one default run of round 2 printed its line and then never exited -- seen once in ~10 runs, not reproduced
    # under faulthandler; whatever finaliser it was, the measurement was complete)
    t = threading.Timer(20.0, lambda: os._exit(0))
    t.daemon = True
    t.start()
    for g in graphs:
        try:
            g.reset()
        except Exception:
            pass
    for m in models:
        try:
            m._release()
        except Exception:
            pass
    try:
        torch.cuda.synchronize()
    except Exception:
        pass
    if world > 1:
        try:
            dist.barrier()
            dist.destroy_process_group()
        except Exception:
            pass
    t.cancel()
    faulthandler.dump_traceback_later(30.0, exit=True)
    sys.stdout.flush()
    sys.stderr.flush()


# ----------------------------------------------------------------------------------------------------------------------
def timed_ms(torch, fn, reps, warm=2):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps


DUMP_BYTES = 64 << 20


def dump_outputs(d, per_rank):
    """--dump-outputs: the last step's per-rank (logits, is_true) as d/logits.npy and d/is_true.npy, rows of all ranks in
    rank order, float32.  Beyond DUMP_BYTES in all, both keep the same fixed, seeded sample of rows (in row order)."""
    import numpy as np
    import torch
    arrays = {"logits": torch.cat([r[0] for r in per_rank]).cpu().numpy(),
              "is_true": torch.cat([r[1] for r in per_rank]).cpu().numpy()}
    n = arrays["logits"].shape[0]
    row_bytes = 4 * sum(a.shape[1] for a in arrays.values())
    if n * row_bytes > DUMP_BYTES:
        keep = np.sort(np.random.default_rng(0).choice(n, DUMP_BYTES // row_bytes, replace=False))
        arrays = {k: a[keep] for k, a in arrays.items()}
    os.makedirs(d, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(d, k + ".npy"), np.ascontiguousarray(a, dtype=np.float32))


def other_configs(torch, dev, peaks):
    """BASELINE cfg3 (one GPU, all 65 536 windows), cfg4 (T=32 pairs / triples), cfg5 (decode) and the streaming
    per-frame latency, each device-timed after warm-up on an explicit stream.  Rank 0, N=1 only."""
    import numpy as np
    from oracle.synth import Cfg, make_episode, make_heatmaps, make_state_dict
    from tests.util import Args, make_model, torch_sd
    out = {}

    def guard(name, fn):
        try:
            out[name] = fn()
        except Exception as e:                       # a secondary measurement must never take the headline line down
            out[name] = {"error": repr(e)[:300]}
        torch.cuda.synchronize()

    def cfg3():
        cfg = Cfg(way=60)
        m, _ = make_model(cfg, 0)
        B = 65536
        support, _, query, planted = make_episode(cfg, B, 61, "structured")
        m.set_support(poses=torch.from_numpy(support[0]).to(dev))
        Q = torch.from_numpy(query).to(dev)
        res = (torch.empty((B, 60), device=dev), torch.empty((B, 1), device=dev))
        ms = timed_ms(torch, lambda: m.score(Q, out=res), 3, warm=1)
        ok = bool((res[0].argmax(1).cpu().numpy() == planted).all())
        tf = 4 * 60 * N_TUP * N_TUP * D * B / ms / 1e9
        return {"workload": "60-way x 65536 windows, T=16 pairs, one GPU", "ms": ms, "windows_per_s": B / ms * 1e3, "path": m.last_path(),
                "attention_tflops_whole_score": tf, "frac_of_bf16_burst_whole_score": tf / peaks["bf16_tflops"], "planted_class_recovered": ok}

    def cfg4():
        cfg = Cfg(way=20, seq_len=32, temp_set=[2, 3])
        m, _ = make_model(cfg, 0)
        B = 2048
        support, _, query, planted = make_episode(cfg, B, 71, "structured")
        m.set_support(poses=torch.from_numpy(support[0]).to(dev))
        Q = torch.from_numpy(query).to(dev)
        ms = timed_ms(torch, lambda: m.score(Q), 3, warm=1)
        lg, _ = m.score(Q)
        r = {"pairs": {"workload": f"20-way, T=32, pair tuples N=496, {B} windows (logits + is_true)", "ms": ms, "windows_per_s": B / ms * 1e3,
                       "path": m.last_path(), "attention_tflops_whole_score": 4 * 20 * 496 * 496 * D * B / ms / 1e9,
                       "planted_class_recovered": bool((lg.argmax(1).cpu().numpy() == planted).all())}}
        Bt = 37
        qf = m.embed(Q[:Bt])
        ms = timed_ms(torch, lambda: m.score_features(1, qf), 2, warm=1)
        lt = m.score_features(1, qf)
        r["triples"] = {"workload": f"20-way, T=32, triple tuples N=4960, {Bt} windows (transformers[1] logits)", "ms": ms,
                        "windows_per_s": Bt / ms * 1e3, "path": m.last_path(), "attention_tflops_whole_score": 4 * 20 * 4960 * 4960 * D * Bt / ms / 1e9,
                        "planted_class_recovered": bool((lt.argmax(1).cpu().numpy() == planted[:Bt]).all())}
        for v in r.values():
            v["frac_of_bf16_burst_whole_score"] = v["attention_tflops_whole_score"] / peaks["bf16_tflops"]
        return r

    def cfg5():
        from isbfsar_b200 import HeatmapDecoder
        g = np.load(os.path.join(ROOT, "tests", "golden", "decode_64.npz"))
        cfg = Cfg()
        m, _ = make_model(cfg, 0)
        dec = HeatmapDecoder(m, g["expand30"], None, g["new_K"], g["homo_inv"])
        nfr = 1024
        hm = torch.from_numpy(make_heatmaps(nfr, seed=2)).to(dev)
        big = torch.cat([hm] * 4)                                          # 302 MB > L2: the decode kernel alone, HBM-resident input
        ms_dec = timed_ms(torch, lambda: dec.decode(big), 10)
        poses, valid = dec.decode(hm)
        support = poses.unfold(0, 16, 1).permute(0, 2, 1)[[0, 200, 400, 600, 800]].contiguous()
        m.set_support(poses=support)

        def e2e():
            p, _ = dec.decode(hm)
            return m.score_frames(p)                                     # 1009 sliding windows formed on the device
        ms = timed_ms(torch, e2e, 10)

        def e2e_windows():
            p, _ = dec.decode(hm)
            return m.score(p.unfold(0, 16, 1).permute(0, 2, 1).contiguous())
        ms_w = timed_ms(torch, e2e_windows, 10)
        by = 4 * nfr * (73728 + 360)
        return {"decode_kernel": {"workload": "4096 frames (8,8,288) fp32 -> 30-joint poses", "ms": ms_dec, "frames_per_s": 4 * nfr / ms_dec * 1e3,
                                  "achieved_gbs": by / ms_dec / 1e6, "frac_of_hbm": by / ms_dec / 1e6 / peaks["hbm_gbs"], "bound": "hbm",
                                  "algorithmic_bytes_per_frame": 73728 + 360},
                "end_to_end": {"workload": "1024 heatmap frames -> decode -> 1009 sliding windows (frame-stream form: every frame embedded "
                                           "once, windows formed on the device) -> 5-way scoring", "ms": ms, "frames_per_s": nfr / ms * 1e3,
                               "valid_frames": int(valid.sum()), "ms_with_explicit_windows": ms_w}}

    def stream():
        from isbfsar_b200 import ActionRecognizer
        cfg = Cfg()
        ar = ActionRecognizer(Args(cfg), state_dict=torch_sd(make_state_dict(cfg, 0)))
        rng = np.random.default_rng(7)
        for n in "abcde":
            ar.train({"flag": n, "data": {"poses": (0.17 * rng.standard_normal((16, 90))).astype(np.float32)}, "requires_focus": False})
        frames = (0.17 * rng.standard_normal((500, 90))).astype(np.float32)
        for f in range(100):
            ar.inference({"sk": frames[f]})
        torch.cuda.synchronize()
        t = []
        for f in range(100, 500):
            t0 = time.perf_counter()
            ar.inference({"sk": frames[f]})
            t.append(time.perf_counter() - t0)
        t = np.array(t) * 1e6
        return {"workload": "ActionRecognizer.inference, one camera frame per call, 5 classes (ar.py:30-84)",
                "us_per_frame_median": float(np.median(t)), "us_per_frame_p90": float(np.percentile(t, 90)), "frames": len(t)}

    guard("cfg3_one_gpu", cfg3)
    guard("cfg4", cfg4)
    guard("cfg5", cfg5)
    guard("stream", stream)
    return out


def cfg3_sharded(torch, dist, dev, world, rank, steps):
    """BASELINE cfg3: 60-way x 65 536 windows split contiguously over the ranks.  Every step: rank 0 processes the support
    set, NCCL-broadcasts the support tuple embeddings, every rank scores its shard, the scores are all-gathered."""
    import numpy as np
    from oracle.synth import Cfg, make_episode
    from tests.util import make_model
    from isbfsar_b200.dist import ScoreGatherer, broadcast_support, shard_bounds
    cfg = Cfg(way=60)
    B = 65536
    m, sd = make_model(cfg, 0)
    support, labels, query, planted = make_episode(cfg, B, 61, "structured")
    s, e = shard_bounds(B, world, rank)
    Q = torch.from_numpy(query[s:e]).to(dev)
    S = torch.from_numpy(support[0]).to(dev)
    gat = ScoreGatherer(e - s, 60, True, dev, depth=1)

    def step():
        if rank == 0:
            m.set_support(poses=S)
        if world > 1:
            broadcast_support(m, 60, src=0, device=dev)
            torch.cuda.current_stream().wait_stream(_comm_stream(dev))
        m.score(Q, out=gat.out())
        return gat.gather()

    def _comm_stream(d):
        from isbfsar_b200 import dist as D_
        return D_._comm_streams[torch.device(d)]

    for _ in range(2):
        res = step()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(steps):
        res = step()
    b.record()
    torch.cuda.synchronize()
    ms = a.elapsed_time(b) / steps
    t = torch.tensor([ms], dtype=torch.float64, device=dev)
    # every rank must hold the SAME gathered scores (bit equality through a checksum of the raw bits) and they must be right
    full = torch.cat([r[0] for r in res])
    chk = full.view(torch.int32).to(torch.int64).sum().reshape(1)
    agree = True
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        lo_, hi_ = chk.clone(), chk.clone()
        dist.all_reduce(lo_, op=dist.ReduceOp.MIN)
        dist.all_reduce(hi_, op=dist.ReduceOp.MAX)
        agree = bool((lo_ == hi_).item())
    ok = bool((full.argmax(1).cpu().numpy() == planted).all())
    ms = float(t[0])
    tf = 4 * 60 * N_TUP * N_TUP * D * B / ms / 1e9
    return {"workload": f"60-way x 65536 windows, T=16 pairs, split contiguously over {world} rank(s); every step: support set on rank 0, NCCL "
                        "broadcast of the support tuple embeddings, shard scoring, all-gather of [logits | is_true]",
            "metric": "query windows/sec (60-way 1-shot, T=16)", "value": B / ms * 1e3, "ms_per_step": ms, "steps": steps, "scaling": "strong",
            "attention_tflops_aggregate": tf, "gathered_scores_bit_identical_on_all_ranks": agree, "planted_class_recovered": ok}, res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="cfg2", choices=["cfg2", "cfg3"])
    ap.add_argument("--windows", type=int, default=WINDOWS_PER_GPU, help="query windows per GPU per step")
    ap.add_argument("--force-path", type=int, default=0, help="0 auto, 1 fp32 kernels, 2 tcgen05 kernels")
    ap.add_argument("--chunk", type=int, default=0, help="windows per internal pass of arx_score (0 = library default)")
    ap.add_argument("--cpu-seconds", type=float, default=12.0)
    ap.add_argument("--sustained-seconds", type=float, default=2.0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip sustained / other configs / cfg3 (headline numbers only)")
    ap.add_argument("--no-step-graph", action="store_true", help="launch every step eagerly instead of replaying one CUDA graph per step")
    ap.add_argument("--static-support", action="store_true",
                    help="diagnostic: set the support set once before timing instead of in every step")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the last timed step's logits / is_true as DIR/<name>.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3)
    if args.impl == "reference":
        return run_reference(args)

    import numpy as np
    import torch
    import torch.distributed as dist
    from oracle.synth import Cfg, make_episode, make_state_dict
    from tests.util import make_model
    from isbfsar_b200.dist import ScoreGatherer, broadcast_support

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}: launch with torch.distributed.run for N>1")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        # the only collective in a step is a 24-byte-per-window all-gather: keep NCCL's footprint to a couple of CTAs
        os.environ.setdefault("NCCL_MAX_NCHANNELS", "2")
        os.environ.setdefault("TORCH_NCCL_HIGH_PRIORITY", "1")
        dist.init_process_group("nccl", device_id=dev)
    peaks = measured_peaks()

    if args.config == "cfg3":
        torch.cuda.set_stream(torch.cuda.Stream(device=dev))
        sampler = ClockSampler(local).start() if rank == 0 else None
        r, res = cfg3_sharded(torch, dist, dev, world, rank, args.steps)
        if rank == 0 and args.dump_outputs:
            dump_outputs(args.dump_outputs, res)
        if rank == 0:
            line = {"metric": r["metric"], "value": r["value"], "unit": UNIT, "n_gpus": world, "steps": r["steps"], "warmup": 2,
                    "ms_per_step": r["ms_per_step"], "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f16",
                    "data": "synthetic", "config": {"workload": "cfg3: " + r["workload"]}, "clocks": sampler.stop(), "cfg3": r}
            print(json.dumps(line), flush=True)
        teardown(torch, dist, world)
        return

    cfg = Cfg()
    B = args.windows
    model, sd = make_model(cfg, 0, force_path=args.force_path, max_chunk=args.chunk)
    support, labels, query, planted = make_episode(cfg, B, 1 + rank, "structured")
    # every rank scores ITS OWN B windows (weak scaling); the support set is rank 0's
    support0 = make_episode(cfg, 1, 1, "structured")[0]
    q_dev = torch.from_numpy(query).to(dev)
    q_pin = torch.from_numpy(query).pin_memory()
    s_dev = torch.from_numpy(support0[0]).to(dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)           # > 126 MB L2

    # everything below runs on an explicit stream: the legacy default stream cannot be captured
    stream = torch.cuda.Stream(device=dev)
    torch.cuda.set_stream(stream)
    gatherer = ScoreGatherer(B, WAY, True, dev, depth=2)
    in_flight = []

    def step_eager():
        # every rank processes the (replicated) support poses itself -- asynchronously on the scorer's side stream --
        # scores its own shard, and the scores are all-gathered (one NCCL call per batch).  The collective of batch k runs
        # on a communication stream and is joined after batch k+1 has been scored; `drain()` joins the last one.
        if not args.static_support:
            model.set_support(poses=s_dev)
        model.score(q_dev, out=gatherer.out())
        in_flight.append(gatherer.gather_async())
        return gatherer.wait(in_flight.pop(0)) if len(in_flight) > 1 else None

    def drain():
        res = None
        while in_flight:
            res = gatherer.wait(in_flight.pop(0))
        return res

    # once, before timing (north_star: "broadcast the support-set tuple embeddings once"): rank 0 processes the support
    # set and NCCL-broadcasts the tuple embeddings; the other ranks import them and must reproduce their own local result
    model.set_support(poses=s_dev)
    ref_logits, ref_true = model.score(q_dev)
    if world > 1:
        broadcast_support(model, WAY, src=0, device=dev)
        torch.cuda.synchronize()
        got_logits, got_true = model.score(q_dev)
        if not (torch.equal(got_logits, ref_logits) and torch.equal(got_true, ref_true)):
            raise SystemExit("bench: scores with NCCL-broadcast support embeddings differ from locally computed ones")
        model.set_support(poses=s_dev)

    # correctness guard on the exact tensors being timed (oracle = checker only, small subset)
    step_eager()
    per_rank = drain()
    torch.cuda.synchronize()
    logits = per_rank[rank][0]
    mine = logits[:32].cpu().numpy()
    from oracle.trx_oracle import TrxOracle
    lo, it = TrxOracle(cfg, sd).score(support0, labels, query[:32])
    err = float(np.abs(mine / lo - 1).max())
    if not err < 1e-3:
        raise SystemExit(f"bench: parity check failed before timing (max rel err {err:.3e})")

    # ---- the step as ONE CUDA graph (set_support + score + all-gather): a step costs the host one graph launch, which is
    # what keeps 8 ranks sharing the box's cores in step; the library's own kernels are captured as plain launches
    # (arx_score notices the capture), the support chain's side stream forks and joins inside the graph.
    graph_steps = [None, None]
    launches_per_graph = 0
    gats = [ScoreGatherer(B, WAY, True, dev, depth=1) for _ in range(2)]
    comm_stream = torch.cuda.Stream(device=dev)
    step_no = [0]
    if not args.no_step_graph:
        try:
            def body(i):
                # graph i scores into buffer set i; the all-gather of the OTHER set (filled by the previous step) runs on a forked
                # branch beside this step's kernels, so the collective is off the critical path; the last one is done eagerly
                if world > 1:
                    comm_stream.wait_stream(torch.cuda.current_stream())
                    with torch.cuda.stream(comm_stream):
                        gats[1 - i].gather()
                if not args.static_support:
                    model.set_support(poses=s_dev)
                model.score(q_dev, out=gats[i].out())
                if world > 1:
                    torch.cuda.current_stream().wait_stream(comm_stream)
            for _ in range(2):                       # warm-up of exactly this call sequence (allocations, one-time inits, NCCL)
                body(0)
                body(1)
            torch.cuda.synchronize()
            for i in range(2):
                l0 = model.launch_count()
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g, stream=stream, capture_error_mode="thread_local"):
                    body(i)
                launches_per_graph = model.launch_count() - l0
                graph_steps[i] = g
            for i in range(2):
                graph_steps[i].replay()
            gats[1].gather()
            torch.cuda.synchronize()
            for i in range(2):
                res = gats[i]._result(0)[rank]
                if not (torch.equal(res[0], ref_logits) and torch.equal(res[1], ref_true)):
                    raise RuntimeError("graph replay does not reproduce the eager scores")
        except Exception as e:                           # never lose the run over the launch mode
            sys.stderr.write(f"bench: whole-step graphs unavailable ({e!r}); steps are launched eagerly\n")
            for g in graph_steps:
                try:
                    if g is not None:
                        g.reset()
                except Exception:
                    pass
            graph_steps = [None, None]
            try:
                torch.cuda.synchronize()
            except Exception:
                pass
    use_graph = graph_steps[0] is not None and graph_steps[1] is not None
    if world > 1:                                        # every rank must take the same mode: the collective sequence differs
        ok = torch.tensor([1 if use_graph else 0], device=dev)
        dist.all_reduce(ok, op=dist.ReduceOp.MIN)
        use_graph = int(ok.item()) == 1

    def step():
        if use_graph:
            graph_steps[step_no[0] & 1].replay()
            step_no[0] += 1
        else:
            step_eager()

    def finish():
        """Joins the last step; -> its per-rank (logits, is_true), as the caller of the step receives them."""
        if use_graph:
            # the last step's scores (every earlier gather rode inside the next graph; no collective at N=1)
            return gats[(step_no[0] - 1) & 1].gather()
        return drain()

    for _ in range(args.warmup):
        flush.fill_(1)
        step()
    finish()
    torch.cuda.synchronize()

    def timed_block(K):
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(K)]
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        for k in range(K):
            flush.fill_(k & 0xFF)                       # L2 flush between timed iterations (outside the events)
            ev[k][0].record()
            step()
            if k == K - 1:
                last = finish()                         # eager mode: the last collective is joined inside the last timed interval
            ev[k][1].record()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        return sum(a.elapsed_time(b) for a, b in ev), last

    sampler = ClockSampler(local)
    if rank == 0:            # one sampler per job: the ranks share few host cores
        sampler.start()
    l0 = model.launch_count()
    total_ms, last = timed_block(args.steps)
    n_steps_total = args.steps
    launches = (model.launch_count() - l0) + (launches_per_graph * n_steps_total if use_graph else 0)
    clocks = sampler.stop()
    if rank == 0 and args.dump_outputs:
        dump_outputs(args.dump_outputs, last)

    # ---- stage timers: the same steps launched eagerly with CUDA events between the stages (arx_profile_*)
    model.profile(True)
    model.profile_read(reset=True)
    for k in range(args.steps):
        flush.fill_(k & 0xFF)
        step_eager()
    drain()
    torch.cuda.synchronize()
    stage_ms, chunks = model.profile_read(reset=True)
    model.profile(False)
    stage_ms = {k: v / max(1, args.steps) for k, v in stage_ms.items()}

    # ---- sustained: >= 2 s of back-to-back steps over a ring of 8 input batches (189 MB > L2), no flush, clocks sampled
    sustained = None
    if not args.no_extras:
        ring = [torch.from_numpy(np.roll(query, 7 * i, axis=0)).to(dev) for i in range(8)]
        outs_r = (torch.empty((B, WAY), device=dev), torch.empty((B, 1), device=dev))

        def sstep(i):
            if not args.static_support:
                model.set_support(poses=s_dev)
            model.score(ring[i & 7], out=outs_r)
        for i in range(24):
            sstep(i)
        torch.cuda.synchronize()
        per = timed_ms(torch, lambda: sstep(0), 16, warm=0)
        n_s = max(64, int(args.sustained_seconds * 1e3 / per))
        smp = ClockSampler(local)
        if rank == 0:
            smp.start()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for i in range(n_s):
            sstep(i)
        b.record()
        torch.cuda.synchronize()
        s_ms = a.elapsed_time(b)
        s_clk = smp.stop()
        # the same loop with the stage timers armed (kernels launched one by one): attention time at sustained clocks
        model.profile(True)
        model.profile_read(reset=True)
        n_p = max(32, n_s // 2)
        smp2 = ClockSampler(local)
        if rank == 0:
            smp2.start()
        for i in range(n_p):
            sstep(i)
        torch.cuda.synchronize()
        sst, _ = model.profile_read(reset=True)
        p_clk = smp2.stop()
        model.profile(False)
        attn_s = sst["cross_attention"] / n_p
        ach = B * ATTN_FLOP_PER_WINDOW / (attn_s * 1e-3) / 1e12 if attn_s > 0 else 0.0
        sustained = {"seconds": s_ms * 1e-3, "steps": n_s, "value": B * n_s / (s_ms * 1e-3), "unit": UNIT + " per GPU", "ms_per_step": s_ms / n_s,
                     "inputs": "ring of 8 batches (189 MB > 126 MB L2), no flush, one GPU's share of the job", "clocks": s_clk,
                     "attention": {"ms_per_launch": attn_s, "achieved_tflops": ach, "peak_tflops": peaks["bf16_tflops_sustained"],
                                   "frac": ach / peaks["bf16_tflops_sustained"], "peak_source": peaks["source"] + " bf16 sustained",
                                   "how": f"stage timers over {n_p} further back-to-back steps", "clocks": p_clk}}
        model.set_support(poses=s_dev)

    # ---- end to end through the host-buffer entry points: pinned H2D of the windows + D2H of the scores, every step.
    model.set_support(poses=s_dev)
    outs = [(torch.empty((B, WAY), dtype=torch.float32).pin_memory(), torch.empty((B, 1), dtype=torch.float32).pin_memory())
            for _ in range(3)]
    for _ in range(2):
        model.score_host(q_pin, out=outs[0])
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    e2e_steps = max(20, min(args.steps * 4, 200))
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        model.score_host(q_pin, out=outs[0])
    torch.cuda.synchronize()
    e2e_sync_s = time.perf_counter() - t0
    for k in range(2):
        model.score_host_async(q_pin, out=outs[k]).result()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    t0 = time.perf_counter()
    pending = []
    for k in range(e2e_steps):
        pending.append(model.score_host_async(q_pin, out=outs[k % 3]))
        if len(pending) == 2:
            pending.pop(0).result()
    for tk in pending:
        tk.result()
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    e2e_check = float((outs[(e2e_steps - 1) % 3][0] - ref_logits.cpu()).abs().max())
    # the same with fp16 host rows (arx_score_host_submit_f16): half the H2D bytes, for producers that emit fp16
    q_pin16 = torch.from_numpy(query).to(torch.float16).pin_memory()
    for k in range(6):
        model.score_host_async(q_pin16, out=outs[k % 3]).result()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    t0 = time.perf_counter()
    pending = []
    for k in range(e2e_steps):
        pending.append(model.score_host_async(q_pin16, out=outs[k % 3]))
        if len(pending) == 2:
            pending.pop(0).result()
    for tk in pending:
        tk.result()
    torch.cuda.synchronize()
    e2e16_s = time.perf_counter() - t0

    t = torch.tensor([total_ms, e2e_s, float(launches), e2e_sync_s, e2e16_s], dtype=torch.float64, device=dev)
    if world > 1:
        tmax = t.clone()
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        tsum = t.clone()
        dist.all_reduce(tsum, op=dist.ReduceOp.SUM)
        total_ms, e2e_s, launches, e2e_sync_s, e2e16_s = float(tmax[0]), float(tmax[1]), float(tsum[2]), float(tmax[3]), float(tmax[4])
    value = world * B * n_steps_total / (total_ms * 1e-3)
    e2e_val = world * B * e2e_steps / e2e_s

    cfg3 = None
    if not args.no_extras:
        try:
            cfg3, _ = cfg3_sharded(torch, dist, dev, world, rank, 5)
        except Exception as e:
            cfg3 = {"error": repr(e)[:300]}
            if world > 1:
                raise
        torch.cuda.synchronize()

    if rank == 0:
        path = model.last_path()
        ncu = ncu_dram_bytes()
        attn_ms = stage_ms["cross_attention"]
        achieved = B * ATTN_FLOP_PER_WINDOW / (attn_ms * 1e-3) / 1e12 if attn_ms > 0 else 0.0
        peak = peaks["bf16_tflops"]
        roofline = {"bound": "tensor", "kernel": "cross_attention k_attn_tc3 (tcgen05, fp16 operands / fp32 accumulate)", "achieved": achieved, "peak": peak,
                    "unit": "TFLOP/s", "frac": achieved / peak, "traffic": ncu_lookup(ncu, "k_attn_tc3") if B == WINDOWS_PER_GPU else None,
                    "traffic_unit": "bytes per launch (ncu --set full, profiles/)", "peak_source": peaks["source"] + " bf16 burst",
                    "algorithmic_flop_per_launch": B * ATTN_FLOP_PER_WINDOW, "ms_per_launch": attn_ms, "stage_ms_per_step": stage_ms}

        def hbm_row(name, stage, alg_bytes, moved_bytes, kernels, note):
            ms = stage_ms[stage]
            return {"kernel": name, "stage": stage, "bound": "hbm", "ms": ms, "algorithmic_bytes": alg_bytes, "moved_bytes": moved_bytes,
                    "achieved_gbs": alg_bytes / ms / 1e6 if ms > 0 else None, "achieved_gbs_moved": moved_bytes / ms / 1e6 if ms > 0 else None,
                    "peak_gbs": peaks["hbm_gbs"], "frac": alg_bytes / ms / 1e6 / peaks["hbm_gbs"] if ms > 0 else None,
                    "frac_moved": moved_bytes / ms / 1e6 / peaks["hbm_gbs"] if ms > 0 else None,
                    "dram_bytes_ncu": ncu_lookup(ncu, *kernels) if B == WINDOWS_PER_GPU else None, "note": note}
        rows = B * T
        per_kernel = [
            hbm_row("k1 frame MLP (k_mlp_p: poses -> fc1 -> fc2 -> feature image, one launch)", "embed_mlp", B * T * J3 * 4 + rows * F * 2,
                    rows * (J3 * 4 + 320 * 2), ("k_mlp_p",),
                    "algorithmic = fp32 poses in + fp16 features out; moved adds the one-hot positional sub-tile written beside the features "
                    "(round 2 until the fused kernel: three launches, 149 MB moved); the kernel is paced by its per-tile epilogue chain and "
                    "the 144 KB weight load per CTA, not by HBM (timeline trace, tools/trace_mlp.py)"),
            hbm_row("k3a per-frame K/V projection (k_gemm_p<256,F32C>)", "kv_projection", rows * (F * 2 + 4 * D * 4), rows * (320 * 2 + 4 * D * 4),
                    ("F32C",), "SURVEY 8d target: fused (0 bytes); as built the fp32 projections are materialised once"),
            hbm_row("k2 tuple gather + LayerNorm -> operand images (k_tuple_img)", "tuple_build_ln", B * 128 * 128 * 2, rows * 2 * D * 4 + B * 128 * 128 * 2,
                    ("k_tuple_img",), "SURVEY 8d target for k2 is 0 HBM bytes (fused into attention); algorithmic here = the operand image written"),
            {"kernel": "k3b cross-attention + distances (k_attn_tc3)", "stage": "cross_attention", "bound": "tensor", "ms": attn_ms,
             "algorithmic_flop": B * ATTN_FLOP_PER_WINDOW, "achieved_tflops": achieved, "peak_tflops": peak, "frac": achieved / peak,
             "dram_bytes_ncu": ncu_lookup(ncu, "k_attn_tc3") if B == WINDOWS_PER_GPU else None},
            hbm_row("k4 open-set head (k_head2_tc + fc1 + fc2/fc3/sigmoid + finish)", "open_set_head", B * (128 * 128 * 2 + N_TUP * T * 2 + (WAY + 1) * 4),
                    B * (128 * 128 * 2 + 2 * N_TUP * T * 2 + 256 * 2 * 2 + (WAY + 1) * 4), ("k_head2_tc", "k_finish", "SIGMOID", "IMG16, 4"),
                    "SURVEY 8d allows 'outputs only' when fused behind the attention; as built the winning class's tile is recomputed from the Kq image"),
        ]
        cpu = None
        if not args.no_cpu_baseline and world == 1:       # the CPU arm is timed at N=1 only (the other ranks' processes share the host cores)
            cpu = cpu_baseline(cfg, sd, support0, labels, query, args.cpu_seconds, os.cpu_count() or 1)
        extras = None
        if not args.no_extras and world == 1:
            extras = other_configs(torch, dev, peaks)
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": total_ms / n_steps_total, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "f16" if path >= 2 else "f32", "data": "synthetic",
                "config": {"workload": f"cfg2: {B} query windows per GPU x 5-way 1-shot, T=16, J=30, pair tuples (N=120); "
                                       + ("step = score shard + all-gather scores (support set processed once, --static-support)" if args.static_support
                                          else "step = process support set (every rank, replicated poses) + score shard + all-gather scores; "
                                               "NCCL broadcast of the support tuple embeddings done and verified once before timing"),
                           "l2": "flushed between timed steps (256 MiB write)", "path": path,
                           "launch": ("one CUDA graph per step (set_support + score; with N>1 the all-gather of the previous step's scores rides on a forked "
                                      "branch of the same graph, the last one is joined inside the last timed step)" if use_graph
                                      else "eager launches; the collective of batch k is joined after batch k+1 is scored"),
                           "timing": f"CUDA events per step on the launching stream, summed over exactly {args.steps} steps "
                                     "(bracketed by barrier + synchronize); max over ranks; stage timers from a further pass of the same "
                                     "steps launched eagerly with events between stages"},
                "timed_steps_total": n_steps_total, "timed_ms_total": total_ms,
                "clocks": clocks,
                "e2e": {"value": e2e_val, "unit": UNIT, "h2d_bytes_per_step": world * B * T * J3 * 4,
                        "d2h_bytes_per_step": world * B * (WAY + 1) * 4, "steps": e2e_steps,
                        "mode": "streaming: arx_score_host_submit/_wait, two requests in flight, pinned host buffers",
                        "blocking_value": world * B * e2e_steps / e2e_sync_s,
                        "blocking_mode": "one synchronous arx_score_host call at a time",
                        "f16_rows_value": world * B * e2e_steps / e2e16_s, "f16_rows_h2d_bytes_per_step": world * B * T * J3 * 2,
                        "f16_rows_mode": "streaming, host rows already fp16 (arx_score_host_submit_f16): bit-identical scores for fp16-representable inputs",
                        "max_abs_diff_vs_device_path": e2e_check,
                        "timing": "host wall clock from first submit to last result, max over ranks"},
                "gpu_launches": int(launches), "roofline": roofline, "roofline_per_kernel": per_kernel, "sustained": sustained,
                "cfg3": cfg3, "other_configs": extras, "cpu_baseline": cpu, "parity_check_max_rel_err": err}
        print(json.dumps(line), flush=True)
    teardown(torch, dist, world, [g for g in graph_steps if g is not None], [model])


if __name__ == "__main__":
    main()
