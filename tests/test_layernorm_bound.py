"""The tensor-core routes across the LayerNorm-affine range of norm_k, held to the float64 oracle.

Whether a transformer scores on tensor cores is decided from one number computed at weight load, the static softmax
bound |S| <= (max|gamma| sqrt(D) + ||beta||_2)^2 / sqrt(D) (arx_api.cu, arx_load_weights).  Two limits apply to it
(DESIGN 4):
  - overflow: |S| log2(e) < 100 keeps exp2 without max-subtraction inside fp32 range.  It picks the row-max variant of
    the tiled kernels and bounds what force_path = 2 may run on the kernels without it;
  - accuracy: |S| < ACCURACY_BOUND (ACCURACY_BOUND_FEW_TUPLES below 120 tuples, where a logit averages the operand
    rounding over fewer tuples) keeps the fp16 QK^T and bf16 P.V operands within the stated 1e-3 relative tolerance.
    It admits weights to the pair and tiled routes by default; past it they score on the fp32 kernels.
Both limits are mirrored here, so changing either in the C sources without these tests fails a test."""
import math
from math import comb

import numpy as np
import pytest
import torch

from oracle.synth import Cfg, make_episode, make_state_dict
from oracle.trx_oracle import TrxOracle
from tests.util import Args, rel_err, torch_sd

pytestmark = pytest.mark.gpu

D = 128
LOG2E = 1.4426950408889634                    # ARX_SOFTMAX_LOG2E
OVERFLOW_BOUND = 100.0 / LOG2E                # 69.3: |S| log2(e) < 100
ACCURACY_BOUND = 19.0                         # ARX_TC_ACCURACY_BOUND (arx_internal.cuh), set from profiles/r03_ln_bound_sweep.txt
ACCURACY_BOUND_FEW_TUPLES = 12.0              # ARX_TC_ACCURACY_BOUND_FEW_TUPLES, below FEW_TUPLES query tuples
FEW_TUPLES = 120                              # ARX_TC_FEW_TUPLES
TOL = 1e-3                                    # stated tolerance (BASELINE north star)
TOL_REDUCED = 3e-2                            # force_path = 2 past the accuracy bound

# route shape -> (config, windows, transformer scored); transformer 1 is scored through score_features(1, ...)
SHAPES = {
    "t16_pairs": (Cfg(), 256, 0),
    "t32_pairs": (Cfg(way=20, seq_len=32), 32, 0),
    "t8_pairs": (Cfg(seq_len=8), 256, 0),
    "t16_triples": (Cfg(temp_set=[2, 3]), 8, 1),
}
KINDS = ["structured", "iid", "support"]


def softmax_bound(g, b):
    """arx_load_weights: the bound in double, stored as float."""
    r = np.abs(np.asarray(g, np.float64)).max() * math.sqrt(D) + math.sqrt((np.asarray(b, np.float64) ** 2).sum())
    return float(np.float32(r * r / math.sqrt(D)))


def within_overflow(bound):
    return bool(np.float32(bound) * np.float32(LOG2E) < np.float32(100.0))


def accuracy_bound(shape):
    cfg, _, ti = SHAPES[shape]
    return ACCURACY_BOUND if comb(cfg.seq_len, cfg.temp_set[ti]) >= FEW_TUPLES else ACCURACY_BOUND_FEW_TUPLES


def within_accuracy(bound, shape):
    return bool(np.float32(bound) < np.float32(accuracy_bound(shape)))


def expected_path(shape, bound, force=0):
    """1 = fp32 kernels, 2 = T=16 pair pipeline, 3 = tiled kernels (arx_last_path)."""
    if force == 1 or (force == 0 and not within_accuracy(bound, shape)):
        return 1
    return 2 if shape == "t16_pairs" and within_overflow(bound) else 3


# ---- LayerNorm affines of norm_k: (gamma, beta) of D channels ---------------------------------------------------------
def uniform(bound):
    """gamma = const, beta = 0: the bound is gamma^2 sqrt(D), and a query equal to a support window reaches it."""
    return np.full(D, math.sqrt(bound / math.sqrt(D)), np.float32), np.zeros(D, np.float32)


def beta_dominated(bound, gamma=0.5, seed=3):
    """small gamma, ||beta||_2 makes up the rest of the bound; random signs"""
    bn = math.sqrt(bound * math.sqrt(D)) - gamma * math.sqrt(D)
    s = np.random.default_rng(seed).choice([-1.0, 1.0], D)
    return np.full(D, gamma, np.float32), (s * bn / math.sqrt(D)).astype(np.float32)


def per_channel(bound, seed=4):
    """gamma_d ~ U(0.5, 1) gmax with one channel at gmax, beta = 0"""
    g, b = uniform(bound)
    rng = np.random.default_rng(seed)
    g = (g * rng.uniform(0.5, 1.0, D)).astype(np.float32)
    g[rng.integers(D)] = uniform(bound)[0][0]
    return g, b


def golden_affine():
    """the draw of the cfg1_w5_t16_affine golden case: gamma ~ U(0.5, 1.5), beta ~ U(-0.2, 0.2)"""
    sd = make_state_dict(Cfg(), 0, affine_ln=True)
    return sd["transformers.0.norm_k.weight"], sd["transformers.0.norm_k.bias"]


# name -> affine, given the accuracy bound of the route shape
AFFINES = {
    "gamma1": lambda lim: uniform(math.sqrt(D)),
    "golden_affine": lambda lim: golden_affine(),
    "uniform_below": lambda lim: uniform(0.97 * lim),
    "uniform_above": lambda lim: uniform(1.03 * lim),
    "uniform_2.45": lambda lim: uniform(2.45 ** 2 * math.sqrt(D)),
    "beta_45": lambda lim: beta_dominated(45.0),
    "beta_68": lambda lim: beta_dominated(68.0),
    "per_channel": lambda lim: per_channel(0.97 * lim),
}


def ln_state_dict(cfg, g, b, wseed=0):
    """synthetic weights with the LayerNorm affine (g, b) on norm_k of every transformer"""
    sd = dict(make_state_dict(cfg, wseed))
    for i in range(len(cfg.temp_set)):
        sd[f"transformers.{i}.norm_k.weight"] = np.asarray(g, np.float32)
        sd[f"transformers.{i}.norm_k.bias"] = np.asarray(b, np.float32)
    return sd


def load_model(cfg, sd, force_path=0):
    from isbfsar_b200 import TRXOS
    m = TRXOS(Args(cfg))
    missing, unexpected = m.load_state_dict(torch_sd(sd), strict=False)
    assert not unexpected and all(k.startswith("post_resnet.") for k in missing), (missing, unexpected)
    m.force_path = force_path
    return m.cuda()


def episode(cfg, B, kind, seed=17):
    """support (1,W,T,90), labels, query (B,T,90); kind "support" queries the support windows themselves"""
    support, labels, query, planted = make_episode(cfg, B, seed, "iid" if kind == "iid" else "structured")
    if kind == "support":
        query = np.ascontiguousarray(support[0, planted])
    return support, labels, query


def reference(cfg, sd, ti, support, labels, query):
    """float64 oracle: logits (B,W) and, for transformer 0 of a DISC model, is_true (B,1)"""
    o = TrxOracle(cfg, sd, dtype=torch.float64)
    if ti == 0:
        return o.score(support, labels, query, chunk=64)
    with torch.no_grad():
        ssf = o.embed(torch.from_numpy(support).double())
        ref = o.cross_transformer(ssf.expand(query.shape[0], -1, -1, -1), torch.from_numpy(labels).long(),
                                  o.embed(torch.from_numpy(query).double()).unsqueeze(1), ti=ti)
    return ref["logits"].numpy(), None


def run(m, ti, support, query):
    m.set_support(poses=torch.from_numpy(support[0]).cuda())
    Q = torch.from_numpy(query).cuda()
    if ti == 0:
        logits, is_true = m.score(Q)
        return logits.cpu().numpy(), is_true.cpu().numpy()
    return m.score_features(ti, m.embed(Q)).cpu().numpy(), None


def check_parity(logits, is_true, lo, it, tol=TOL):
    """logits within tol; argmax wherever the float64 margin exceeds 2 tol; is_true on the windows whose winner agrees (a
    different winner is a different discriminator input), and accept / reject wherever is_true is farther than tol from
    the 0.5 threshold"""
    assert np.isfinite(logits).all()
    assert rel_err(logits, lo).max() < tol, rel_err(logits, lo).max()
    srt = np.sort(lo, 1)
    sure = (srt[:, -1] - srt[:, -2]) / np.abs(srt[:, -1]) > 2 * tol
    assert np.array_equal(logits.argmax(1)[sure], lo.argmax(1)[sure])
    if it is not None:
        same = logits.argmax(1) == lo.argmax(1)
        assert np.isfinite(is_true).all()
        assert rel_err(is_true[same], it[same]).max() < tol, rel_err(is_true[same], it[same]).max()
        clear = same[:, None] & (np.abs(it - 0.5) > tol * 0.5)
        assert np.array_equal(is_true[clear] > 0.5, it[clear] > 0.5)


def test_bound_constants():
    """The affines of the sweep sit where their names say, against both limits."""
    for shape in SHAPES:
        bounds = {k: softmax_bound(*f(accuracy_bound(shape))) for k, f in AFFINES.items()}
        assert abs(bounds["gamma1"] - math.sqrt(D)) < 1e-3 and within_accuracy(bounds["gamma1"], shape)
        assert 29.0 < bounds["golden_affine"] < 30.0
        assert abs(bounds["uniform_2.45"] - 67.9) < 0.1 and within_overflow(bounds["uniform_2.45"])
        assert abs(bounds["beta_45"] - 45.0) < 0.01 and abs(bounds["beta_68"] - 68.0) < 0.01
        assert within_accuracy(bounds["uniform_below"], shape) and within_accuracy(bounds["per_channel"], shape)
        assert not within_accuracy(bounds["uniform_above"], shape)
    assert accuracy_bound("t8_pairs") == ACCURACY_BOUND_FEW_TUPLES and accuracy_bound("t16_triples") == ACCURACY_BOUND
    assert ACCURACY_BOUND < OVERFLOW_BOUND


# ---- a. parity sweep: every route shape, every affine, three kinds of query --------------------------------------------
@pytest.mark.parametrize("affine", list(AFFINES))
@pytest.mark.parametrize("shape", list(SHAPES))
def test_parity_against_float64(shape, affine):
    cfg, B, ti = SHAPES[shape]
    g, b = AFFINES[affine](accuracy_bound(shape))
    bound = softmax_bound(g, b)
    sd = ln_state_dict(cfg, g, b)
    m = load_model(cfg, sd)
    for kind in KINDS:
        support, labels, query = episode(cfg, B, kind)
        logits, is_true = run(m, ti, support, query)
        lo, it = reference(cfg, sd, ti, support, labels, query)
        check_parity(logits, is_true, lo, it)
        assert m.last_path() == expected_path(shape, bound), (kind, bound, m.last_path())


# ---- b. every entry point inside the band [accuracy bound, overflow bound) ---------------------------------------------
def test_entry_points_in_band(capfd):
    cfg = Cfg()
    g, b = uniform(0.5 * (ACCURACY_BOUND + OVERFLOW_BOUND))
    bound = softmax_bound(g, b)
    assert not within_accuracy(bound, "t16_pairs") and within_overflow(bound)
    sd = ln_state_dict(cfg, g, b)
    o = TrxOracle(cfg, sd, dtype=torch.float64)
    m = load_model(cfg, sd)
    support, labels, query = episode(cfg, 96, "structured", seed=23)
    m.set_support(poses=torch.from_numpy(support[0]).cuda())
    lo, it = o.score(support, labels, query)

    logits, is_true = m.score(torch.from_numpy(query).cuda())
    assert m.last_path() == 1
    check_parity(logits.cpu().numpy(), is_true.cpu().numpy(), lo, it)

    hl, hi = m.score_host(torch.from_numpy(query).pin_memory())
    check_parity(hl.numpy(), hi.numpy(), lo, it)
    tickets = [m.score_host_async(torch.from_numpy(query[i::2].copy()).pin_memory()) for i in range(2)]
    for i, t in enumerate(tickets):
        al, ai = t.result()
        check_parity(al.numpy(), ai.numpy(), lo[i::2], it[i::2])

    frames = np.concatenate([query[0], query[1], query[2]])                       # 48 frames -> 33 windows
    fl, fi = m.score_frames(torch.from_numpy(frames).cuda())
    windows = np.stack([frames[i:i + 16] for i in range(33)])
    wl, wi = o.score(support, labels, windows)
    check_parity(fl.cpu().numpy(), fi.cpu().numpy(), wl, wi)

    rng = np.random.default_rng(29)
    sup_b = (0.17 * rng.standard_normal((6, 5, 16, 90))).astype(np.float32)
    q_b = (sup_b[np.arange(6), rng.integers(0, 5, 6)] + 0.05 * rng.standard_normal((6, 16, 90))).astype(np.float32)
    el, ei = m.score_episodes(torch.from_numpy(q_b).cuda(), poses=torch.from_numpy(sup_b).cuda())
    ref = o.forward({"sk": sup_b}, np.tile(np.arange(5), (6, 1)), {"sk": q_b})
    check_parity(el.cpu().numpy(), ei.cpu().numpy(), ref["logits"].numpy(), ref["is_true"].numpy())

    m.set_support(poses=torch.from_numpy(support[0]).cuda())
    with pytest.raises(ValueError):
        m.stream_push(frames[0])
    err = capfd.readouterr().err
    assert err.count("outside the fp16 tensor-core bound") == 1                  # said once per handle, not per call

    # the recogniser: the resident streaming path refuses these weights, ar.py falls back to the per-window path
    from isbfsar_b200 import ActionRecognizer
    ar = ActionRecognizer(Args(cfg), state_dict=torch_sd(sd))
    for i, n in enumerate(["a", "b", "c", "d", "e"]):
        ar.train({"flag": n, "data": {"poses": support[0, i]}, "requires_focus": False})
    got = []
    for f in frames[:20]:
        res, os_, _ = ar.inference({"sk": f})
        if res:
            got.append(np.concatenate([[res[k] for k in "abcde"], os_]))
    assert not ar._stream_ok and len(got) == 5
    rl, ri = o.score(support, labels, windows[:5])
    ref = np.concatenate([torch.softmax(torch.from_numpy(rl), 1).numpy(), ri], axis=1)
    assert rel_err(np.array(got), ref).max() < 2 * TOL                          # softmax of logits within 1e-3
    assert capfd.readouterr().err.count("outside the fp16 tensor-core bound") == 1


# ---- c. the overflow edge under force_path = 2 ------------------------------------------------------------------------
@pytest.mark.parametrize("poly", [0, 2])
@pytest.mark.parametrize("shape", ["t16_pairs", "t32_pairs"])
@pytest.mark.parametrize("scale", [0.995, 1.01])
def test_overflow_edge_forced(shape, scale, poly):
    """Queries equal to the support windows put the exp2 arguments at |S| log2(e) = 99.5 just inside the bound (no
    row max: T=16 pairs on the pair pipeline, T=32 on the tiled kernels without it) and past 100 just outside it (the
    tiled row-max variant).  Debug key 4 = 2 moves half the exponentials of the pair pipeline to the FMA-pipe
    polynomial, whose exponent shift-add holds for |x| < 100 only."""
    cfg, B, ti = SHAPES[shape]
    g, b = uniform(scale * OVERFLOW_BOUND)
    bound = softmax_bound(g, b)
    assert within_overflow(bound) == (scale < 1)
    sd = ln_state_dict(cfg, g, b)
    m = load_model(cfg, sd, force_path=2)
    if poly:
        m.debug_set(4, poly)
    support, labels, query = episode(cfg, min(B, 64), "support")
    logits, is_true = run(m, ti, support, query)
    assert m.last_path() == expected_path(shape, bound, force=2)
    lo, it = reference(cfg, sd, ti, support, labels, query)
    assert np.isfinite(logits).all() and np.isfinite(is_true).all()
    assert rel_err(logits, lo).max() < TOL_REDUCED
    assert np.array_equal(logits.argmax(1), lo.argmax(1))
    assert rel_err(is_true, it).max() < TOL_REDUCED


# ---- d. the accuracy bound: the route flips there, for every way of building the support operands -------------------
@pytest.mark.parametrize("shape", ["t16_pairs", "t32_pairs", "t8_pairs"])
@pytest.mark.parametrize("force", [0, 2])
@pytest.mark.parametrize("scale", [0.99, 1.01])
def test_route_flips_at_accuracy_bound(shape, force, scale):
    cfg, _, _ = SHAPES[shape]
    g, b = uniform(scale * accuracy_bound(shape))
    bound = softmax_bound(g, b)
    assert within_accuracy(bound, shape) == (scale < 1)
    sd = ln_state_dict(cfg, g, b)
    path = expected_path(shape, bound, force)
    assert path == ((2 if shape == "t16_pairs" else 3) if force == 2 or scale < 1 else 1)
    support, labels, query = episode(cfg, 16, "structured")
    lo, it = reference(cfg, sd, 0, support, labels, query)
    m = load_model(cfg, sd, force_path=force)
    Q = torch.from_numpy(query).cuda()
    m.set_support(poses=torch.from_numpy(support[0]).cuda())
    a = m.score(Q)
    assert m.last_path() == path
    m.set_support(features=m.embed(torch.from_numpy(support[0]).cuda()))
    f = m.score(Q)
    assert m.last_path() == path
    src = load_model(cfg, sd, force_path=1)                                       # the blob does not depend on the route
    src.set_support(poses=torch.from_numpy(support[0]).cuda())
    m2 = load_model(cfg, sd, force_path=force)
    m2.import_support(src.export_support(), cfg.way)
    i = m2.score(Q)
    assert m2.last_path() == path
    for logits, is_true in (a, f, i):
        check_parity(logits.cpu().numpy(), is_true.cpu().numpy(), lo, it)
