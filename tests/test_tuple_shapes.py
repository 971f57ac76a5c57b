"""Every sequence length and tuple cardinality arx_create accepts, against the float64 oracle.

arx_create takes seq_len T = 2..64 and temp_set entries c = 1..min(4, T), up to four transformers.  (T, c) picks the
kernels (DESIGN 6):
  T = 16, c = 2        the pair pipeline (path 2);
  other T, c = 2 or 3  the tiled any-N kernels (path 3), the open-set head with pair tuples up to T = 64;
  c = 1 or 4           the fp32 CUDA-core kernels (path 1): arx_tcn_supported is c in {2, 3};
  N = C(T, c) < 28     the fp32 CUDA-core kernels too (pairs up to T = 7, triples up to T = 6): ARX_TC_MIN_TUPLES.
The shapes below sit on the boundaries of the tiled kernels: tuple tiles of 128 (N = C(T, c) at 1..4 tiles and one
short of a tile), selection sub-tiles nsel = ceil(2cT / 64) (1 -> 2 at T = 17 pairs and T = 11 triples; 3, 4, 5, 6 at
T = 22, 33, 43, 54 triples), the head width K1 = N*T at every residue mod 4 (scalar head and tail of the streaming fc1),
windows that straddle 128-row front-end tiles (T not dividing 128) and N = 1 (T = 2 pairs, T = 3 triples, T = 4 with
c = 4).  Batches hold more than one 128-row tile of frames wherever the oracle allows it.

The oracle materialises B x N x N scores per class, so B, way and the oracle's windows per call are chosen to keep one
call under about 1 GB: triples past T = 40 are checked against the fp32 kernels (force_path = 1) instead."""
import itertools
import math

import numpy as np
import pytest
import torch

from oracle.synth import Cfg, make_episode
from oracle.trx_oracle import ActionRecognizerOracle, TrxOracle
from tests.util import Args, make_model, rel_err, torch_sd

pytestmark = pytest.mark.gpu

TOL = 1e-3                      # relative, logits and is_true, every route
TOL_PROBS = 2e-3                # softmax of logits held to TOL
NOTICE = "fp32 CUDA-core kernels"
# ARX_TC_MIN_TUPLES: with fewer query tuples nothing averages the rounding of the fp16 / bf16 operands, and the tiled route
# errs past TOL whatever the affine (1.05e-3 at N = 21, 2.5e-3 at N = 10, 1.3e-2 at N = 1 on a B200 at a 1000 W power
# limit, against 5.7e-4 at N = 36).  Those transformers score on the fp32 kernels.
MIN_TUPLES = 28

PAIR_T = [2, 3, 4, 5, 6, 7, 9, 12, 15, 17, 20, 23, 25, 31]      # N = 1, 3, 6, 10, 15, 21, 36, 66, 105, 136, 190, 253, 300, 465
TRIPLE_T = [3, 4, 5, 9, 10, 11, 13, 21, 22, 33, 40]             # N = 1, 4, 10, 84, 120, 165, 286, 1330, 1540, 5456, 9880
TRIPLE_T_FP32 = [43, 48, 64]                                    # N = 12341, 17296, 41664: too big for the oracle
C1_T = [2, 16, 32, 64]
C4_T = [4, 8, 16, 20]                                           # N = 1, 70, 1820, 4845


def expected_path(T, c):
    """the kernels arx_score takes for transformer cardinality c at sequence length T (default weights, J = 30)"""
    if c not in (2, 3) or math.comb(T, c) < MIN_TUPLES:
        return 1
    return 2 if (T == 16 and c == 2) else 3


def model_kind(c):
    """the discriminator is sized for pair tuples (model.py:282-285): other cardinalities score without it"""
    return "DISC" if c == 2 else "NONE"


def windows_for(T):
    """windows whose frame rows fill more than two 128-row tiles, the last one ragged"""
    return 300 // T + 1


def oracle_batch(T, c):
    """(way, windows, oracle windows per call) keeping one oracle call of C(T, c)^2 float64 scores under about 1 GB"""
    N = math.comb(T, c)
    if N <= 2000:                                                # at most 32 MB a window
        return 5, windows_for(T), windows_for(T)
    if N <= 6000:                                                # c = 4 at T = 20, triples at T = 33: 0.19 and 0.24 GB a window
        return 3, 4, 1
    return 2, 2, 1                                               # triples at T = 40: 0.78 GB a window


@pytest.fixture(scope="module")
def models():
    """(cfg, model, state dict, float64 oracle) per configuration, built once per module"""
    cache = {}

    def get(T, temp_set=(2,), model="DISC", way=5, max_chunk=0, force_path=0):
        key = (T, tuple(temp_set), model, way, max_chunk, force_path)
        if key not in cache:
            cfg = Cfg(way=way, seq_len=T, temp_set=list(temp_set), model=model)
            m, sd = make_model(cfg, 0, force_path=force_path, max_chunk=max_chunk)
            cache[key] = (cfg, m, sd, TrxOracle(cfg, sd, dtype=torch.float64))
        return cache[key]

    yield get
    cache.clear()


def check_oracle(lo, it, rl, ri, planted=None, tol=TOL):
    lo, rl = np.asarray(lo, dtype=np.float64), np.asarray(rl, dtype=np.float64)
    e = rel_err(lo, rl).max()
    assert e < tol, f"logits: max relative error {e:.3g}"
    if planted is not None:
        assert np.array_equal(rl.argmax(1), planted), "the oracle does not pick the planted class"
        assert np.array_equal(lo.argmax(1), planted)
    else:                       # argmax compared where the reference margin exceeds the tolerance twice over
        srt = np.sort(rl, 1)
        ok = (srt[:, -1] - srt[:, -2]) / np.abs(srt[:, -1]) > 2 * tol
        assert np.array_equal(lo.argmax(1)[ok], rl.argmax(1)[ok])
    assert (it is None) == (ri is None)
    if it is not None:
        it, ri = np.asarray(it, dtype=np.float64), np.asarray(ri, dtype=np.float64)
        e = rel_err(it, ri).max()
        assert e < TOL, f"is_true: max relative error {e:.3g}"
        assert np.array_equal(it > 0.5, ri > 0.5)


def cpu(x):
    return None if x is None else x.cpu()


def bit_equal(a, b):
    return all((x is None and y is None) or (x is not None and y is not None and torch.equal(x.cpu(), y.cpu())) for x, y in zip(a, b))


def scored(m, support, query):
    m.set_support(poses=torch.from_numpy(support[0]).cuda())
    return m.score(torch.from_numpy(query).cuda())


# ---- 1. the tuple table, every (T, c) --------------------------------------------------------------------------------------
@pytest.mark.parametrize("T", range(2, 65))
def test_tuple_table_matches_itertools(T):
    cs = list(range(1, min(4, T) + 1))
    m, _ = make_model(Cfg(seq_len=T, temp_set=cs, model="NONE"), 0)
    try:
        for ti, c in enumerate(cs):
            got = m.tuple_table(ti).cpu().numpy()
            ref = np.array(list(itertools.combinations(range(T), c)), dtype=np.int32).reshape(-1, c)
            assert got.shape == ref.shape and np.array_equal(got, ref), (T, c)
    finally:
        m._release()


# ---- 1b. the tuple count that admits the tensor-core routes -----------------------------------------------------------------
@pytest.mark.parametrize("T,c", [(7, 2), (8, 2), (6, 3), (7, 3)])      # N = 21, 28, 20, 35
def test_min_tuples_route(models, T, c, capfd):
    cfg, m, _, _ = models(T, (c,), model_kind(c))
    support, _, query, _ = make_episode(cfg, 4, 50 + T, "structured")
    scored(m, support, query)
    assert m.last_path() == (1 if math.comb(T, c) < MIN_TUPLES else 3)
    _, f, _, _ = models(T, (c,), model_kind(c), force_path=2)           # forced: the tiled kernels at any N
    scored(f, support, query)
    assert f.last_path() == 3
    assert NOTICE not in capfd.readouterr().err                          # no LayerNorm notice: the affine is not the reason


# ---- 2. pairs with the open-set head, T <= 32: TRXOS.forward from poses and from ss_features -------------------------------
@pytest.mark.parametrize("kind", ["structured", "iid"])
@pytest.mark.parametrize("T", PAIR_T)
def test_pairs_forward_matches_oracle(models, T, kind, capfd):
    cfg, m, _, o = models(T)
    support, labels, query, planted = make_episode(cfg, windows_for(T), 100 + T, kind)
    expect = planted if kind == "structured" else None
    S, L, Q = torch.from_numpy(support).cuda(), torch.from_numpy(labels).cuda(), torch.from_numpy(query).cuda()
    out = m({"sk": S}, L, {"sk": Q})
    assert m.last_path() == expected_path(T, 2)
    ref = o.forward({"sk": support}, labels, {"sk": query})
    check_oracle(cpu(out["logits"]), cpu(out["is_true"]), ref["logits"], ref["is_true"], expect)
    ssf = ref["support_features"].float()
    out2 = m(None, L, {"sk": Q}, ss_features=ssf.cuda())
    assert m.last_path() == expected_path(T, 2)
    ref2 = o.forward(None, labels, {"sk": query}, ss_features=ssf)
    check_oracle(cpu(out2["logits"]), cpu(out2["is_true"]), ref2["logits"], ref2["is_true"], expect)
    assert NOTICE not in capfd.readouterr().err


# ---- 3. triples: against the oracle, and past its reach against the fp32 kernels --------------------------------------------
@pytest.mark.parametrize("kind", ["structured", "iid"])
@pytest.mark.parametrize("T", TRIPLE_T)
def test_triples_match_oracle(models, T, kind, capfd):
    way, B, per_call = oracle_batch(T, 3)
    cfg, m, _, o = models(T, (3,), "NONE", way)
    support, labels, query, planted = make_episode(cfg, B, 200 + T, kind)
    lo, it = scored(m, support, query)
    assert it is None and m.last_path() == expected_path(T, 3)
    rl, ri = o.score(support, labels, query, chunk=per_call)
    check_oracle(lo.cpu(), None, rl, ri, planted if kind == "structured" else None)
    assert NOTICE not in capfd.readouterr().err


@pytest.mark.parametrize("T", TRIPLE_T_FP32)
def test_long_triples_match_fp32_kernels(models, T, capfd):
    cfg, m, _, _ = models(T, (3,), "NONE", 3)
    support, _, query, planted = make_episode(cfg, 3, 300 + T, "structured")     # 3T > 128 frame rows: two row tiles
    lo, it = scored(m, support, query)
    assert it is None and m.last_path() == expected_path(T, 3)
    _, f, _, _ = models(T, (3,), "NONE", 3, force_path=1)
    lf, _ = scored(f, support, query)
    assert f.last_path() == 1
    e = rel_err(lo.cpu(), lf.cpu()).max()
    assert e < TOL, f"max relative error {e:.3g}"
    assert np.array_equal(lo.argmax(1).cpu().numpy(), planted) and np.array_equal(lf.argmax(1).cpu().numpy(), planted)
    assert NOTICE not in capfd.readouterr().err


@pytest.mark.parametrize("T", [11, 33])
def test_second_transformer_triples_match_oracle(models, T):
    way, B, per_call = oracle_batch(T, 3)
    cfg, m, _, o = models(T, (2, 3), "DISC", way)
    support, labels, query, planted = make_episode(cfg, B, 400 + T, "structured")
    ssf = o.embed(torch.from_numpy(support).double())                                  # (1, way, T, F)
    qf = o.embed(torch.from_numpy(query).double()).float()                             # (B, T, F)
    m.set_support(features=ssf[0].float().cuda())
    lg = m.score_features(1, qf.cuda())
    assert m.last_path() == expected_path(T, 3)
    ref = torch.cat([o.cross_transformer(ssf.float().double().expand(b1 - b0, -1, -1, -1), torch.from_numpy(labels),
                                         qf[b0:b1].double().unsqueeze(1), ti=1)["logits"]
                     for b0, b1 in ((i, min(i + per_call, B)) for i in range(0, B, per_call))])
    check_oracle(lg.cpu(), None, ref.numpy(), None, planted)


# ---- 4. cardinality 1 and 4: the fp32 kernels -----------------------------------------------------------------------------
C14 = [(T, 1) for T in C1_T] + [(T, 4) for T in C4_T]


@pytest.mark.parametrize("T,c", C14)
def test_c1_c4_match_oracle(models, T, c):
    way, B, per_call = oracle_batch(T, c)
    cfg, m, _, o = models(T, (c,), "NONE", way)
    support, labels, query, planted = make_episode(cfg, B, 500 + 10 * T + c, "structured")
    lo, it = scored(m, support, query)
    assert it is None and m.last_path() == 1
    rl, ri = o.score(support, labels, query, chunk=per_call)
    check_oracle(lo.cpu(), None, rl, ri, planted)


@pytest.mark.parametrize("T,c", [(16, 1), (64, 1), (4, 4), (16, 4)])
def test_c1_c4_refuse_forced_tensor_core_kernels(models, T, c):
    cfg, m, _, _ = models(T, (c,), "NONE", force_path=2)
    support, _, query, _ = make_episode(cfg, 2, 600 + T, "structured")
    with pytest.raises(ValueError, match="force_path=2 but no tcgen05 path"):
        scored(m, support, query)


@pytest.mark.parametrize("c", [1, 4])
def test_discriminator_with_c1_c4_is_refused(models, c):
    cfg, m, _, _ = models(8, (c,), "DISC")
    support, labels, query, _ = make_episode(cfg, 3, 700 + c, "structured")
    S, L, Q = torch.from_numpy(support).cuda(), torch.from_numpy(labels).cuda(), torch.from_numpy(query).cuda()
    with pytest.raises(ValueError, match="pair tuples"):
        m({"sk": S}, L, {"sk": Q})
    with pytest.raises(ValueError, match="pair tuples"):
        scored(m, support, query)
    with pytest.raises(ValueError, match="pair tuples"):
        m.score_frames(Q.reshape(-1, Q.shape[-1]))
    with pytest.raises(ValueError, match="pair tuples"):
        m.score_episodes(Q, poses=S.expand(Q.shape[0], -1, -1, -1))
    m.set_support(poses=S[0])
    with pytest.raises(ValueError, match="pair tuples"):
        m.stream_push(query[0, 0])


# ---- 5. four transformers on one handle ------------------------------------------------------------------------------------
def test_four_transformers_on_one_handle(models, capfd):
    temp_set = (2, 1, 3, 4)
    cfg, m, _, o = models(16, temp_set, "DISC")
    B = 12                                                       # 192 query frame rows: two row tiles
    support, labels, query, planted = make_episode(cfg, B, 800, "structured")
    S, L, Q = torch.from_numpy(support).cuda(), torch.from_numpy(labels).cuda(), torch.from_numpy(query).cuda()
    out = m({"sk": S}, L, {"sk": Q})
    assert m.last_path() == expected_path(16, 2)
    ref = o.forward({"sk": support}, labels, {"sk": query})
    check_oracle(cpu(out["logits"]), cpu(out["is_true"]), ref["logits"], ref["is_true"], planted)
    ssf = ref["support_features"]                                # float64 (1, way, T, F)
    qf = o.embed(torch.from_numpy(query).double()).float()
    lab = torch.from_numpy(labels)
    for source in ("poses", "features"):
        if source == "poses":
            m.set_support(poses=S[0])
            ss = ssf
        else:
            m.set_support(features=ssf[0].float().cuda())
            ss = ssf.float().double()
        for ti in (1, 2, 3):
            lg = m.score_features(ti, qf.cuda())
            assert m.last_path() == expected_path(16, temp_set[ti]), (source, ti)
            rl = o.cross_transformer(ss.expand(B, -1, -1, -1), lab, qf.double().unsqueeze(1), ti=ti)["logits"]
            check_oracle(lg.cpu(), None, rl.numpy(), None, planted)
    # the support blob of all four transformers, into a fresh handle
    m.set_support(poses=S[0])
    a = m.score(Q)
    blob = m.export_support()
    assert blob.numel() == sum(2 * cfg.way * math.comb(16, c) * 128 for c in temp_set)
    fresh, _ = make_model(cfg, 0)
    fresh.import_support(blob, cfg.way)
    assert bit_equal(a, fresh.score(Q)) and fresh.last_path() == expected_path(16, 2)
    for ti in (1, 2, 3):
        assert torch.equal(m.score_features(ti, qf.cuda()), fresh.score_features(ti, qf.cuda())), ti
        assert fresh.last_path() == expected_path(16, temp_set[ti])
    assert NOTICE not in capfd.readouterr().err


# ---- 6. the other entry points at the new shapes ------------------------------------------------------------------------------
ENTRY_SHAPES = [(5, 2), (17, 2), (11, 3)]


@pytest.mark.parametrize("T,c", [(5, 2), (17, 2), (23, 2), (11, 3)])
def test_chunked_is_bit_identical(models, T, c):
    cfg, m, _, _ = models(T, (c,), model_kind(c))
    support, _, query, _ = make_episode(cfg, windows_for(T), 900 + T, "structured")
    a = scored(m, support, query)
    assert m.last_path() == expected_path(T, c)
    for mc in (1, 3):
        _, r, _, _ = models(T, (c,), model_kind(c), max_chunk=mc)
        assert bit_equal(a, scored(r, support, query)), mc
        assert r.last_path() == expected_path(T, c)


@pytest.mark.parametrize("T,c", ENTRY_SHAPES)
def test_score_frames_matches_windows_and_oracle(models, T, c):
    cfg, m, _, o = models(T, (c,), model_kind(c))
    rng = np.random.default_rng(1000 + T)
    support = (0.17 * rng.standard_normal((cfg.way, T, 90))).astype(np.float32)
    frames = (0.17 * rng.standard_normal((300, 90))).astype(np.float32)
    frames[150:150 + T] = support[2] + 0.05 * rng.standard_normal((T, 90)).astype(np.float32)     # in the second row tile
    m.set_support(poses=torch.from_numpy(support).cuda())
    F = torch.from_numpy(frames).cuda()
    lo_s, it_s = m.score_frames(F)
    assert m.last_path() == expected_path(T, c) and lo_s.shape == (300 - T + 1, cfg.way)
    windows = F.unfold(0, T, 1).permute(0, 2, 1).contiguous()
    lo_w, it_w = m.score(windows)
    if expected_path(T, c) == 1:                                 # the fp32 kernels add the positional table after the accumulation
        assert bit_equal((lo_s, it_s), (lo_w, it_w))
    assert rel_err(lo_s.cpu(), lo_w.cpu()).max() < TOL
    assert (it_s is None) == (it_w is None) and (it_s is None or rel_err(it_s.cpu(), it_w.cpu()).max() < TOL)
    pick = [0, 120, 130, 150, 230, 300 - T]
    lo, it = o.score(support[None], np.arange(cfg.way)[None], windows[pick].cpu().numpy(), chunk=len(pick))
    check_oracle(lo_s[pick].cpu(), None if it_s is None else it_s[pick].cpu(), lo, it, None)
    assert int(lo_s[150].argmax()) == 2


@pytest.mark.parametrize("T,c", ENTRY_SHAPES)
def test_score_episodes_matches_oracle_and_loop(models, T, c):
    cfg, m, _, o = models(T, (c,), model_kind(c))
    b, way = 20, cfg.way                                         # a pool of 100 support classes
    rng = np.random.default_rng(1100 + T)
    support = (0.17 * rng.standard_normal((b, way, T, 90))).astype(np.float32)
    pick = rng.integers(0, way, b)
    query = (support[np.arange(b), pick] + 0.05 * rng.standard_normal((b, T, 90))).astype(np.float32)
    S, Q = torch.from_numpy(support).cuda(), torch.from_numpy(query).cuda()
    lg, it = m.score_episodes(Q, poses=S)
    assert m.last_path() == expected_path(T, c)
    ref = o.forward({"sk": support}, np.tile(np.arange(way, dtype=np.int32), (b, 1)), {"sk": query})
    check_oracle(lg.cpu(), cpu(it), ref["logits"], ref.get("is_true"), pick)
    rl, ri = [], []
    for e in range(b):                                           # set_support + a one-window score per episode
        m.set_support(poses=S[e])
        x, y = m.score(Q[e:e + 1])
        rl.append(x)
        ri.append(y)
    assert m.last_path() == expected_path(T, c)
    assert torch.equal(lg, torch.cat(rl))
    assert (it is None and ri[0] is None) or torch.equal(it, torch.cat(ri))


@pytest.mark.parametrize("T,c", ENTRY_SHAPES)
def test_host_rows_are_bit_identical(models, T, c):
    cfg, m, _, _ = models(T, (c,), model_kind(c))
    support, _, query, _ = make_episode(cfg, windows_for(T), 1200 + T, "structured")
    q16 = torch.from_numpy(query).to(torch.float16)
    q32 = q16.to(torch.float32)                                  # the same values, representable in fp16
    m.set_support(poses=torch.from_numpy(support[0]).cuda())
    d = m.score(q32.cuda())
    assert bit_equal(m.score_host(q32.pin_memory()), d)
    assert bit_equal(m.score_host_async(q32.pin_memory()).result(), d)
    if expected_path(T, c) != 1:
        assert bit_equal(m.score_host(q16.pin_memory()), d)
        assert bit_equal(m.score_host_async(q16.pin_memory()).result(), d)
    else:                                                        # fp16 rows need the tensor-core linears
        with pytest.raises(ValueError, match="fp16 rows"):
            m.score_host(q16.pin_memory())
        with pytest.raises(ValueError, match="fp16 rows"):
            m.score_host_async(q16.pin_memory())
    assert m.last_path() == expected_path(T, c)


# ---- 7. the resident streaming scorer and the ActionRecognizer --------------------------------------------------------------
@pytest.mark.parametrize("T", [10, 11, 17, 31])                 # K1 = N*T = 450, 605, 2312, 14415: every residue mod 4
def test_stream_push_matches_score(models, T, capfd):
    cfg, m, _, _ = models(T)
    rng = np.random.default_rng(1300 + T)
    support = (0.17 * rng.standard_normal((cfg.way, T, 90))).astype(np.float32)
    frames = np.concatenate([support[3] + 0.05 * rng.standard_normal((T, 90)), 0.17 * rng.standard_normal((8, 90))]).astype(np.float32)
    m.set_support(poses=torch.from_numpy(support).cuda())
    m.stream_reset()
    got = []
    for i, f in enumerate(frames):                               # from the second call on, the per-frame graph is replayed
        probs, is_true, valid = m.stream_push(f)
        assert m.last_path() == 3
        assert valid == (i >= T - 1)
        if valid:
            got.append((probs, is_true))
    windows = np.stack([frames[i:i + T] for i in range(len(frames) - T + 1)])
    lo, it = m.score(torch.from_numpy(windows).cuda())
    probs_ref = torch.softmax(lo, 1).cpu().numpy()
    assert len(got) == len(windows) == 9
    assert rel_err(np.stack([g[0] for g in got]), probs_ref).max() < TOL_PROBS
    assert rel_err(np.stack([g[1] for g in got]), it.cpu().numpy()).max() < TOL
    assert int(got[0][0].argmax()) == 3
    assert NOTICE not in capfd.readouterr().err


@pytest.mark.parametrize("T", [2, 3, 5, 7])                     # N = 1, 3, 10, 21: the tiled kernels miss TOL there
def test_stream_push_refused_below_min_tuples(models, T):
    cfg, m, _, _ = models(T)
    support, _, query, _ = make_episode(cfg, 1, 1350 + T, "structured")
    m.set_support(poses=torch.from_numpy(support[0]).cuda())
    with pytest.raises(ValueError, match="resident streaming path"):
        m.stream_push(query[0, 0])


@pytest.mark.parametrize("T", [3, 17])
def test_action_recognizer_matches_oracle(models, T):
    from isbfsar_b200 import ActionRecognizer
    cfg, _, sd, _ = models(T)
    ar = ActionRecognizer(Args(cfg), state_dict=torch_sd(sd))
    oa = ActionRecognizerOracle(cfg, sd)
    rng = np.random.default_rng(1400 + T)
    poses = (0.17 * rng.standard_normal((3, T, 90))).astype(np.float32)
    frames = (poses[1][np.arange(T + 5) % T] + 0.05 * rng.standard_normal((T + 5, 90))).astype(np.float32)
    for i, n in enumerate(["a", "b", "c"]):
        inp = {"flag": n, "data": {"poses": poses[i]}, "requires_focus": False}
        ar.train(inp)
        oa.train(inp)
    n_valid = 0
    for f in frames:
        r, o_, _ = ar.inference({"sk": f})
        ro, oo, _ = oa.inference({"sk": f})
        assert (len(r) == 0) == (len(ro) == 0)
        if not r:
            continue
        n_valid += 1
        assert list(r) == ["a", "b", "c"]
        p, po = np.array([r[k] for k in r]), np.array([ro[k] for k in r])
        assert rel_err(p, po).max() < TOL_PROBS
        assert rel_err(o_, oo).max() < TOL
        srt = np.sort(po)                                        # argmax where the margin allows
        if (srt[-1] - srt[-2]) / srt[-1] > 2 * TOL_PROBS:
            assert p.argmax() == po.argmax()
    assert n_valid == 6
    # arx_stream_push, or (N < MIN_TUPLES) the batch fallback on the fp32 kernels
    assert ar._stream_ok == (expected_path(T, 2) == 3) and ar.ar.last_path() == expected_path(T, 2)
