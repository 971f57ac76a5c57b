"""Pair-tuple open-set scoring at sequence lengths 33..64 on the tiled tensor-core kernels.

The reference builds Discriminator(seq_len=C(T,2), l=T) for any T (model.py:282-285).  The head's L = T columns live on
TMEM lanes of the MODE 1 accumulator of k_attn_tcn, so the tiled route serves the head up to T = 64 (DESIGN 5).  T = 34
and 35 have K = N*T of discriminator.fc1 not a multiple of 4 (scalar head / tail of the streaming fc1), T = 33 an odd
number of tuple tiles (N = 528, 5 tiles), T = 64 sixteen tiles (N = 2016)."""
import numpy as np
import pytest
import torch

from oracle.synth import Cfg, make_episode
from oracle.trx_oracle import ActionRecognizerOracle, TrxOracle
from tests.util import Args, make_model, rel_err, torch_sd

pytestmark = pytest.mark.gpu

TOL = 1e-3                      # relative, logits and is_true
TOL_PROBS = 2e-3                # softmax of logits held to TOL
NOTICE = "fp32 CUDA-core kernels"


@pytest.fixture(scope="module")
def models():
    """(cfg, model, state dict, float64 oracle) per (T, way), built once per module"""
    cache = {}

    def get(T, way=5):
        if (T, way) not in cache:
            cfg = Cfg(way=way, seq_len=T)
            m, sd = make_model(cfg, 0)
            cache[(T, way)] = (cfg, m, sd, TrxOracle(cfg, sd, dtype=torch.float64))
        return cache[(T, way)]

    yield get
    cache.clear()


def check_oracle(lo, it, rl, ri, planted=None):
    lo, it, rl, ri = (np.asarray(x, dtype=np.float64) for x in (lo, it, rl, ri))
    assert rel_err(lo, rl).max() < TOL
    assert rel_err(it, ri).max() < TOL
    if planted is not None:
        assert np.array_equal(lo.argmax(1), rl.argmax(1)) and np.array_equal(lo.argmax(1), planted)
    else:                       # iid inputs: argmax compared where the reference margin exceeds the tolerance twice over
        srt = np.sort(rl, 1)
        ok = (srt[:, -1] - srt[:, -2]) / np.abs(srt[:, -1]) > 2 * TOL
        assert np.array_equal(lo.argmax(1)[ok], rl.argmax(1)[ok])
    assert np.array_equal(it > 0.5, ri > 0.5)


# ---- 1. TRXOS.forward against the float64 oracle, from poses and from ss_features ---------------------------------------
@pytest.mark.parametrize("kind", ["structured", "iid"])
@pytest.mark.parametrize("T", [33, 34, 35, 40, 48, 64])
def test_forward_matches_oracle(models, T, kind, capfd):
    cfg, m, _, o = models(T)
    B = 6
    support, labels, query, planted = make_episode(cfg, B, 100 + T, kind)
    S, L, Q = torch.from_numpy(support).cuda(), torch.from_numpy(labels).cuda(), torch.from_numpy(query).cuda()
    out = m({"sk": S}, L, {"sk": Q})
    assert m.last_path() == 3
    ref = o.forward({"sk": support}, labels, {"sk": query})
    check_oracle(out["logits"].cpu(), out["is_true"].cpu(), ref["logits"], ref["is_true"], planted if kind == "structured" else None)
    ssf = ref["support_features"].float()
    out2 = m(None, L, {"sk": Q}, ss_features=ssf.cuda())
    assert m.last_path() == 3
    ref2 = o.forward(None, labels, {"sk": query}, ss_features=ssf)
    check_oracle(out2["logits"].cpu(), out2["is_true"].cpu(), ref2["logits"], ref2["is_true"], planted if kind == "structured" else None)
    assert NOTICE not in capfd.readouterr().err


def test_t64_20way_matches_oracle(models, capfd):
    cfg, m, _, o = models(64, 20)
    support, labels, query, planted = make_episode(cfg, 3, 7, "structured")
    out = m({"sk": torch.from_numpy(support).cuda()}, torch.from_numpy(labels).cuda(), {"sk": torch.from_numpy(query).cuda()})
    assert m.last_path() == 3
    ref = o.forward({"sk": support}, labels, {"sk": query})
    check_oracle(out["logits"].cpu(), out["is_true"].cpu(), ref["logits"], ref["is_true"], planted)
    assert NOTICE not in capfd.readouterr().err


# ---- 2. the tiled route against the fp32 kernels (force_path = 1) --------------------------------------------------------
@pytest.mark.parametrize("T", [35, 64])
def test_tiled_matches_fp32_kernels(models, T):
    cfg, m, _, _ = models(T)
    support, _, query, _ = make_episode(cfg, 8, 200 + T, "structured")
    S, Q = torch.from_numpy(support[0]).cuda(), torch.from_numpy(query).cuda()
    m.set_support(poses=S)
    lo, it = m.score(Q)
    assert m.last_path() == 3
    f, _ = make_model(cfg, 0, force_path=1)
    f.set_support(poses=S)
    lf, itf = f.score(Q)
    assert f.last_path() == 1
    assert rel_err(lo.cpu(), lf.cpu()).max() < TOL and rel_err(it.cpu(), itf.cpu()).max() < TOL
    assert torch.equal(lo.argmax(1), lf.argmax(1)) and torch.equal(it > 0.5, itf > 0.5)


# ---- 3. chunking does not change a bit ------------------------------------------------------------------------------------
def test_chunked_is_bit_identical(models):
    cfg, m, _, _ = models(40)
    support, _, query, _ = make_episode(cfg, 8, 300, "structured")
    S, Q = torch.from_numpy(support[0]).cuda(), torch.from_numpy(query).cuda()
    m.set_support(poses=S)
    a = m.score(Q)
    c, _ = make_model(cfg, 0, max_chunk=3)                       # 3 + 3 + 2 windows
    c.set_support(poses=S)
    b = c.score(Q)
    assert m.last_path() == 3 and c.last_path() == 3
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])


# ---- 4. frame streams, episodes, host rows --------------------------------------------------------------------------------
def test_score_frames_matches_explicit_windows(models):
    cfg, m, _, o = models(40)
    T = cfg.seq_len
    rng = np.random.default_rng(41)
    support = (0.17 * rng.standard_normal((cfg.way, T, 90))).astype(np.float32)
    frames = (0.17 * rng.standard_normal((T + 11, 90))).astype(np.float32)
    frames[4:4 + T] = support[2] + 0.05 * rng.standard_normal((T, 90)).astype(np.float32)
    m.set_support(poses=torch.from_numpy(support).cuda())
    F = torch.from_numpy(frames).cuda()
    lo_s, it_s = m.score_frames(F)
    assert m.last_path() == 3 and lo_s.shape == (12, cfg.way)
    windows = F.unfold(0, T, 1).permute(0, 2, 1).contiguous()
    lo_w, it_w = m.score(windows)
    assert rel_err(lo_s.cpu(), lo_w.cpu()).max() < TOL and rel_err(it_s.cpu(), it_w.cpu()).max() < TOL
    lo, it = o.score(support[None], np.arange(cfg.way)[None], windows[:6].cpu().numpy(), chunk=6)
    check_oracle(lo_s[:6].cpu(), it_s[:6].cpu(), lo, it, None)
    assert int(lo_s[4].argmax()) == 2


def test_score_episodes_matches_oracle_and_loop(models):
    cfg, m, _, o = models(48)
    b, way, T = 4, cfg.way, cfg.seq_len
    rng = np.random.default_rng(48)
    support = (0.17 * rng.standard_normal((b, way, T, 90))).astype(np.float32)
    pick = rng.integers(0, way, b)
    query = (support[np.arange(b), pick] + 0.05 * rng.standard_normal((b, T, 90))).astype(np.float32)
    S, Q = torch.from_numpy(support).cuda(), torch.from_numpy(query).cuda()
    lg, it = m.score_episodes(Q, poses=S)
    assert m.last_path() == 3
    ref = o.forward({"sk": support}, np.tile(np.arange(way, dtype=np.int32), (b, 1)), {"sk": query})
    check_oracle(lg.cpu(), it.cpu(), ref["logits"], ref["is_true"], pick)
    rl, ri = [], []
    for e in range(b):                                           # set_support + a one-window score per episode
        m.set_support(poses=S[e])
        x, y = m.score(Q[e:e + 1])
        rl.append(x)
        ri.append(y)
    assert m.last_path() == 3
    assert torch.equal(lg, torch.cat(rl)) and torch.equal(it, torch.cat(ri))


def test_host_rows_are_bit_identical(models):
    cfg, m, _, _ = models(40)
    support, _, query, _ = make_episode(cfg, 20, 400, "structured")
    q16 = torch.from_numpy(query).to(torch.float16)
    q32 = q16.to(torch.float32)                                  # the same values, representable in fp16
    m.set_support(poses=torch.from_numpy(support[0]).cuda())
    d = m.score(q32.cuda())
    a = m.score_host(q32.pin_memory())
    b = m.score_host(q16.pin_memory())
    c = m.score_host_async(q16.pin_memory()).result()
    assert m.last_path() == 3
    for x in (a, b, c):
        assert torch.equal(x[0], d[0].cpu()) and torch.equal(x[1], d[1].cpu())


# ---- 5. the resident streaming scorer and the ActionRecognizer ------------------------------------------------------------
@pytest.mark.parametrize("T", [34, 40])
def test_stream_push_matches_score(models, T, capfd):
    cfg, m, _, _ = models(T)
    rng = np.random.default_rng(500 + T)
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


def test_action_recognizer_matches_oracle(models):
    from isbfsar_b200 import ActionRecognizer
    cfg, _, sd, _ = models(34)
    T = cfg.seq_len
    ar = ActionRecognizer(Args(cfg), state_dict=torch_sd(sd))
    oa = ActionRecognizerOracle(cfg, sd)
    rng = np.random.default_rng(34)
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
        assert rel_err(np.array([r[k] for k in r]), np.array([ro[k] for k in r])).max() < TOL_PROBS
        assert rel_err(o_, oo).max() < TOL
        assert max(r, key=r.get) == "b"
    assert n_valid == 6
    assert ar._stream_ok and ar.ar.last_path() == 3              # served by arx_stream_push, not the batch fallback


# ---- 6. what stays out of scope -------------------------------------------------------------------------------------------
def test_triples_with_discriminator_still_refused():
    cfg = Cfg(seq_len=33, temp_set=[3])
    m, _ = make_model(cfg, 0)
    support, _, query, _ = make_episode(cfg, 2, 600, "structured")
    m.set_support(poses=torch.from_numpy(support[0]).cuda())
    with pytest.raises(ValueError, match="pair tuples"):
        m.score(torch.from_numpy(query).cuda())
    with pytest.raises(ValueError, match="pair tuples"):
        m.stream_push(query[0, 0])
