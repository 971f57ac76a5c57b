"""Every joint count the front end accepts, against the float64 oracle.

The frame MLP is 3J -> 6J -> 256 (model.py:146,175-180), and J picks its kernels (DESIGN 5):
  J <= 32   tensor-core linears: fc1 is one 192-column tile, fc2 reads ceil(6J/64) K sub-tiles of it (1 up to J = 10,
            2 for J = 11..21, 3 from J = 22); at J = 30 big pair-pipeline batches take the fused k_mlp_p instead;
  J >= 33   fp32 CUDA-core linears (tensor-core linears need 6J <= 192); T=16 pairs then score on the tiled route.
The resident streaming scorer serves J <= 42 (6J <= 256), the fp16 host rows J <= 32.

fc1 writes its whole column tile, pad columns included, into the hidden image fc2 reads: a pass of more than 128 frame rows
(several row tiles) is where a too narrow image would let one row tile overwrite the next, so the passes here hold several
row tiles, and a pass of exactly one row tile (max_chunk = 128 / T windows) is their bit-exact reference.  The joint counts
cover both ends of each row above, fc1's K at one and two sub-tiles (3J = 63 / 66), 6J = 192 exactly and the stream limit."""
import numpy as np
import pytest
import torch

from oracle.synth import Cfg, make_episode
from oracle.trx_oracle import ActionRecognizerOracle, TrxOracle
from tests.util import Args, make_model, rel_err, torch_sd

pytestmark = pytest.mark.gpu

TOL = 1e-3                      # relative, logits and is_true
TOL_PROBS = 2e-3                # softmax of logits held to TOL
TOL_FP32 = 5e-5                 # fp32 CUDA-core linears: summation-order noise only
# One joint: the frame features are nearly the fc biases, the distances are small differences of nearly equal V rows, and
# the fp16 operands of the front end and the projection cost more of them (1.05e-3 measured on a B200 at a 1000 W power
# limit, against 2.4e-4 at J = 30; the same passes of one row tile give the same bits).
TOL_ONE_JOINT = 2e-3
NOTICE = "fp32 CUDA-core kernels"

JOINTS = [1, 10, 17, 21, 22, 25, 30, 32, 33, 42, 43]
TC_JOINTS = [J for J in JOINTS if J <= 32]          # tensor-core front end
BIG_JOINTS = [10, 17, 25, 32]                       # one per fc2 sub-tile count, and 6J = 192
SOME_JOINTS = [10, 17, 25, 33]                      # one per fc2 sub-tile count, and the first fp32 front end


@pytest.fixture(scope="module")
def models():
    """(cfg, model, state dict, float64 oracle) per (J, T, way, max_chunk), built once per module"""
    cache = {}

    def get(J, T=16, way=5, max_chunk=0):
        key = (J, T, way, max_chunk)
        if key not in cache:
            cfg = Cfg(way=way, seq_len=T, n_joints=J)
            m, sd = make_model(cfg, 0, max_chunk=max_chunk)
            cache[key] = (cfg, m, sd, TrxOracle(cfg, sd, dtype=torch.float64))
        return cache[key]

    yield get
    cache.clear()


def pair_path(J, T):
    """T=16 pairs take the pair pipeline when the tensor-core linears serve the front end; all else the tiled route"""
    return 2 if T == 16 and J <= 32 else 3


def one_tile(T):
    """windows per pass that make exactly one 128-row tile of frames"""
    return 128 // T


def big_batch(T):
    """windows enough for the persistent front end of the pair pipeline (two row tiles per SM), plus a ragged tail"""
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    return -(-2 * 128 * sms // T) + 13


def planted_is_argmax(J):
    """the planted class as the expected argmax: one joint (three coordinates) through the MLP does not separate the
    planted classes even in float64, so there the argmax is compared with the oracle's where its margin allows"""
    return J > 1


def check_oracle(lo, it, rl, ri, planted=None, tol=TOL):
    lo, it, rl, ri = (np.asarray(x, dtype=np.float64) for x in (lo, it, rl, ri))
    assert rel_err(lo, rl).max() < tol
    assert rel_err(it, ri).max() < TOL
    if planted is not None:
        assert np.array_equal(lo.argmax(1), rl.argmax(1)) and np.array_equal(lo.argmax(1), planted)
    else:                       # argmax compared where the reference margin exceeds the tolerance twice over
        srt = np.sort(rl, 1)
        ok = (srt[:, -1] - srt[:, -2]) / np.abs(srt[:, -1]) > 2 * tol
        assert np.array_equal(lo.argmax(1)[ok], rl.argmax(1)[ok])
    assert np.array_equal(it > 0.5, ri > 0.5)


def bit_equal(a, b):
    return all(torch.equal(x.cpu(), y.cpu()) for x, y in zip(a, b))


def scored(m, support, query):
    m.set_support(poses=torch.from_numpy(support[0]).cuda())
    return m.score(torch.from_numpy(query).cuda())


# ---- 1. which kernels serve each joint count ------------------------------------------------------------------------------
@pytest.mark.parametrize("J", JOINTS)
def test_route(models, J, capfd):
    for T, way in ((16, 5), (32, 20)):
        cfg, m, _, _ = models(J, T, way)
        support, _, query, _ = make_episode(cfg, 2, 1, "structured")
        scored(m, support, query)
        assert m.last_path() == pair_path(J, T), (T, m.last_path())
    assert NOTICE not in capfd.readouterr().err


# ---- 2. TRXOS.forward against the float64 oracle, from poses and from ss_features ---------------------------------------
@pytest.mark.parametrize("kind", ["structured", "iid"])
@pytest.mark.parametrize("J", JOINTS)
def test_forward_matches_oracle(models, J, kind, capfd):
    cfg, m, _, o = models(J)
    B = 24                                                       # 384 query frame rows: three row tiles
    support, labels, query, planted = make_episode(cfg, B, 100 + J, kind)
    expect = planted if kind == "structured" and planted_is_argmax(J) else None
    tol = TOL if J > 1 else TOL_ONE_JOINT
    S, L, Q = torch.from_numpy(support).cuda(), torch.from_numpy(labels).cuda(), torch.from_numpy(query).cuda()
    out = m({"sk": S}, L, {"sk": Q})
    assert m.last_path() == pair_path(J, 16)
    ref = o.forward({"sk": support}, labels, {"sk": query})
    check_oracle(out["logits"].cpu(), out["is_true"].cpu(), ref["logits"], ref["is_true"], expect, tol)
    ssf = ref["support_features"].float()
    out2 = m(None, L, {"sk": Q}, ss_features=ssf.cuda())
    assert m.last_path() == pair_path(J, 16)
    ref2 = o.forward(None, labels, {"sk": query}, ss_features=ssf)
    check_oracle(out2["logits"].cpu(), out2["is_true"].cpu(), ref2["logits"], ref2["is_true"], expect, tol)
    assert NOTICE not in capfd.readouterr().err


@pytest.mark.parametrize("J", SOME_JOINTS)
def test_t32_20way_matches_oracle(models, J):
    cfg, m, _, o = models(J, 32, 20)                             # 640 support frame rows: five row tiles
    support, labels, query, planted = make_episode(cfg, 8, 200 + J, "structured")
    out = m({"sk": torch.from_numpy(support).cuda()}, torch.from_numpy(labels).cuda(), {"sk": torch.from_numpy(query).cuda()})
    assert m.last_path() == 3
    ref = o.forward({"sk": support}, labels, {"sk": query})
    check_oracle(out["logits"].cpu(), out["is_true"].cpu(), ref["logits"], ref["is_true"], planted)


# ---- 3. a pass of one row tile is the bit-exact reference of a pass of several ----------------------------------------------
@pytest.mark.parametrize("T", [16, 32])
@pytest.mark.parametrize("J", TC_JOINTS)
def test_one_row_tile_pass_is_bit_identical(models, J, T):
    cfg, m, _, _ = models(J, T)
    _, r, _, _ = models(J, T, max_chunk=one_tile(T))
    support, _, query, _ = make_episode(cfg, 24, 300 + J, "iid")
    a = scored(m, support, query)
    b = scored(r, support, query)
    assert m.last_path() == r.last_path() == pair_path(J, T)
    assert bit_equal(a, b)


# ---- 4. big batches: the persistent front end, every window against the oracle ------------------------------------------
@pytest.mark.parametrize("J", BIG_JOINTS)
def test_big_batch(models, J):
    cfg, m, _, o = models(J)
    B = big_batch(16)
    support, labels, query, planted = make_episode(cfg, B, 400 + J, "structured")
    lo, it = scored(m, support, query)
    assert m.last_path() == 2
    rl, ri = o.score(support, labels, query, chunk=512)
    check_oracle(lo.cpu(), it.cpu(), rl, ri, planted)
    # the one-tile-per-CTA GEMMs (debug variant 1024), and passes of one row tile
    v, _ = make_model(cfg, 0)
    v.debug_set(0, 1024)
    assert bit_equal((lo, it), scored(v, support, query)) and v.last_path() == 2
    _, r, _, _ = models(J, max_chunk=one_tile(16))
    assert bit_equal((lo, it), scored(r, support, query)) and r.last_path() == 2
    # host rows, staged in passes of their own
    q16 = torch.from_numpy(query).to(torch.float16)
    q32 = q16.to(torch.float32)                                  # the same values, representable in fp16
    d = m.score(q32.cuda())
    for x in (m.score_host(q32.pin_memory()), m.score_host(q16.pin_memory()), m.score_host_async(q16.pin_memory()).result()):
        assert bit_equal(x, d)


# ---- 5. frame streams longer than one row tile --------------------------------------------------------------------------
@pytest.mark.parametrize("J", [17, 25, 33])
def test_score_frames_matches_windows_and_oracle(models, J):
    cfg, m, _, o = models(J)
    T, J3 = cfg.seq_len, 3 * J
    rng = np.random.default_rng(500 + J)
    support = (0.17 * rng.standard_normal((cfg.way, T, J3))).astype(np.float32)
    frames = (0.17 * rng.standard_normal((300, J3))).astype(np.float32)
    frames[150:150 + T] = support[2] + 0.05 * rng.standard_normal((T, J3)).astype(np.float32)     # in the second row tile
    m.set_support(poses=torch.from_numpy(support).cuda())
    F = torch.from_numpy(frames).cuda()
    lo_s, it_s = m.score_frames(F)
    assert m.last_path() == pair_path(J, T) and lo_s.shape == (300 - T + 1, cfg.way)
    windows = F.unfold(0, T, 1).permute(0, 2, 1).contiguous()
    lo_w, it_w = m.score(windows)
    assert rel_err(lo_s.cpu(), lo_w.cpu()).max() < TOL and rel_err(it_s.cpu(), it_w.cpu()).max() < TOL
    pick = [0, 120, 130, 150, 230, 284]                          # windows in row tile 0, across 0 and 1, in 1, 1, 1 and 2
    lo, it = o.score(support[None], np.arange(cfg.way)[None], windows[pick].cpu().numpy(), chunk=6)
    check_oracle(lo_s[pick].cpu(), it_s[pick].cpu(), lo, it, None)
    assert int(lo_s[150].argmax()) == 2


# ---- 6. per-episode support sets --------------------------------------------------------------------------------------------
@pytest.mark.parametrize("T", [16, 32])
@pytest.mark.parametrize("J", SOME_JOINTS)
def test_score_episodes_matches_oracle_and_loop(models, J, T):
    cfg, m, _, o = models(J, T)
    b, way, J3 = 20, cfg.way, 3 * J                              # a pool of 100 classes: 1600 or 3200 support frame rows
    rng = np.random.default_rng(600 + J + T)
    support = (0.17 * rng.standard_normal((b, way, T, J3))).astype(np.float32)
    pick = rng.integers(0, way, b)
    query = (support[np.arange(b), pick] + 0.05 * rng.standard_normal((b, T, J3))).astype(np.float32)
    S, Q = torch.from_numpy(support).cuda(), torch.from_numpy(query).cuda()
    lg, it = m.score_episodes(Q, poses=S)
    assert m.last_path() == pair_path(J, T)
    ref = o.forward({"sk": support}, np.tile(np.arange(way, dtype=np.int32), (b, 1)), {"sk": query})
    check_oracle(lg.cpu(), it.cpu(), ref["logits"], ref["is_true"], pick)
    rl, ri = [], []
    for e in range(b):                                           # set_support + a one-window score per episode
        m.set_support(poses=S[e])
        x, y = m.score(Q[e:e + 1])
        rl.append(x)
        ri.append(y)
    assert m.last_path() == pair_path(J, T)
    assert torch.equal(lg, torch.cat(rl)) and torch.equal(it, torch.cat(ri))


# ---- 7. host rows -------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("J", JOINTS)
def test_host_rows(models, J):
    cfg, m, _, _ = models(J)
    support, _, query, _ = make_episode(cfg, 24, 700 + J, "structured")
    q16 = torch.from_numpy(query).to(torch.float16)
    q32 = q16.to(torch.float32)                                  # the same values, representable in fp16
    m.set_support(poses=torch.from_numpy(support[0]).cuda())
    d = m.score(q32.cuda())
    assert bit_equal(m.score_host(q32.pin_memory()), d)
    assert bit_equal(m.score_host_async(q32.pin_memory()).result(), d)
    if J <= 32:
        assert bit_equal(m.score_host(q16.pin_memory()), d)
        assert bit_equal(m.score_host_async(q16.pin_memory()).result(), d)
    else:                                                        # fp16 rows need the tensor-core linears
        with pytest.raises(ValueError, match="fp16 rows"):
            m.score_host(q16.pin_memory())
        with pytest.raises(ValueError, match="fp16 rows"):
            m.score_host_async(q16.pin_memory())
    assert m.last_path() == pair_path(J, 16)


# ---- 8. the resident streaming scorer and the ActionRecognizer --------------------------------------------------------------
@pytest.mark.parametrize("J", [17, 33, 42])
def test_stream_push_matches_score(models, J, capfd):
    cfg, m, _, _ = models(J)
    T, J3 = cfg.seq_len, 3 * J
    rng = np.random.default_rng(800 + J)
    support = (0.17 * rng.standard_normal((cfg.way, T, J3))).astype(np.float32)
    frames = np.concatenate([support[3] + 0.05 * rng.standard_normal((T, J3)), 0.17 * rng.standard_normal((8, J3))]).astype(np.float32)
    m.set_support(poses=torch.from_numpy(support).cuda())
    m.stream_reset()
    got = []
    for i, f in enumerate(frames):
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


def test_stream_push_refused_past_42_joints(models):
    cfg, m, _, _ = models(43)
    support, _, query, _ = make_episode(cfg, 1, 900, "structured")
    m.set_support(poses=torch.from_numpy(support[0]).cuda())
    with pytest.raises(ValueError, match="resident streaming path"):
        m.stream_push(query[0, 0])


@pytest.mark.parametrize("J,streamed", [(17, True), (43, False)])
def test_action_recognizer_matches_oracle(models, J, streamed):
    from isbfsar_b200 import ActionRecognizer
    cfg, _, sd, _ = models(J)
    T, J3 = cfg.seq_len, 3 * J
    ar = ActionRecognizer(Args(cfg), state_dict=torch_sd(sd))
    oa = ActionRecognizerOracle(cfg, sd)
    rng = np.random.default_rng(J)
    poses = (0.17 * rng.standard_normal((3, T, J3))).astype(np.float32)
    frames = (poses[1][np.arange(T + 5) % T] + 0.05 * rng.standard_normal((T + 5, J3))).astype(np.float32)
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
        srt = np.sort(po)                                        # the three classes are close: argmax where the margin allows
        if (srt[-1] - srt[-2]) / srt[-1] > 2 * TOL_PROBS:
            assert p.argmax() == po.argmax()
    assert n_valid == 6
    assert ar._stream_ok == streamed and ar.ar.last_path() == 3      # arx_stream_push, or the batch fallback past J = 42


# ---- 9. support_features(): the fp32 frame MLP (arx_embed) ------------------------------------------------------------------
@pytest.mark.parametrize("J", [1, 17, 43])
def test_support_features_match_oracle(models, J):
    cfg, m, _, o = models(J)
    rng = np.random.default_rng(1000 + J)
    support = (0.17 * rng.standard_normal((20, cfg.seq_len, 3 * J))).astype(np.float32)      # 320 frame rows
    m.set_support(poses=torch.from_numpy(support).cuda())
    got = m.support_features().cpu().numpy()
    ref = o.embed(torch.from_numpy(support).to(torch.float64)).numpy()
    np.testing.assert_allclose(got, ref, rtol=TOL_FP32, atol=1e-6)
