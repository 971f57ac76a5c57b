"""Per-episode support sets on the tiled tensor-core kernels (arx_score_episodes, episode mode of k_attn_tcn).

Every batch row is its own episode (train.py:110-120, compute_fsos.py:89-98).  On the tiled route all episodes of a
pass share one pool of support classes and window b attends pool classes [b*way, (b+1)*way); a pass holds as many
episodes as fit the 1 GiB pool budget (at most 256).  The pool holds transformers[0] only."""
import numpy as np
import pytest
import torch

from isbfsar_b200._lib import ArxError
from isbfsar_b200.eval import evaluate_fsos, synthetic_fsos_episodes
from oracle.synth import Cfg, make_state_dict
from oracle.trx_oracle import TrxOracle
from tests.util import Args, make_model, rel_err, torch_sd

pytestmark = pytest.mark.gpu

TOL_TC = 1e-3
D = 128
OVERFLOW_BOUND = 100.0 / 1.4426950408889634       # |S| log2(e) < 100 (arx_tcn_needs_rowmax)

CFG_T32 = Cfg(way=20, seq_len=32, temp_set=[2, 3])


def episodes(cfg, b, way, seed):
    """support (b,way,T,90), query (b,T,90): query i is a noisy copy of one of its own support classes"""
    rng = np.random.default_rng(seed)
    support = (0.17 * rng.standard_normal((b, way, cfg.seq_len, 90))).astype(np.float32)
    pick = rng.integers(0, way, b)
    query = (support[np.arange(b), pick] + 0.05 * rng.standard_normal((b, cfg.seq_len, 90))).astype(np.float32)
    return support, query


def check_oracle(out, ref):
    lo, it = out["logits"].cpu().numpy(), out["is_true"].cpu().numpy()
    rl, ri = ref["logits"].numpy(), ref["is_true"].numpy()
    assert rel_err(lo, rl).max() < TOL_TC
    assert rel_err(it, ri).max() < TOL_TC
    assert np.array_equal(lo.argmax(1), rl.argmax(1))
    assert np.array_equal(it > 0.5, ri > 0.5)


def loop(m, support, query):
    """what arx_score_episodes did for these shapes before: set_support + a one-window score per episode"""
    lg, it = [], []
    for e in range(len(query)):
        m.set_support(poses=support[e])
        a, b = m.score(query[e:e + 1])
        lg.append(a)
        it.append(b)
    return torch.cat(lg), torch.cat(it)


# ---- 1. against the oracle, through TRXOS.forward with per-row support -----------------------------------------------
@pytest.mark.parametrize("cfg,b,debug", [
    (CFG_T32, 1, 0), (CFG_T32, 7, 0), (CFG_T32, 28, 0),
    (Cfg(seq_len=24), 9, 0),          # N=276: three query tiles, the odd tile pair
    (Cfg(seq_len=8), 300, 0),         # one tile, no normaliser pass; 300 episodes
    (Cfg(), 28, 4096),                # T=16 pairs moved off the pair pipeline by debug bit 4096
], ids=["t32_b1", "t32_b7", "t32_b28", "t24_b9", "t8_b300", "t16_bit4096_b28"])
def test_forward_per_row_support_matches_oracle(cfg, b, debug):
    m, sd = make_model(cfg, 0)
    o = TrxOracle(cfg, sd)
    if debug:
        m.debug_set(0, debug)
    support, query = episodes(cfg, b, cfg.way, 7 + b)
    labels = np.tile(np.arange(cfg.way, dtype=np.int32), (b, 1))
    S, L, Q = torch.from_numpy(support).cuda(), torch.from_numpy(labels).cuda(), torch.from_numpy(query).cuda()
    out = m({"sk": S}, L, {"sk": Q})
    assert m.last_path() == 3
    ref = o.forward({"sk": support}, labels, {"sk": query})
    check_oracle(out, ref)
    ssf = o.embed(torch.from_numpy(support))
    out2 = m(None, L, {"sk": Q}, ss_features=ssf.cuda())
    assert m.last_path() == 3
    check_oracle(out2, o.forward(None, labels, {"sk": query}, ss_features=ssf))


# ---- 2. batched == the per-episode sequence, bit for bit ---------------------------------------------------------------
def rowmax_model(cfg):
    """force_path = 2 with gamma past the overflow bound: the ROWMAX instance of the tiled kernel"""
    sd = dict(make_state_dict(cfg, 0))
    g = np.full(D, np.sqrt(1.01 * OVERFLOW_BOUND / np.sqrt(D)), np.float32)
    sd["transformers.0.norm_k.weight"] = g
    sd["transformers.0.norm_k.bias"] = np.zeros(D, np.float32)
    from isbfsar_b200 import TRXOS
    m = TRXOS(Args(cfg))
    m.load_state_dict(torch_sd(sd), strict=False)
    m.force_path = 2
    return m.cuda()


@pytest.mark.parametrize("shape", ["t32_pairs", "t8_pairs", "rowmax"])
def test_batched_equals_loop_bitwise(shape):
    if shape == "rowmax":
        cfg, b = Cfg(way=20, seq_len=32), 9
        m = rowmax_model(cfg)
    else:
        cfg, b = (CFG_T32, 28) if shape == "t32_pairs" else (Cfg(seq_len=8), 60)
        m, _ = make_model(cfg, 0)
    support, query = episodes(cfg, b, cfg.way, 11)
    S, Q = torch.from_numpy(support).cuda(), torch.from_numpy(query).cuda()
    lg, it = m.score_episodes(Q, poses=S)
    assert m.last_path() == 3
    rl, ri = loop(m, S, Q)
    assert m.last_path() == 3
    assert torch.equal(lg, rl) and torch.equal(it, ri)


# ---- 3. one pass split into several chunks (cls_base != 0) ------------------------------------------------------------
def test_chunked_pass_is_bit_identical():
    support, query = episodes(CFG_T32, 28, 20, 13)
    S, Q = torch.from_numpy(support).cuda(), torch.from_numpy(query).cuda()
    res = []
    for mc in (0, 3):
        m, _ = make_model(CFG_T32, 0, max_chunk=mc)
        res.append(m.score_episodes(Q, poses=S))
        assert m.last_path() == 3
    assert torch.equal(res[0][0], res[1][0]) and torch.equal(res[0][1], res[1][1])


# ---- 4. launches of one pass do not grow with the batch ---------------------------------------------------------------
def test_launch_count_one_pass():
    m, _ = make_model(CFG_T32, 0)
    support, query = episodes(CFG_T32, 28, 20, 17)
    S, Q = torch.from_numpy(support).cuda(), torch.from_numpy(query).cuda()
    m.score_episodes(Q, poses=S)                                 # one-time tables and allocations
    counts = []
    for b in (7, 28):
        l0 = m.launch_count()
        m.score_episodes(Q[:b], poses=S[:b])
        counts.append(m.launch_count() - l0)
    assert m.last_path() == 3
    assert counts[0] == counts[1] < 60, counts


# ---- 5. the pool is sized by memory and holds transformers[0] only ----------------------------------------------------
def test_pool_budget_and_transformer_state():
    cfg = CFG_T32
    m, sd = make_model(cfg, 0)
    o = TrxOracle(cfg, sd)
    support, query = episodes(cfg, 300, 20, 19)
    S, Q = torch.from_numpy(support).cuda(), torch.from_numpy(query).cuda()
    m.set_support(poses=S[0])
    torch.cuda.synchronize()
    free0 = torch.cuda.mem_get_info()[0]
    lg, it = m.score_episodes(Q, poses=S)
    torch.cuda.synchronize()
    drop = free0 - torch.cuda.mem_get_info()[0]
    assert drop < 4.5 * (1 << 30), drop / (1 << 30)
    e = slice(44, 54)                                            # across the boundary of the first pass (49 episodes)
    ref = o.forward({"sk": support[e]}, np.tile(np.arange(20, dtype=np.int32), (10, 1)), {"sk": query[e]})
    assert rel_err(lg[e].cpu(), ref["logits"]).max() < TOL_TC and rel_err(it[e].cpu(), ref["is_true"]).max() < TOL_TC
    # transformers[1] has no support operands until the support set is set again
    qf = m.embed(Q[:2])
    with pytest.raises(ArxError, match="ARX_ERR_STATE"):
        m.score_features(1, qf)
    m.set_support(poses=S[3])
    lo, io = m.score(Q[:4])
    rl, ri = o.score(support[3:4], np.arange(20)[None], query[:4])
    assert rel_err(lo.cpu(), rl).max() < TOL_TC and rel_err(io.cpu(), ri).max() < TOL_TC
    # triples (N=4960): the oracle would hold GBs of attention probabilities per window, so the reference is a handle
    # that never scored episodes (the same kernels and operands: bit-identical)
    fresh, _ = make_model(cfg, 0)
    fresh.set_support(poses=S[3])
    assert torch.equal(m.score_features(1, qf), fresh.score_features(1, fresh.embed(Q[:2])))


# ---- 6. the evaluation driver at the cfg4 shape -----------------------------------------------------------------------
def test_fsos_driver_cfg4_shape():
    m, sd = make_model(CFG_T32, 0)
    o = TrxOracle(CFG_T32, sd)
    kw = dict(n_batches=2, batch=8, way=20, seq_len=32, n_classes=30)
    got = evaluate_fsos(m, synthetic_fsos_episodes(**kw), 20, device="cuda")
    assert m.last_path() == 3
    ref = evaluate_fsos(lambda s, l, q: o.forward(s, l, q), synthetic_fsos_episodes(**kw), 20)
    assert got == ref and got["episodes"] == 16
    assert got["FS-ACC"] == 1.0


# ---- 7. the T=16 pair pipeline keeps 256 episodes per pass ------------------------------------------------------------
def test_pair_pipeline_unchanged():
    cfg = Cfg()
    m, _ = make_model(cfg, 0)
    support, query = episodes(cfg, 256, 5, 23)
    S, Q = torch.from_numpy(support).cuda(), torch.from_numpy(query).cuda()
    counts = {}
    for b in (28, 256):
        for _ in range(3):                                       # eager, captured, replayed: the same count
            l0 = m.launch_count()
            m.score_episodes(Q[:b], poses=S[:b])
            counts[b] = m.launch_count() - l0
            assert m.last_path() == 2
    assert counts[28] == counts[256], counts


# ---- 8. the pair pipeline with a pass larger than one chunk scores episode by episode ----------------------------------
def test_pair_pipeline_past_one_chunk_equals_loop():
    cfg = Cfg()
    m, _ = make_model(cfg, 0, max_chunk=100)                     # 256 episodes per pass do not fit one chunk
    support, query = episodes(cfg, 256, 5, 29)
    S, Q = torch.from_numpy(support).cuda(), torch.from_numpy(query).cuda()
    loop(m, S[:1], Q[:1])                                        # one-time tables of the handle's first scoring pass
    l0 = m.launch_count()
    lg, it = m.score_episodes(Q, poses=S)
    l1 = m.launch_count()
    assert m.last_path() == 2
    rl, ri = loop(m, S, Q)
    l2 = m.launch_count()
    assert torch.equal(lg, rl) and torch.equal(it, ri)
    assert l1 - l0 == l2 - l1, (l1 - l0, l2 - l1)
