"""Parity of the CUDA path (through the C ABI / the reference-shaped Python API) against the CPU oracle
and the golden vectors frozen from the unmodified reference.

Tolerances (BASELINE.json north_star): tuple indices bit-exact; logits and is_true within 1e-3 relative;
identical argmax and accept/reject on >= 99.9 % of windows.  The fp32 CUDA-core path is held to 5e-5."""
import os
from itertools import combinations

import numpy as np
import pytest
import torch

from oracle.synth import Cfg, make_episode, make_state_dict, make_heatmaps  # noqa: F401
from oracle.trx_oracle import TrxOracle
from tests.util import Args, make_model, rel_err, torch_sd

pytestmark = pytest.mark.gpu

TOL_TC = 1e-3       # stated tolerance (fp16 operands, fp32 accumulate)
TOL_FP32 = 5e-5     # fp32 path: summation-order noise only

CASES = [
    ("cfg1_w5_t16_structured", Cfg()),
    ("cfg1_w5_t16_iid", Cfg()),
    ("cfg1_w5_t16_affine", Cfg()),
    ("w3_t16_structured", Cfg()),
    ("cfg3_w60_t16", Cfg(way=60)),
    ("cfg4_w20_t32_pairs", Cfg(way=20, seq_len=32, temp_set=[2, 3])),
]
PATHS = [1, 0]      # 1 = fp32 kernels forced, 0 = auto (tcgen05 where available)


def tol_for(model):
    return TOL_FP32 if model.last_path() == 1 else TOL_TC


@pytest.mark.parametrize("T,c", [(4, 2), (8, 2), (16, 2), (32, 2), (8, 3), (16, 3), (32, 3)])
def test_tuple_table_bit_exact(T, c):
    m, _ = make_model(Cfg(seq_len=T, temp_set=[c], model="DISC" if c == 2 else "NONE"))
    tab = m.tuple_table(0).cpu().numpy()
    ref = np.array(list(combinations(range(T), c)), dtype=np.int32)
    assert tab.dtype == np.int32 and np.array_equal(tab, ref)
    assert [t.tolist() for t in m.transformers[0].tuples] == ref.tolist()
    assert m.transformers[0].tuples[0].dtype == torch.int64


@pytest.mark.parametrize("path", PATHS)
@pytest.mark.parametrize("name,cfg", CASES)
def test_scores_match_reference_golden(golden_dir, name, cfg, path):
    g = np.load(os.path.join(golden_dir, name + ".npz"))
    way, T, B, wseed, iseed, affine = [int(x) for x in g["meta"][:6]]
    m, sd = make_model(cfg, wseed, affine=bool(affine), force_path=path)
    support, labels, query, planted = make_episode(cfg, B, iseed, str(g["kind"]), way=way)
    m.set_support(poses=torch.from_numpy(support[0]).cuda())
    logits, is_true = m.score(torch.from_numpy(query).cuda())
    tol = tol_for(m)
    logits, is_true = logits.cpu().numpy(), is_true.cpu().numpy()
    assert rel_err(logits, g["logits"]).max() < tol
    assert rel_err(is_true, g["is_true"]).max() < tol
    if str(g["kind"]) == "structured":
        assert np.array_equal(logits.argmax(1), g["logits"].argmax(1))
    assert np.array_equal(is_true > 0.5, g["is_true"] > 0.5)
    np.testing.assert_allclose(m.support_features().cpu().numpy()[:2], g["support_features"], rtol=tol, atol=1e-6)


@pytest.mark.parametrize("path", PATHS)
@pytest.mark.parametrize("kind", ["structured", "iid"])
def test_scores_match_oracle_b512(kind, path):
    cfg = Cfg()
    m, sd = make_model(cfg, 0, force_path=path)
    support, labels, query, planted = make_episode(cfg, 512, 11, kind)
    o = TrxOracle(cfg, sd)
    lo, it = o.score(support, labels, query)
    m.set_support(poses=torch.from_numpy(support[0]).cuda())
    logits, is_true, chosen = m.score(torch.from_numpy(query).cuda(), want_chosen=True)
    tol = tol_for(m)
    logits, is_true = logits.cpu().numpy(), is_true.cpu().numpy()
    assert rel_err(logits, lo).max() < tol
    assert rel_err(is_true, it).max() < tol
    assert np.array_equal(chosen.cpu().numpy(), logits.argmax(1))
    if kind == "structured":
        assert (logits.argmax(1) == lo.argmax(1)).mean() >= 0.999
        assert (logits.argmax(1) == planted).all()
    else:   # ill-posed margins (SURVEY 8d): compare argmax only where the reference margin exceeds 2*tol
        srt = np.sort(lo, 1)
        ok = (srt[:, -1] - srt[:, -2]) / np.abs(srt[:, -1]) > 2 * tol
        assert (logits.argmax(1)[ok] == lo.argmax(1)[ok]).all()
    assert ((is_true > 0.5) == (it > 0.5)).mean() >= 0.999


def test_forward_reference_api():
    """forward(ss_data, ss_labels, query_data, ss_features) -- return dict, label order, cached/uncached."""
    cfg = Cfg()
    m, sd = make_model(cfg, 0)
    o = TrxOracle(cfg, sd)
    support, labels, query, _ = make_episode(cfg, 8, 21, "structured")
    S, Q = torch.from_numpy(support).cuda(), torch.from_numpy(query).cuda()
    out = m({"sk": S}, torch.from_numpy(labels).cuda(), {"sk": Q})
    assert set(out) == {"logits", "is_true", "prototypes", "support_features"}
    assert out["logits"].shape == (8, 5) and out["is_true"].shape == (8, 1)
    assert out["support_features"].shape == (1, 5, 16, 256)      # batch dim of the support given (model.py:315-317)
    ref = o.forward({"sk": np.repeat(support, 8, 0)}, labels, {"sk": query}, want=("prototypes",))
    tol = tol_for(m)
    assert rel_err(out["logits"].cpu(), ref["logits"]).max() < tol
    assert rel_err(out["is_true"].cpu(), ref["is_true"]).max() < tol
    np.testing.assert_allclose(out["support_features"][0].cpu().numpy(), ref["support_features"][0].numpy(), rtol=tol, atol=1e-6)
    # prototypes: list of W (b,1,N,D) (fp32 debug kernels)
    protos = out["prototypes"]
    assert len(protos) == 5 and protos[0].shape == (8, 1, 120, 128)
    np.testing.assert_allclose(protos[3].cpu().numpy(), ref["prototypes"][3].numpy(), rtol=1e-3, atol=2e-5)
    # cached path: ss_features expanded over the batch (ar.py:56-61 / SURVEY 3.3)
    ssf = out["support_features"][:1]
    out2 = m(None, torch.from_numpy(labels).cuda(), {"sk": Q}, ss_features=ssf.expand(8, -1, -1, -1))
    # (features given in fp32 enter the fp16 pipeline one stage later than poses do: equal within the tolerance)
    assert rel_err(out2["logits"].cpu(), out["logits"].cpu()).max() < tol
    assert rel_err(out2["logits"].cpu(), ref["logits"]).max() < tol
    # label permutation: logits column k belongs to class ss_labels[0][k]
    perm = np.array([[3, 1, 4, 0, 2]], dtype=np.int32)
    out3 = m({"sk": S}, torch.from_numpy(perm).cuda(), {"sk": Q})
    assert rel_err(out3["logits"].cpu(), out["logits"].cpu()[:, perm[0]]).max() < 1e-5
    # a subset of the classes (ar.py:51: labels = range(n) with a zero-padded feature stack)
    sub = np.array([[0, 1, 2]], dtype=np.int32)
    out4 = m(None, torch.from_numpy(sub).cuda(), {"sk": Q}, ss_features=ssf)
    assert out4["logits"].shape == (8, 3)
    ref4 = o.forward(None, sub, {"sk": query}, ss_features=ref["support_features"])
    assert rel_err(out4["logits"].cpu(), ref4["logits"]).max() < tol


def test_forward_per_episode_support():
    """Training/eval call shape (train.py:110-120): every batch row has its own support set."""
    cfg = Cfg()
    m, sd = make_model(cfg, 0)
    o = TrxOracle(cfg, sd)
    rng = np.random.default_rng(5)
    b = 4
    support = (0.17 * rng.standard_normal((b, 5, 16, 90))).astype(np.float32)
    query = (support[np.arange(b), rng.integers(0, 5, b)] + 0.05 * rng.standard_normal((b, 16, 90))).astype(np.float32)
    labels = np.tile(np.arange(5, dtype=np.int32), (b, 1))
    out = m({"sk": torch.from_numpy(support).cuda()}, torch.from_numpy(labels).cuda(), {"sk": torch.from_numpy(query).cuda()})
    ref = o.forward({"sk": support}, labels, {"sk": query})
    tol = tol_for(m)
    assert rel_err(out["logits"].cpu(), ref["logits"]).max() < tol
    assert rel_err(out["is_true"].cpu(), ref["is_true"]).max() < tol
    assert out["support_features"].shape == (b, 5, 16, 256)


@pytest.mark.parametrize("name,cfg,way_run", [("w5_t16_triples", Cfg(way=5, seq_len=16, temp_set=[2, 3]), 5),
                                              ("cfg4_w20_t32_triples", Cfg(way=20, seq_len=32, temp_set=[2, 3]), 20)])
def test_triple_transformer_logits(golden_dir, name, cfg, way_run):
    """Cardinality-3 transformer validated against ref.transformers[1](...)['logits'] (SURVEY 8d cfg4)."""
    g = np.load(os.path.join(golden_dir, name + ".npz"))
    way, T, B, wseed, iseed, ti = [int(x) for x in g["meta"][:6]]
    m, sd = make_model(cfg, wseed)
    support, labels, query, _ = make_episode(cfg, B, iseed, "structured")
    m.set_support(poses=torch.from_numpy(support[0]).cuda())
    qf = m.embed(torch.from_numpy(query).cuda())
    logits = m.score_features(ti, qf).cpu().numpy()
    assert rel_err(logits, g["logits"]).max() < tol_for(m)
    assert np.array_equal(m.tuple_table(ti).cpu().numpy(), g["tuples"].astype(np.int32))


def test_action_recognizer_stream(golden_dir):
    from isbfsar_b200 import ActionRecognizer
    g = np.load(os.path.join(golden_dir, "ar_stream.npz"))
    cfg = Cfg()
    ar = ActionRecognizer(Args(cfg), state_dict=torch_sd(make_state_dict(cfg, 0)))
    rng = np.random.default_rng(7)
    poses = (0.17 * rng.standard_normal((3, 16, 90))).astype(np.float32)
    frames = (0.17 * rng.standard_normal((23, 90))).astype(np.float32)
    frames[5:21] = poses[1] + 0.05 * rng.standard_normal((16, 90)).astype(np.float32)
    assert ar.inference(None) == ({}, 0, {})
    assert ar.inference({"sk": frames[0]}) == ({}, 0, {})
    for i, n in enumerate(["wave", "clap", "kick"]):
        ar.train({"flag": n, "data": {"poses": poses[i]}, "requires_focus": bool(i % 2)})
    probs, os_, empties = [], [], 0
    for f in range(20):
        res, o, rf = ar.inference({"sk": frames[f]})
        if len(res) == 0:
            empties += 1
            continue
        assert list(res.keys()) == ["wave", "clap", "kick"] and rf == {"wave": False, "clap": True, "kick": False}
        assert isinstance(o, np.ndarray) and o.shape == (1,)
        probs.append([res[k] for k in res])
        os_.append(float(o[0]))
    assert empties == int(g["empties"])
    assert rel_err(np.array(probs), g["probs"]).max() < 2e-3      # softmax of logits within 1e-3 relative
    assert rel_err(np.array(os_), g["open_set"]).max() < 1e-3
    assert np.array_equal(np.argmax(probs, 1), np.argmax(g["probs"], 1))
    feats = torch.stack([ar.support_set[k]["features"] for k in ["wave", "clap", "kick"]]).cpu().numpy()
    np.testing.assert_allclose(feats[:, :2], g["features"], rtol=1e-3, atol=1e-6)
    assert ar.remove("clap") and not ar.remove("nope")
    probs2 = []
    for f in range(20, 23):
        res, o, rf = ar.inference({"sk": frames[f]})
        probs2.append([res[k] for k in ["wave", "kick"]])
    assert rel_err(np.array(probs2), g["probs_after_remove"]).max() < 2e-3


def test_decode_heatmaps(golden_dir):
    from isbfsar_b200 import HeatmapDecoder
    g = np.load(os.path.join(golden_dir, "decode_64.npz"))
    m, _ = make_model(Cfg(), 0)
    dec = HeatmapDecoder(m, g["expand30"], None, g["new_K"], g["homo_inv"])
    hm = make_heatmaps(64, seed=2)
    poses, valid = dec.decode(torch.from_numpy(hm).cuda())
    assert valid.all() and np.array_equal(valid.cpu().numpy(), g["valid"])
    # fp32 soft-argmax vs the reference's float64 tail: 1e-4 of the pose scale
    ref = g["poses"]
    assert np.abs(poses.cpu().numpy() - ref).max() < 1e-4 * np.abs(ref).max()
    assert (poses[:, :3] == 0).all()           # root joint exactly zero (main.py:103)
    # frames with fewer than 1/4 of the joints inside the FOV are dropped (hpe.py:152-153)
    bad = torch.zeros((3, 8, 8, 288), device="cuda")
    bad[:, 0, 0, :] = 30.0                      # every joint piles up in the corner -> outside [18,238]
    p, v = dec.decode(bad)
    assert not v.any() and (p == 0).all()


def test_score_host_matches_device_and_chunking():
    cfg = Cfg()
    m, sd = make_model(cfg, 0, max_chunk=96)       # ragged chunks: 300 = 3*96 + 12
    support, labels, query, _ = make_episode(cfg, 300, 31, "structured")
    m.set_support(poses=torch.from_numpy(support[0]).cuda())
    a, b = m.score(torch.from_numpy(query).cuda())
    hq = torch.from_numpy(query).pin_memory()
    ha, hb = m.score_host(hq)
    assert torch.equal(a.cpu(), ha) and torch.equal(b.cpu(), hb)
    m2, _ = make_model(cfg, 0)
    m2.set_support(poses=torch.from_numpy(support[0]).cuda())
    a2, b2 = m2.score(torch.from_numpy(query).cuda())
    assert torch.equal(a2, a) and torch.equal(b2, b)                 # results independent of chunking
    # empty batch
    e, f = m.score(torch.zeros((0, 16, 90)).cuda())
    assert e.shape == (0, 5) and f.shape == (0, 1)


def test_full_size_properties_cfg2():
    """BASELINE cfg2 (4096 windows, 5-way): size-independent properties instead of the slow oracle."""
    cfg = Cfg()
    m, sd = make_model(cfg, 0)
    support, labels, query, planted = make_episode(cfg, 4096, 41, "structured")
    S, Q = torch.from_numpy(support[0]).cuda(), torch.from_numpy(query).cuda()
    m.set_support(poses=S)
    logits, is_true = m.score(Q)
    assert torch.isfinite(logits).all() and (logits < 0).all() and ((is_true > 0) & (is_true < 1)).all()
    assert (logits.argmax(1).cpu().numpy() == planted).all()
    # windows are independent: a permuted batch gives permuted rows, bit-identical
    perm = torch.randperm(4096, generator=torch.Generator().manual_seed(0)).cuda()
    l2, t2 = m.score(Q[perm])
    assert torch.equal(l2, logits[perm]) and torch.equal(t2, is_true[perm])
    # class permutation of the support set permutes the columns
    cp = torch.tensor([2, 0, 4, 1, 3]).cuda()
    m.set_support(poses=S[cp])
    l3, t3 = m.score(Q)
    assert rel_err(l3.cpu(), logits[:, cp].cpu()).max() < 1e-5
    assert rel_err(t3.cpu(), is_true.cpu()).max() < 1e-5
    # a query identical to a support class: that class wins
    m.set_support(poses=S)
    l4, _ = m.score(S)
    assert (l4.argmax(1).cpu() == torch.arange(5)).all()
    # subset oracle check on 64 of the windows
    o = TrxOracle(cfg, sd)
    lo, it = o.score(support, labels, query[:64])
    assert rel_err(logits[:64].cpu(), lo).max() < tol_for(m)
    assert rel_err(is_true[:64].cpu(), it).max() < tol_for(m)


def test_errors_are_loud():
    cfg = Cfg()
    m, _ = make_model(cfg, 0)
    with pytest.raises(RuntimeError):
        m.score(torch.zeros((1, 16, 90)).cuda())            # support not set
    from isbfsar_b200 import TRXOS
    cpu_model = TRXOS(Args(cfg))
    with pytest.raises(RuntimeError):
        cpu_model({"sk": torch.zeros(1, 5, 16, 90)}, torch.arange(5)[None], {"sk": torch.zeros(1, 16, 90)})


@pytest.mark.parametrize("B", [1, 3, 129, 257])
@pytest.mark.parametrize("way", [1, 2, 7])
def test_ragged_batches_and_odd_ways(B, way):
    """Tail handling of the persistent kernels: odd window counts (groups of 2), odd class counts."""
    cfg = Cfg(way=way)
    m, sd = make_model(cfg, 0)
    support, labels, query, planted = make_episode(cfg, B, 51 + B + way, "structured")
    o = TrxOracle(cfg, sd)
    lo, it = o.score(support, labels, query)
    m.set_support(poses=torch.from_numpy(support[0]).cuda())
    logits, is_true = m.score(torch.from_numpy(query).cuda())
    assert m.last_path() == 2
    assert rel_err(logits.cpu(), lo).max() < TOL_TC and rel_err(is_true.cpu(), it).max() < TOL_TC
    assert np.array_equal(logits.argmax(1).cpu().numpy(), lo.argmax(1))


def test_cfg3_60way_at_scale():
    """BASELINE cfg3 shape on one GPU: 60-way support, a rank's shard of the 65 536 windows (8192)."""
    cfg = Cfg(way=60)
    m, sd = make_model(cfg, 0)
    B = 8192
    support, labels, query, planted = make_episode(cfg, B, 61, "structured")
    m.set_support(poses=torch.from_numpy(support[0]).cuda())
    logits, is_true = m.score(torch.from_numpy(query).cuda())
    assert m.last_path() == 2 and logits.shape == (B, 60)
    assert (logits.argmax(1).cpu().numpy() == planted).all()
    o = TrxOracle(cfg, sd)
    idx = np.r_[0:16, B - 16:B]
    lo, it = o.score(support, labels, query[idx], chunk=16)
    assert rel_err(logits[idx].cpu(), lo).max() < TOL_TC and rel_err(is_true[idx].cpu(), it).max() < TOL_TC


def test_cfg5_heatmaps_to_scores_end_to_end(golden_dir):
    """BASELINE cfg5: 1024 synthetic heatmap frames -> decode kernel -> 1009 sliding windows -> AR scoring."""
    from isbfsar_b200 import HeatmapDecoder
    from oracle import decode_oracle as D
    g = np.load(os.path.join(golden_dir, "decode_64.npz"))
    cfg = Cfg()
    m, sd = make_model(cfg, 0)
    hm = make_heatmaps(1024, seed=2)
    dec = HeatmapDecoder(m, g["expand30"], None, g["new_K"], g["homo_inv"])
    poses, valid = dec.decode(torch.from_numpy(hm).cuda())
    assert valid.all()
    ref_poses, ref_valid = D.decode_frames(hm[:96], g["expand30"], np.arange(30), g["new_K"], g["homo_inv"])
    assert np.abs(poses[:96].cpu().numpy() - ref_poses).max() < 1e-4 * np.abs(ref_poses).max()
    windows = poses.unfold(0, 16, 1).permute(0, 2, 1).contiguous()            # (1009, 16, 90) sliding windows
    assert windows.shape == (1009, 16, 90)
    support = windows[[0, 200, 400, 600, 800]].clone()                          # 5 of the windows act as the support set
    m.set_support(poses=support)
    logits, is_true = m.score(windows)
    assert (logits[[0, 200, 400, 600, 800]].argmax(1).cpu() == torch.arange(5)).all()
    # oracle on the oracle-decoded poses of the first 80 windows (decode error 1e-4 of scale feeds through)
    o = TrxOracle(cfg, sd)
    ref_w = np.stack([ref_poses[i:i + 16] for i in range(80)]).astype(np.float32)
    lo, it = o.score(support.cpu().numpy()[None], np.arange(5)[None], ref_w)
    assert rel_err(logits[:80].cpu(), lo).max() < 5e-3
    assert np.array_equal(logits[:80].argmax(1).cpu().numpy(), lo.argmax(1))


def test_large_layernorm_affine_falls_back_to_fp32_kernels(capfd):
    """exp2 without max-subtraction and fp16 QK^T operands are only used inside the static LayerNorm bound (DESIGN 4);
    beyond it the fp32 kernels with an online max take over -- results stay within tolerance -- and the library says so
    once on stderr.  force_path=2 keeps such weights on tensor cores (row-max variant of the tiled kernels): overflow
    safe, but outside the 1e-3 tolerance, which is why it is not the default."""
    cfg = Cfg()
    sd = dict(make_state_dict(cfg, 0))
    sd["transformers.0.norm_k.weight"] = np.full((128,), 3.0, np.float32)
    support, labels, query, _ = make_episode(cfg, 64, 71, "structured")
    lo, it = TrxOracle(cfg, sd).score(support, labels, query)
    for force, path, tol in [(0, 1, 1e-3), (2, 3, 3e-2)]:
        m, _ = make_model(cfg, 0, force_path=force)
        with torch.no_grad():
            m.transformers[0].norm_k.weight.fill_(3.0)
        m.set_support(poses=torch.from_numpy(support[0]).cuda())
        logits, is_true = m.score(torch.from_numpy(query).cuda())
        logits2, _ = m.score(torch.from_numpy(query).cuda())
        assert m.last_path() == path
        assert rel_err(logits.cpu(), lo).max() < tol and rel_err(is_true.cpu(), it).max() < 1e-3
        assert np.array_equal(logits.argmax(1).cpu().numpy(), lo.argmax(1))
        err = capfd.readouterr().err
        assert err.count("outside the fp16 tensor-core bound") == (1 if force == 0 else 0)      # said once, not per call


def test_t8_runs_on_generic_tensor_core_kernels():
    """T=8 pairs (N=28): tiled any-N tcgen05 kernels (single tile), head by linearity on the same kernel."""
    cfg = Cfg(seq_len=8)
    m, sd = make_model(cfg, 0)
    support, labels, query, _ = make_episode(cfg, 130, 81, "structured")
    m.set_support(poses=torch.from_numpy(support[0]).cuda())
    logits, is_true = m.score(torch.from_numpy(query).cuda())
    assert m.last_path() == 3
    lo, it = TrxOracle(cfg, sd).score(support, labels, query)
    assert rel_err(logits.cpu(), lo).max() < TOL_TC and rel_err(is_true.cpu(), it).max() < TOL_TC


@pytest.mark.parametrize("variant,path", [(4, 3), (1024, 2), (2048, 2), (4096, 3), (4096 + 4, 3)])
def test_kernel_variants_agree(variant, path):
    """Kernel variants behind debug key 0 stay green: fp32 linear layers in front of the tiled attention (4),
    one-tile-per-CTA frame-MLP GEMMs (1024), head projection on the caller's stream (2048), the metric shape on the
    tiled any-N kernels (4096)."""
    cfg = Cfg()
    m, sd = make_model(cfg, 0)
    support, labels, query, _ = make_episode(cfg, 131, 91, "structured")
    lo, it = TrxOracle(cfg, sd).score(support, labels, query)
    m.debug_set(0, variant)                                    # before the support set: it selects the operands built
    m.set_support(poses=torch.from_numpy(support[0]).cuda())
    logits, is_true = m.score(torch.from_numpy(query).cuda())
    assert m.last_path() == path
    assert rel_err(logits.cpu(), lo).max() < TOL_TC and rel_err(is_true.cpu(), it).max() < TOL_TC
    assert np.array_equal(logits.argmax(1).cpu().numpy(), lo.argmax(1))


@pytest.mark.parametrize("key,value", [(3, 0), (3, 1000), (4, 2), (4, 3)])
def test_attention_schedule_knobs_agree(key, value):
    """Softmax-group scheduling (free-running / staggered instead of the MUFU token) and the FMA-pipe exp2 share of
    the attention kernel change timing, not results (odd window count: exercises the single-window tail group)."""
    cfg = Cfg()
    m, sd = make_model(cfg, 0)
    support, labels, query, _ = make_episode(cfg, 333, 92, "structured")
    lo, it = TrxOracle(cfg, sd).score(support, labels, query)
    m.set_support(poses=torch.from_numpy(support[0]).cuda())
    m.debug_set(key, value)
    logits, is_true = m.score(torch.from_numpy(query).cuda())
    assert m.last_path() == 2
    assert rel_err(logits.cpu(), lo).max() < TOL_TC and rel_err(is_true.cpu(), it).max() < TOL_TC


def test_persistent_gemm_path_large_batch():
    """Batches of >= 2 row tiles per SM take the persistent weight-resident frame-MLP GEMMs; same scores as the
    one-tile-per-CTA kernels (variant 1024) on the same windows, and parity with the oracle on a sample."""
    cfg = Cfg()
    m, sd = make_model(cfg, 0)
    n = 2 * 148 * 8 + 13                      # > 2 tiles per SM, ragged tail
    support, labels, query, _ = make_episode(cfg, n, 93, "structured")
    m.set_support(poses=torch.from_numpy(support[0]).cuda())
    Q = torch.from_numpy(query).cuda()
    a_lo, a_it = m.score(Q)
    m.debug_set(0, 1024)
    b_lo, b_it = m.score(Q)
    assert torch.equal(a_lo, b_lo) and torch.equal(a_it, b_it)
    lo, it = TrxOracle(cfg, sd).score(support, labels, query[-64:])
    assert rel_err(a_lo[-64:].cpu(), lo).max() < TOL_TC and rel_err(a_it[-64:].cpu(), it).max() < TOL_TC


def test_fused_frame_mlp_is_bit_identical():
    """Big batches embed the frames with ONE fused kernel (poses -> fc1 -> fc2 -> feature image, arx_mlp_p.cu); variant 8192 keeps
    the three launches it replaces.  Same operands, same rounding: the scores must agree bit for bit -- fp32 rows on the device,
    fp32 and fp16 rows through the host-buffer entry points (ragged last row tile)."""
    cfg = Cfg()
    m, sd = make_model(cfg, 0)
    n = 2 * 148 * 8 + 13
    support, labels, query, _ = make_episode(cfg, n, 95, "structured")
    m.set_support(poses=torch.from_numpy(support[0]).cuda())
    Q = torch.from_numpy(query).cuda()
    a_lo, a_it = m.score(Q)
    launches = m.launch_count()
    m.score(Q)
    fused_launches = m.launch_count() - launches
    m.debug_set(0, 8192)
    b_lo, b_it = m.score(Q)
    launches = m.launch_count()
    m.score(Q)
    assert m.launch_count() - launches == fused_launches + 2          # pose image + fc1 + fc2 instead of one launch
    assert torch.equal(a_lo, b_lo) and torch.equal(a_it, b_it)
    lo, it = TrxOracle(cfg, sd).score(support, labels, query[-64:])
    assert rel_err(a_lo[-64:].cpu(), lo).max() < TOL_TC and rel_err(a_it[-64:].cpu(), it).max() < TOL_TC
    # host rows: two chunks of >= 2 tiles per SM each, fp32 and fp16
    nb = 2 * (2 * 148 * 8 + 40)
    support, labels, query, _ = make_episode(cfg, nb, 96, "structured")
    q16 = torch.from_numpy(query).to(torch.float16)
    q32 = q16.to(torch.float32)
    res = {}
    for bits in (0, 8192):
        m.debug_set(0, bits)
        res[bits] = (m.score_host(q32.pin_memory()), m.score_host(q16.pin_memory()))
    m.debug_set(0, 0)
    for k in range(2):
        assert torch.equal(res[0][0][k], res[8192][0][k]) and torch.equal(res[0][1][k], res[8192][1][k])
        assert torch.equal(res[0][0][k], res[0][1][k])


@pytest.mark.parametrize("variant", [16384, 32768, 8192 | 16384 | 32768])
def test_big_batch_scheduling_variants_are_bit_identical(variant):
    """Debug bits that only change SCHEDULING -- no L2 prefetch in the head kernel (16384), front-end kernels on every SM while the
    support chain is still in flight (32768) -- must not change a single bit; the support set is re-processed right before
    every scoring pass so that the reserved-SM path is the one exercised."""
    cfg = Cfg()
    m, sd = make_model(cfg, 0)
    n = 2 * 148 * 8 + 77
    support, labels, query, _ = make_episode(cfg, n, 97, "iid")
    S, Q = torch.from_numpy(support[0]).cuda(), torch.from_numpy(query).cuda()
    out = {}
    for bits in (0, variant):
        m.debug_set(0, bits)
        for _ in range(2):                                         # second pass: the replayed graphs
            m.set_support(poses=S)
            lo, it = m.score(Q)
        out[bits] = (lo.clone(), it.clone())
    m.debug_set(0, 0)
    assert torch.equal(out[0][0], out[variant][0]) and torch.equal(out[0][1], out[variant][1])
    rlo, rit = TrxOracle(cfg, sd).score(support, labels, query[:64])
    assert rel_err(out[0][0][:64].cpu(), rlo).max() < TOL_TC and rel_err(out[0][1][:64].cpu(), rit).max() < TOL_TC


def test_streaming_host_api_matches_device_path():
    """arx_score_host_submit/_wait: several requests in flight, interleaved with blocking and device-side calls and a
    support-set change; every result equals the device path bit for bit."""
    cfg = Cfg()
    m, sd = make_model(cfg, 0)
    support, labels, query, _ = make_episode(cfg, 700, 101, "structured")
    S = torch.from_numpy(support[0]).cuda()
    m.set_support(poses=S)
    qs = [torch.from_numpy(query[i * 100:(i + 1) * 100 + 37 * (i % 2)]).pin_memory() for i in range(6)]   # ragged sizes
    tickets = [m.score_host_async(q) for q in qs[:3]]
    dev = [m.score(q.cuda()) for q in qs]                       # device-side calls share the workspace with the streamed ones
    tickets += [m.score_host_async(q) for q in qs[3:]]
    blocking = m.score_host(qs[0])
    for q, t, d in zip(qs, tickets, dev):
        lo, it = t.result()
        assert torch.equal(lo, d[0].cpu()) and torch.equal(it, d[1].cpu())
    assert torch.equal(blocking[0], dev[0][0].cpu())
    # change the support set while nothing is in flight, stream again
    m.set_support(poses=S.flip(0))
    t = m.score_host_async(qs[1])
    lo, it = t.result()
    ref = m.score(qs[1].cuda())
    assert torch.equal(lo, ref[0].cpu()) and torch.equal(lo, dev[1][0].cpu().flip(1))


def test_export_import_support_roundtrip():
    """The NCCL payload: tuple embeddings exported from one handle and imported into another (same weights) give
    bit-identical scores; the importing handle cannot serve 'support_features'."""
    cfg = Cfg()
    m1, sd = make_model(cfg, 0)
    m2, _ = make_model(cfg, 0)
    support, labels, query, _ = make_episode(cfg, 200, 111, "structured")
    Q = torch.from_numpy(query).cuda()
    m1.set_support(poses=torch.from_numpy(support[0]).cuda())
    blob = m1.export_support()
    assert blob.numel() == 2 * 5 * 120 * 128
    m2.import_support(blob, 5)
    a, b = m1.score(Q)
    c, d = m2.score(Q)
    assert m2.last_path() == 2 and torch.equal(a, c) and torch.equal(b, d)
    with pytest.raises(RuntimeError):
        m2.support_features()


# ----------------------------------------------------------------------------------------------------------------------
# Round 2: the acceptance criteria at FULL size (SURVEY 8d), ties, hooks, cache round trip, episodes, API races
# ----------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kind", ["structured", "iid"])
def test_cfg2_all_4096_windows_against_oracle(kind):
    """BASELINE cfg2 acceptance on EVERY window: logits / is_true within 1e-3 relative; identical argmax and identical
    accept/reject on >= 99.9 % of the windows (structured inputs; iid inputs conditioned on the reference margin)."""
    cfg = Cfg()
    m, sd = make_model(cfg, 0)
    support, labels, query, planted = make_episode(cfg, 4096, 41, kind)
    m.set_support(poses=torch.from_numpy(support[0]).cuda())
    logits, is_true = m.score(torch.from_numpy(query).cuda())
    assert m.last_path() == 2
    lo, it = TrxOracle(cfg, sd).score(support, labels, query)
    logits, is_true = logits.cpu().numpy(), is_true.cpu().numpy()
    assert rel_err(logits, lo).max() < TOL_TC and rel_err(is_true, it).max() < TOL_TC
    if kind == "structured":
        assert (logits.argmax(1) == lo.argmax(1)).mean() >= 0.999
    else:
        srt = np.sort(lo, 1)
        ok = (srt[:, -1] - srt[:, -2]) / np.abs(srt[:, -1]) > 2 * TOL_TC
        assert ok.mean() > 0.5 and (logits.argmax(1)[ok] == lo.argmax(1)[ok]).all()
    assert ((is_true > 0.5) == (it > 0.5)).mean() >= 0.999


def test_cfg3_65536_windows_60way_1024_oracle_checked():
    """BASELINE cfg3 at full size on one GPU: 60-way x 65 536 windows; 1024 windows spread over the batch meet the oracle."""
    cfg = Cfg(way=60)
    m, sd = make_model(cfg, 0)
    B = 65536
    support, labels, query, planted = make_episode(cfg, B, 61, "structured")
    m.set_support(poses=torch.from_numpy(support[0]).cuda())
    logits, is_true = m.score(torch.from_numpy(query).cuda())
    assert m.last_path() == 2 and logits.shape == (B, 60)
    assert (logits.argmax(1).cpu().numpy() == planted).all()
    idx = np.r_[0:256, 20000:20256, 40001:40257, B - 256:B]
    lo, it = TrxOracle(cfg, sd).score(support, labels, query[idx], chunk=64)
    assert rel_err(logits[idx].cpu(), lo).max() < TOL_TC and rel_err(is_true[idx].cpu(), it).max() < TOL_TC
    assert np.array_equal(logits[idx].argmax(1).cpu().numpy(), lo.argmax(1))
    assert np.array_equal((is_true[idx] > 0.5).cpu().numpy(), it > 0.5)


def test_cfg4_t32_pairs_64_windows_against_oracle():
    """BASELINE cfg4 (i): T=32, 20-way, pair tuples N=496 -> logits + is_true (discriminator fc1 = (256, 15 872))."""
    cfg = Cfg(way=20, seq_len=32, temp_set=[2, 3])
    m, sd = make_model(cfg, 0)
    support, labels, query, planted = make_episode(cfg, 64, 5, "structured")
    m.set_support(poses=torch.from_numpy(support[0]).cuda())
    logits, is_true = m.score(torch.from_numpy(query).cuda())
    lo, it = TrxOracle(cfg, sd).score(support, labels, query, chunk=16)
    tol = tol_for(m)
    assert m.last_path() == 3                       # tiled tcgen05 kernels: 4 query tiles x 4 support tiles, two passes
    assert rel_err(logits.cpu(), lo).max() < tol and rel_err(is_true.cpu(), it).max() < tol
    assert np.array_equal(logits.argmax(1).cpu().numpy(), lo.argmax(1)) and (lo.argmax(1) == planted).all()
    assert np.array_equal((is_true > 0.5).cpu().numpy(), it > 0.5)


@pytest.mark.parametrize("T,way,B", [(16, 5, 8), (32, 20, 2)])
def test_triples_against_oracle(T, way, B):
    """Cardinality-3 transformer (cfg4 (ii)) against the oracle's transformers[1] restatement at B >= 2."""
    cfg = Cfg(way=way, seq_len=T, temp_set=[2, 3])
    m, sd = make_model(cfg, 0)
    support, labels, query, _ = make_episode(cfg, B, 9, "structured")
    m.set_support(poses=torch.from_numpy(support[0]).cuda())
    qf = m.embed(torch.from_numpy(query).cuda())
    logits = m.score_features(1, qf).cpu().numpy()
    o = TrxOracle(cfg, sd)
    with torch.no_grad():
        ssf = o.embed(torch.from_numpy(support))
        ref = o.cross_transformer(ssf.expand(B, -1, -1, -1), torch.from_numpy(labels).long(), o.embed(torch.from_numpy(query)).unsqueeze(1), ti=1)
    assert m.last_path() == 3
    assert rel_err(logits, ref["logits"].numpy()).max() < tol_for(m)
    assert np.array_equal(logits.argmax(1), ref["logits"].numpy().argmax(1))


def test_argmax_tie_takes_first_class():
    """model.py:323: torch.argmax returns the FIRST maximal index -- two identical support classes tie exactly."""
    cfg = Cfg()
    m, sd = make_model(cfg, 0)
    support, labels, query, planted = make_episode(cfg, 257, 13, "structured")
    support[0, 3] = support[0, 1]                       # class 3 is a copy of class 1
    query = (support[0, np.where(planted == 3, 1, planted)] + np.float32(0.05) * np.random.default_rng(3).standard_normal(query.shape)).astype(np.float32)
    m.set_support(poses=torch.from_numpy(support[0]).cuda())
    logits, is_true, chosen = m.score(torch.from_numpy(query).cuda(), want_chosen=True)
    lg = logits.cpu().numpy()
    assert np.array_equal(lg[:, 1], lg[:, 3])           # same operands, same arithmetic: bit-identical columns
    ch = chosen.cpu().numpy()
    assert np.array_equal(ch, lg.argmax(1))             # numpy argmax is first-max too
    assert (ch != 3).all() and (ch[(planted == 1) | (planted == 3)] == 1).all()
    lo, it = TrxOracle(cfg, sd).score(support, labels, query)
    assert np.array_equal(ch, lo.argmax(1))
    assert rel_err(is_true.cpu(), it).max() < TOL_TC


def test_add_hook_scores_match_oracle_probs():
    """add_hook=True: transformers[0].scores gets one (b,1,N,N) softmax tensor per class (model.py:110-111), the
    tensor visualize_heatmaps.py:123 reads; columns are normalised over the QUERY axis."""
    from isbfsar_b200 import TRXOS
    cfg = Cfg()
    sd = make_state_dict(cfg, 0)
    m = TRXOS(Args(cfg), add_hook=True)
    m.load_state_dict(torch_sd(sd), strict=False)
    m = m.cuda()
    support, labels, query, _ = make_episode(cfg, 3, 17, "structured")
    out = m({"sk": torch.from_numpy(support).cuda()}, torch.from_numpy(labels).cuda(), {"sk": torch.from_numpy(query).cuda()})
    scores = m.transformers[0].scores
    assert len(scores) == 5 and scores[0].shape == (3, 1, 120, 120)
    ref = TrxOracle(cfg, sd).forward({"sk": np.repeat(support, 3, 0)}, labels, {"sk": query}, want=("probs",))
    for c in range(5):
        got = scores[c].cpu().numpy()
        np.testing.assert_allclose(got, ref["probs"][c].numpy(), rtol=1e-3, atol=1e-7)     # the stated tolerance
        np.testing.assert_allclose(got.sum(axis=-2), 1.0, rtol=1e-5)
    true_index = 2                                       # the consumer's indexing (visualize_heatmaps.py:123)
    assert scores[true_index][0][0].shape == (120, 120)
    m({"sk": torch.from_numpy(support).cuda()}, torch.from_numpy(labels).cuda(), {"sk": torch.from_numpy(query).cuda()})
    assert len(m.transformers[0].scores) == 10           # the hook appends on every forward, like the reference


def test_support_cache_round_trip_is_stable():
    """ar.py:56-74: a support set scored from poses caches its features; afterwards (and after `load` of a saved set) the
    classes re-enter through the features path.  Both routes must give the same result on the same window within the
    tolerance, and both must match the reference logic."""
    from isbfsar_b200 import ActionRecognizer
    from oracle.trx_oracle import ActionRecognizerOracle
    cfg = Cfg()
    sd = make_state_dict(cfg, 0)
    rng = np.random.default_rng(23)
    poses = (0.17 * rng.standard_normal((3, 16, 90))).astype(np.float32)
    frames = (poses[1][np.arange(18) % 16] + 0.05 * rng.standard_normal((18, 90))).astype(np.float32)

    def run(ar, fs):
        out = None
        for f in fs:
            out = ar.inference({"sk": f})
        return out

    ar = ActionRecognizer(Args(cfg), state_dict=torch_sd(sd))
    oa = ActionRecognizerOracle(cfg, sd)
    for i, n in enumerate(["a", "b"]):
        inp = {"flag": n, "data": {"poses": poses[i]}, "requires_focus": False}
        ar.train(inp)
        oa.train(inp)
    assert run(ar, frames[:15]) == ({}, 0, {})
    assert not any("features" in v for v in ar.support_set.values())            # nothing is cached before the first full window
    res1, os1, _ = ar.inference({"sk": frames[15]})                              # poses route
    ro1, oo1, _ = run(oa, frames[:16])
    assert all("features" in v for v in ar.support_set.values())
    for k in res1:
        assert abs(res1[k] / ro1[k] - 1) < 2e-3
    assert abs(os1[0] / oo1[0] - 1) < 1e-3
    # a second recogniser that starts from the CACHED features (what main.py `load` restores): features route, same window
    ar2 = ActionRecognizer(Args(cfg), state_dict=torch_sd(sd))
    for n in ["a", "b"]:
        ar2.support_set[n] = {k: v.clone() for k, v in ar.support_set[n].items()}
        ar2.requires_focus[n] = False
    res3, os3, _ = run(ar2, frames[:16])
    for k in res1:
        assert abs(res3[k] / res1[k] - 1) < 1e-3
    assert abs(os3[0] / os1[0] - 1) < 1e-3
    # the window keeps sliding on both routes
    for f in frames[16:]:
        r1, _, _ = ar.inference({"sk": f})
        r3, _, _ = ar2.inference({"sk": f})
        ro, _, _ = oa.inference({"sk": f})
        for k in r1:
            assert abs(r1[k] / ro[k] - 1) < 2e-3 and abs(r3[k] / ro[k] - 1) < 2e-3
    # a third class arrives without features: the whole set goes back through the poses route (ar.py:62-67)
    inp = {"flag": "c", "data": {"poses": poses[2]}, "requires_focus": False}
    ar.train(inp)
    oa.train(inp)
    r4, _, _ = ar.inference({"sk": frames[-1]})
    ro4, _, _ = oa.inference({"sk": frames[-1]})
    assert list(r4) == ["a", "b", "c"]
    for k in r4:
        assert abs(r4[k] / ro4[k] - 1) < 2e-3
    # in-place edit of a stored tensor must not leave stale operands on the device (ADVICE r1)
    ar.support_set["a"]["poses"].copy_(torch.from_numpy(poses[2]).cuda())
    ar.support_set["a"].pop("features")
    oa.support_set["a"]["poses"] = torch.from_numpy(poses[2])
    oa.support_set["a"].pop("features")
    r5, _, _ = ar.inference({"sk": frames[-1]})
    ro5, _, _ = oa.inference({"sk": frames[-1]})
    for k in r5:
        assert abs(r5[k] / ro5[k] - 1) < 2e-3
    # the caller clears the window (previous_frames = []): the device ring follows
    ar.previous_frames = []
    oa.previous_frames = []
    assert run(ar, frames[:15]) == ({}, 0, {})
    r6, _, _ = ar.inference({"sk": frames[15]})
    ro6, _, _ = run(oa, frames[:16])
    for k in r6:
        assert abs(r6[k] / ro6[k] - 1) < 2e-3


def test_streaming_path_matches_windowed_scoring():
    """arx_stream_push (ring of per-frame projections, one frame per call) against arx_score on the explicit windows."""
    cfg = Cfg()
    m, sd = make_model(cfg, 0)
    rng = np.random.default_rng(31)
    support = (0.17 * rng.standard_normal((5, 16, 90))).astype(np.float32)
    frames = np.concatenate([support[2] + 0.05 * rng.standard_normal((16, 90)), 0.17 * rng.standard_normal((24, 90))]).astype(np.float32)
    m.set_support(poses=torch.from_numpy(support).cuda())
    got = []
    for i, f in enumerate(frames):
        probs, is_true, valid = m.stream_push(f)
        assert valid == (i >= 15)
        if valid:
            got.append(np.concatenate([probs, is_true]))
    assert m.last_path() == 3
    windows = np.stack([frames[i:i + 16] for i in range(len(frames) - 15)])
    lo, it = TrxOracle(cfg, sd).score(support[None], np.arange(5)[None], windows)
    ref = np.concatenate([torch.softmax(torch.from_numpy(lo), 1).numpy(), it], axis=1)
    assert rel_err(np.array(got), ref).max() < 2e-3
    assert np.array_equal(np.array(got)[:, :5].argmax(1), lo.argmax(1))
    # a support-set change between frames is picked up; reset forgets the window
    m.set_support(poses=torch.from_numpy(support[::-1].copy()).cuda())
    probs, is_true, valid = m.stream_push(frames[0])
    w = np.concatenate([frames[-15:], frames[:1]])[None]
    lo2, it2 = TrxOracle(cfg, sd).score(support[::-1].copy()[None], np.arange(5)[None], w)
    assert rel_err(probs, torch.softmax(torch.from_numpy(lo2), 1).numpy()[0]).max() < 2e-3
    m.stream_reset()
    assert m.stream_push(frames[0])[2] is False


@pytest.mark.parametrize("b", [1, 28, 300])
def test_batched_episodes_match_oracle(b):
    """train.py:110-120 / compute_fsos.py:89-98 call shape: every batch row has its own 5-way support set; all rows
    go through ONE batched pass (arx_score_episodes)."""
    cfg = Cfg()
    m, sd = make_model(cfg, 0)
    o = TrxOracle(cfg, sd)
    rng = np.random.default_rng(5 + b)
    support = (0.17 * rng.standard_normal((b, 5, 16, 90))).astype(np.float32)
    query = (support[np.arange(b), rng.integers(0, 5, b)] + 0.05 * rng.standard_normal((b, 16, 90))).astype(np.float32)
    labels = np.tile(np.arange(5, dtype=np.int32), (b, 1))
    l0 = m.launch_count()
    out = m({"sk": torch.from_numpy(support).cuda()}, torch.from_numpy(labels).cuda(), {"sk": torch.from_numpy(query).cuda()})
    assert m.launch_count() - l0 < 60 * (1 + b // 256)         # batched: launches do not grow with b
    ref = o.forward({"sk": support}, labels, {"sk": query})
    assert rel_err(out["logits"].cpu(), ref["logits"]).max() < TOL_TC
    assert rel_err(out["is_true"].cpu(), ref["is_true"]).max() < TOL_TC
    assert np.array_equal(out["logits"].argmax(1).cpu().numpy(), ref["logits"].numpy().argmax(1))
    # features route
    ssf = o.embed(torch.from_numpy(support))
    out2 = m(None, torch.from_numpy(labels).cuda(), {"sk": torch.from_numpy(query).cuda()}, ss_features=ssf.cuda())
    assert rel_err(out2["logits"].cpu(), ref["logits"]).max() < TOL_TC
    # the pool replaced the support set: an ordinary score afterwards needs set_support again and is unaffected
    m.set_support(poses=torch.from_numpy(support[0]).cuda())
    lg, _ = m.score(torch.from_numpy(query[:4]).cuda())
    lo, _ = o.score(support[:1], labels[:1], query[:4])
    assert rel_err(lg.cpu(), lo).max() < TOL_TC


def test_episodes_on_shapes_without_batched_kernels():
    """T=8 has no batched-episode kernels: arx_score_episodes falls back to one episode at a time, same results."""
    cfg = Cfg(seq_len=8)
    m, sd = make_model(cfg, 0)
    o = TrxOracle(cfg, sd)
    rng = np.random.default_rng(2)
    support = (0.17 * rng.standard_normal((5, 5, 8, 90))).astype(np.float32)
    query = (support[np.arange(5), rng.integers(0, 5, 5)] + 0.05 * rng.standard_normal((5, 8, 90))).astype(np.float32)
    labels = np.tile(np.arange(5, dtype=np.int32), (5, 1))
    lg, it = m.score_episodes(torch.from_numpy(query).cuda(), poses=torch.from_numpy(support).cuda())
    ref = o.forward({"sk": support}, labels, {"sk": query})
    assert rel_err(lg.cpu(), ref["logits"]).max() < TOL_TC and rel_err(it.cpu(), ref["is_true"]).max() < TOL_TC


def test_fsos_evaluation_driver_matches_oracle():
    """compute_fsos.py:74-143 over synthetic loader-shaped episodes: identical FS / OS / FSOS accuracies from the
    oracle and from the CUDA path (decisions agree on every episode)."""
    from isbfsar_b200.eval import evaluate_fsos, synthetic_fsos_episodes
    cfg = Cfg()
    m, sd = make_model(cfg, 0)
    o = TrxOracle(cfg, sd)
    kw = dict(n_batches=4, batch=28, way=5, seed=3)
    got = evaluate_fsos(m, synthetic_fsos_episodes(**kw), 5, device="cuda")
    ref = evaluate_fsos(lambda s, l, q: o.forward(s, l, q), synthetic_fsos_episodes(**kw), 5)
    assert got == ref and got["episodes"] == 112
    assert got["FS-ACC"] == 1.0                               # a noisy copy of an exemplar is recognised
    assert 0.0 <= got["FSOS-ACC"] <= 1.0 and 0.0 <= got["OS-ACC"] <= 1.0


def test_reference_support_set_pickle_interchange(golden_dir):
    """main.py:321-333: the GUI saves/loads `ar.support_set` (an OrderedDict of CUDA tensors) with pickle.  The
    reference's own saved file must drop into ActionRecognizer and behave like the reference logic on it."""
    import pickle
    from isbfsar_b200 import ActionRecognizer
    from oracle.trx_oracle import ActionRecognizerOracle
    cfg = Cfg()
    sd = make_state_dict(cfg, 0)
    ar = ActionRecognizer(Args(cfg), state_dict=torch_sd(sd))
    with open(os.path.join(golden_dir, "ref_support_set.pkl"), "rb") as f:
        ar.support_set = pickle.load(f)                      # main.py:329-330
    with open(os.path.join(golden_dir, "ref_requires_focus.pkl"), "rb") as f:
        ar.requires_focus = pickle.load(f)
    assert list(ar.support_set) == ["hello", "get", "lift"] and ar.support_set["get"]["poses"].is_cuda
    oa = ActionRecognizerOracle(cfg, sd)
    for k, v in ar.support_set.items():
        oa.support_set[k] = {kk: vv.detach().cpu().clone() for kk, vv in v.items()}
    oa.requires_focus = dict(ar.requires_focus)
    frames = (ar.support_set["get"]["poses"].cpu().numpy() + 0.02 * np.random.default_rng(1).standard_normal((16, 90))).astype(np.float32)
    for f in frames:
        res, os_, rf = ar.inference({"sk": f})
        ro, oo, _ = oa.inference({"sk": f})
    assert list(res) == ["hello", "get", "lift"] and rf == {"hello": True, "get": True, "lift": False}
    for k in res:                                            # the file carries cached features: features route (ar.py:56-61)
        assert abs(res[k] / ro[k] - 1) < 2e-3
    assert abs(os_[0] / oo[0] - 1) < 1e-3
    # drop the cached features: the poses route on the real recorded skeletons
    for v in ar.support_set.values():
        v.pop("features")
    for v in oa.support_set.values():
        v.pop("features")
    res2, os2, _ = ar.inference({"sk": frames[-1]})
    ro2, oo2, _ = oa.inference({"sk": frames[-1]})
    for k in res2:
        assert abs(res2[k] / ro2[k] - 1) < 2e-3
    assert max(res2, key=res2.get) == max(ro2, key=ro2.get)
    # save -> load round trip (main.py:321-333)
    blob = pickle.dumps(ar.support_set)
    ar.support_set = pickle.loads(blob)
    res3, _, _ = ar.inference({"sk": frames[-1]})
    ar.previous_frames = ar.previous_frames[:-1]
    assert all(abs(res3[k] / res2[k] - 1) < 1e-3 for k in res2)


def test_host_wait_on_old_tickets_and_two_caller_streams():
    """ADVICE r1: waiting on the OLDEST of several in-flight tickets must block until its copies have landed; ticket
    ids stay valid across a staging reallocation; scoring calls on two caller streams do not race on the workspace."""
    cfg = Cfg()
    m, sd = make_model(cfg, 0)
    support, labels, query, _ = make_episode(cfg, 4096, 121, "structured")
    m.set_support(poses=torch.from_numpy(support[0]).cuda())
    ref, _ = m.score(torch.from_numpy(query).cuda())
    ref = ref.cpu()
    q = torch.from_numpy(query).pin_memory()
    for _ in range(2):                                      # sized once: no reallocation (and no device-wide sync) below
        m.score_host_async(q).result()
    tickets = [m.score_host_async(q) for _ in range(5)]
    lo, _ = tickets[0].result()                             # slot already reused twice
    assert torch.equal(lo, ref)
    for t in tickets[1:]:
        assert torch.equal(t.result()[0], ref)
    small = m.score_host_async(q[:100])
    big = m.score_host_async(torch.cat([q, q]).pin_memory())   # larger request: staging reallocated
    assert torch.equal(small.result()[0], ref[:100])
    assert torch.equal(big.result()[0], torch.cat([ref, ref]))
    # two caller streams, same handle
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
    Q1, Q2 = torch.from_numpy(query[:2048]).cuda(), torch.from_numpy(query[2048:]).cuda()
    torch.cuda.synchronize()
    outs = []
    for _ in range(3):
        with torch.cuda.stream(s1):
            a = m.score(Q1)[0]
        with torch.cuda.stream(s2):
            b = m.score(Q2)[0]
        outs.append((a, b))
    torch.cuda.synchronize()
    for a, b in outs:
        assert torch.equal(a.cpu(), ref[:2048]) and torch.equal(b.cpu(), ref[2048:])


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs in one process")
def test_second_device_in_same_process():
    """ADVICE r1: per-device one-time initialisation (__constant__ slot tables, function attributes) is per handle."""
    cfg = Cfg()
    m, sd = make_model(cfg, 0)
    support, labels, query, _ = make_episode(cfg, 300, 131, "structured")
    m.set_support(poses=torch.from_numpy(support[0]).cuda())
    a, b = m.score(torch.from_numpy(query).cuda())
    m2, _ = make_model(cfg, 0)
    m2 = m2.to("cuda:1")
    with torch.cuda.device(1):
        m2.set_support(poses=torch.from_numpy(support[0]).to("cuda:1"))
        c, d = m2.score(torch.from_numpy(query).to("cuda:1"))
    assert torch.equal(a.cpu(), c.cpu()) and torch.equal(b.cpu(), d.cpu())


def test_tta_decode_per_crop_cameras(golden_dir):
    """Test-time augmentation (hpe.py:87-93, misc.py:310-327): five crops, each decoded with its own scaled intrinsics and its own
    rotation/flip, in one launch; per-crop poses against the reference's decode of that crop."""
    from isbfsar_b200 import HeatmapDecoder
    g = np.load(os.path.join(golden_dir, "tta_5.npz"))
    d64 = np.load(os.path.join(golden_dir, "decode_64.npz"))
    m, _ = make_model(Cfg(), 0)
    dec = HeatmapDecoder(m, d64["expand30"], None, g["base_K"], g["base_R"])
    hm = torch.from_numpy(make_heatmaps(5, seed=4)).cuda()
    poses, valid, mean = dec.decode_tta(hm)
    assert valid.all()
    ref = g["poses"]
    assert np.abs(poses.cpu().numpy() - ref).max() < 1e-4 * np.abs(ref).max()
    assert np.abs(mean.cpu().numpy() - ref.mean(0)).max() < 1e-4 * np.abs(ref).max()
    assert (poses[:, :3] == 0).all()
    # one camera for all frames == the per-frame entry point with that camera repeated
    p1, v1 = dec.decode(hm)
    p2, v2 = dec.decode_cams(hm, np.tile(g["base_K"], (5, 1, 1)), np.tile(g["base_R"].reshape(3, 3), (5, 1, 1)))
    assert torch.equal(p1, p2) and torch.equal(v1, v2)


def test_metrabs_heads_gemm_feeds_the_decoder(golden_dir):
    """Linear(1280 -> 288) over the (8,8,1280) feature map (4_create_heads_onnx.py:7-16) on tensor cores, fp16 operands like the
    reference's TensorRT-fp16 engine: logits within 2e-3 of the fp32 product, decoded poses within 1e-3 of the pose scale."""
    from isbfsar_b200 import HeatmapDecoder
    from isbfsar_b200.decode import MetrabsHeads
    from oracle import decode_oracle as D
    d64 = np.load(os.path.join(golden_dir, "decode_64.npz"))
    rng = np.random.default_rng(11)
    B = 70                                                       # 4480 rows: ragged last 128-row tile
    target = make_heatmaps(B, seed=6).reshape(B * 64, 288)
    # features whose exact heads output is a heatmap with planted peaks: feats = target @ pinv(W) (+ null-space noise)
    W = (rng.standard_normal((288, 1280)) / np.sqrt(1280)).astype(np.float32)
    b = (0.1 * rng.standard_normal(288)).astype(np.float32)
    feats = ((target - b) @ np.linalg.pinv(W).T).astype(np.float32).reshape(B, 8, 8, 1280)
    m, _ = make_model(Cfg(), 0)
    heads = MetrabsHeads(m, W, b)
    logits = heads(torch.from_numpy(feats).cuda())
    ref = D.heads_forward(feats.astype(np.float64), W.astype(np.float64), b.astype(np.float64))
    assert logits.shape == (B, 8, 8, 288)
    assert np.abs(logits.cpu().numpy() - ref).max() < 2e-3 * np.abs(ref).max()
    dec = HeatmapDecoder(m, d64["expand30"], None, d64["new_K"], d64["homo_inv"])
    poses, valid = dec.decode(logits)
    rp, rv = D.decode_frames(ref.astype(np.float32), d64["expand30"], np.arange(30), d64["new_K"], d64["homo_inv"])
    assert np.array_equal(valid.cpu().numpy(), rv) and rv.all()
    assert np.abs(poses.cpu().numpy() - rp).max() < 1e-3 * np.abs(rp).max()


def test_fp16_host_rows_are_bit_identical():
    """arx_score_host*_f16: fp16 host rows (half the PCIe bytes) give the same bits as fp32 rows holding the same values, on the
    T=16 pair pipeline and on the tiled kernels; shapes on the fp32 kernels refuse loudly."""
    for cfg, B, path in [(Cfg(), 600, 2), (Cfg(way=20, seq_len=32, temp_set=[2, 3]), 40, 3)]:
        m, sd = make_model(cfg, 0)
        support, labels, query, _ = make_episode(cfg, B, 141, "structured")
        q16 = torch.from_numpy(query).to(torch.float16)
        q32 = q16.to(torch.float32)                               # the same values, representable in fp16
        m.set_support(poses=torch.from_numpy(support[0]).cuda())
        a = m.score_host(q32.pin_memory())
        b = m.score_host(q16.pin_memory())
        c = m.score_host_async(q16.pin_memory()).result()
        assert m.last_path() == path
        assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1]) and torch.equal(a[0], c[0]) and torch.equal(a[1], c[1])
        lo, it = TrxOracle(cfg, sd).score(support, labels, query[:32], chunk=16)
        assert rel_err(b[0][:32], lo).max() < TOL_TC and rel_err(b[1][:32], it).max() < TOL_TC
    m, _ = make_model(Cfg(), 0, force_path=1)
    m.set_support(poses=torch.from_numpy(support[0][:5, :16]).cuda())
    with pytest.raises(ValueError):
        m.score_host(torch.zeros((4, 16, 90), dtype=torch.float16).pin_memory())


@pytest.mark.parametrize("cfg,n_frames,path,force", [(Cfg(), 700, 2, 0), (Cfg(), 16, 2, 0), (Cfg(way=3, seq_len=8), 150, 3, 0),
                                                     (Cfg(way=20, seq_len=32, temp_set=[2, 3]), 60, 3, 0), (Cfg(), 40, 1, 1)])
def test_frame_stream_scoring_equals_explicit_windows(cfg, n_frames, path, force):
    """arx_score_frames: every frame embedded / projected once, windows formed on the device -- against the same windows
    given explicitly to arx_score and against the oracle."""
    T = cfg.seq_len
    m, sd = make_model(cfg, 0, force_path=force)
    rng = np.random.default_rng(7 + n_frames)
    support = (0.17 * rng.standard_normal((cfg.way, T, 90))).astype(np.float32)
    frames = (0.17 * rng.standard_normal((n_frames, 90))).astype(np.float32)
    o = min(5, n_frames - T)
    frames[o:o + T] = support[1] + 0.05 * rng.standard_normal((T, 90)).astype(np.float32)
    m.set_support(poses=torch.from_numpy(support).cuda())
    F = torch.from_numpy(frames).cuda()
    lo_s, it_s = m.score_frames(F)
    assert m.last_path() == path
    windows = F.unfold(0, T, 1).permute(0, 2, 1).contiguous()
    assert lo_s.shape == (n_frames - T + 1, cfg.way)
    lo_w, it_w = m.score(windows)
    tol = tol_for(m)
    assert rel_err(lo_s.cpu(), lo_w.cpu()).max() < tol and rel_err(it_s.cpu(), it_w.cpu()).max() < tol
    if path == 1:       # k_linear adds the positional table after the accumulation, like k_form_windows: the same bits
        assert torch.equal(lo_s, lo_w) and torch.equal(it_s, it_w)
    k = min(48, windows.shape[0])
    lo, it = TrxOracle(cfg, sd).score(support[None], np.arange(cfg.way)[None], windows[:k].cpu().numpy(), chunk=16)
    assert rel_err(lo_s[:k].cpu(), lo).max() < tol and rel_err(it_s[:k].cpu(), it).max() < tol
    assert np.array_equal(lo_s[:k].argmax(1).cpu().numpy(), lo.argmax(1))
    assert int(lo_s[o].argmax()) == 1
    # fewer than seq_len frames: nothing to score
    e_lo, e_it = m.score_frames(F[:T - 1])
    assert e_lo.shape == (0, cfg.way)


@pytest.mark.parametrize("cfg,path,force", [(Cfg(), 1, 1), (Cfg(way=3, seq_len=8), 3, 0), (Cfg(), 2, 0)], ids=["fp32", "tiled", "pair"])
def test_frame_stream_chunks_are_bit_identical(cfg, path, force):
    """arx_score_frames split into passes of 7 windows: every pass starts at its own frame, same bits as one pass."""
    T = cfg.seq_len
    rng = np.random.default_rng(31)
    support = torch.from_numpy((0.17 * rng.standard_normal((cfg.way, T, 90))).astype(np.float32)).cuda()
    frames = torch.from_numpy((0.17 * rng.standard_normal((T + 40, 90))).astype(np.float32)).cuda()
    res = []
    for mc in (0, 7):
        m, _ = make_model(cfg, 0, force_path=force, max_chunk=mc)
        m.set_support(poses=support)
        res.append(m.score_frames(frames))
        assert m.last_path() == path
    assert torch.equal(res[0][0], res[1][0]) and torch.equal(res[0][1], res[1][1])


@pytest.mark.parametrize("cfg,B,max_chunk,path", [(Cfg(), 600, 0, 2), (Cfg(way=20, seq_len=32, temp_set=[2, 3]), 40, 7, 3)],
                         ids=["pair", "tiled_chunked"])
def test_fp16_and_fp32_host_rows_alternate_on_one_handle(cfg, B, max_chunk, path):
    """fp32 and fp16 rows of the same values, alternating on one handle: the first call of each runs eagerly, the second is
    captured, the third replayed (pair pipeline), and a pass never reads the other precision's rows or graph."""
    m, _ = make_model(cfg, 0, max_chunk=max_chunk)
    support, _, query, _ = make_episode(cfg, B, 143, "structured")
    q16 = torch.from_numpy(query).to(torch.float16).pin_memory()
    q32 = q16.to(torch.float32).pin_memory()
    m.set_support(poses=torch.from_numpy(support[0]).cuda())
    ref = m.score_host(q32)
    for _ in range(3):
        for q in (q32, q16):
            for r in (m.score_host(q), m.score_host_async(q).result()):
                assert m.last_path() == path
                assert torch.equal(r[0], ref[0]) and torch.equal(r[1], ref[1])
