"""CPU-only: the episodic evaluation arithmetic (compute_fsos.py:100-133), the reference's frozen scores (and the staged
reference `oracle/_ref`, where present) against the oracle port, and the reference's saved support set through the
oracle's ActionRecognizer restatement."""
import io
import os
import pickle

import numpy as np
import torch

from oracle.synth import Cfg, make_episode, make_state_dict
from oracle.trx_oracle import ActionRecognizerOracle, TrxOracle


def test_fsos_accuracies_by_hand():
    from isbfsar_b200.eval import evaluate_fsos
    # 4 episodes, 3-way: [known+right+accepted, known+wrong+accepted, unknown+rejected, unknown+accepted]
    logits = torch.tensor([[0., -1, -2], [-3., -1, -2], [0., -1, -2], [-5., -1, -9]])
    is_true = torch.tensor([[0.9], [0.8], [0.2], [0.7]])
    batch = {"support_set": {"sk": torch.zeros(4, 3, 16, 90)}, "target_set": {"sk": torch.zeros(4, 16, 90)},
             "support_classes": torch.tensor([[4, 5, 6]] * 4), "target_class": torch.tensor([4, 6, 9, 9]),
             "known": torch.tensor([True, True, False, False])}

    def model(ss, labels, q):
        assert labels.shape == (4, 3) and labels.dtype == torch.int32 and ss["sk"].shape == (4, 3, 16, 90)
        return {"logits": logits, "is_true": is_true}

    r = evaluate_fsos(model, [batch], 3)
    assert r["OS-ACC"] == 0.75 and r["FS-ACC"] == 0.5 and r["FSOS-ACC"] == 0.5 and r["episodes"] == 4 and r["known"] == 2
    assert evaluate_fsos(model, [], 3)["FSOS-ACC"] == -1      # compute_fsos.py:116-132: -1 when nothing was scored


def test_synthetic_episodes_shape_and_oracle_eval():
    from isbfsar_b200.eval import evaluate_fsos, synthetic_fsos_episodes
    cfg = Cfg()
    o = TrxOracle(cfg, make_state_dict(cfg, 0))
    eps = list(synthetic_fsos_episodes(2, batch=6, way=5, seed=1))
    e = eps[0]
    assert e["support_set"]["sk"].shape == (6, 5, 16, 90) and e["target_set"]["sk"].shape == (6, 16, 90)
    assert e["support_classes"].shape == (6, 5) and e["known"].dtype == torch.bool
    inside = (e["support_classes"] == e["target_class"][:, None]).any(1)
    assert torch.equal(inside, e["known"])
    r = evaluate_fsos(lambda s, l, q: o.forward(s, l, q), eps, 5)
    assert r["episodes"] == 12 and r["FS-ACC"] == 1.0


def test_staged_reference_matches_port(golden_dir):
    """The staged reference (oracle/_ref, oracle/build_ref.py: the CPU arm of bench.py) and the oracle port agree on cfg1,
    both held to the scores frozen from the unmodified reference in tests/golden/cfg1_w5_t16_structured.npz
    (oracle/gen_golden.py).  The port half overlaps test_oracle_golden.py::test_trx_oracle_matches_reference on that
    file; the staged half runs wherever oracle/_ref is staged, which a plain checkout does not have."""
    from oracle import ref_runner
    g = np.load(os.path.join(golden_dir, "cfg1_w5_t16_structured.npz"))
    way, T, B, wseed, iseed, affine = [int(x) for x in g["meta"][:6]]
    cfg = Cfg()
    assert (way, T, affine, str(g["kind"])) == (cfg.way, cfg.seq_len, 0, "structured")
    sd = make_state_dict(cfg, wseed)
    support, labels, query, _ = make_episode(cfg, B, iseed, "structured")
    lo, it = g["logits"], g["is_true"]
    lo2, it2 = TrxOracle(cfg, sd).score(support, labels, query)
    assert np.abs(lo / lo2 - 1).max() < 2e-5 and np.abs(it / it2 - 1).max() < 2e-5
    if ref_runner.available():
        lo3, it3 = ref_runner.ReferenceScorer(cfg, sd).score(support, labels, query)
        assert np.abs(lo3 / lo - 1).max() < 2e-5 and np.abs(it3 / it - 1).max() < 2e-5


class _CpuUnpickler(pickle.Unpickler):
    """The fixture holds CUDA tensors (main.py:321-326 pickles them as they are): map the storages to the CPU."""

    def find_class(self, module, name):
        if module == "torch.storage" and name == "_load_from_bytes":
            return lambda b: torch.load(io.BytesIO(b), map_location="cpu", weights_only=False)
        return super().find_class(module, name)


def test_reference_support_set_fixture_through_oracle(golden_dir):
    with open(os.path.join(golden_dir, "ref_support_set.pkl"), "rb") as f:
        ss = _CpuUnpickler(f).load()
    assert list(ss) == ["hello", "get", "lift"]
    for v in ss.values():
        assert v["poses"].shape == (16, 90) and v["features"].shape == (16, 256)
        assert float(v["poses"][:, :3].abs().max()) == 0.0          # root-centred skeletons (main.py:103)
    cfg = Cfg()
    oa = ActionRecognizerOracle(cfg, make_state_dict(cfg, 0))
    oa.support_set = ss
    oa.requires_focus = pickle.load(open(os.path.join(golden_dir, "ref_requires_focus.pkl"), "rb"))
    for v in ss.values():
        v.pop("features")                                           # features of the TRAINED weights: not ours
    for f in ss["lift"]["poses"].numpy():
        res, os_, rf = oa.inference({"sk": f})
    assert max(res, key=res.get) == "lift" and rf == {"hello": True, "get": True, "lift": False}


def test_tta_helpers_match_reference_golden(golden_dir):
    """get_augmentations / tta_cameras (misc.py:310-327, hpe.py:88-93): product host code and oracle against arrays frozen from
    the reference's own functions."""
    from isbfsar_b200 import decode as P
    from oracle import decode_oracle as D
    g = np.load(os.path.join(golden_dir, "tta_5.npz"))
    for mod in (P, D):
        flip, rotflip, gammas, scales = mod.get_augmentations(5)
        assert np.array_equal(flip, g["flip"]) and np.array_equal(rotflip, g["rotflip"])
        assert np.array_equal(gammas, g["gammas"]) and np.array_equal(scales, g["scales"])
        K, R, f2 = mod.tta_cameras(g["base_K"], g["base_R"], 5)
        assert np.array_equal(K, g["new_K"]) and np.array_equal(R, g["homo_inv"]) and np.array_equal(f2, g["flip"])
    from oracle.synth import make_heatmaps
    d64 = np.load(os.path.join(golden_dir, "decode_64.npz"))
    poses, valid = D.decode_frames_cams(make_heatmaps(5, seed=4), d64["expand30"], np.arange(30), g["new_K"], g["homo_inv"])
    assert valid.all() and np.allclose(poses, g["poses"], rtol=1e-12, atol=1e-13)
