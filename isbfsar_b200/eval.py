"""Episodic few-shot open-set evaluation driver (reference: modules/ar/utils/test/compute_fsos.py:74-143).

The reference script walks an NTU-RGB+D-derived dataset with `FSOSEpisodicLoader` (dataloader.py:131-205) and, for
every batch of episodes, calls `model(support_set, support_labels, target_set)` and accumulates three accuracies:

  OS-ACC    `(is_true > 0.5) == known`                                        (compute_fsos.py:100-102)
  FS-ACC    `argmax(logits) == target` over the KNOWN episodes only           (compute_fsos.py:104-108)
  FSOS-ACC  known: class right AND accepted; unknown: rejected                (compute_fsos.py:110-114)

This module reproduces that arithmetic over any iterable of episode batches in the loader's dict format
(`support_set`/`target_set` dicts keyed "sk", `support_classes`, `target_class`, `known`); the dataset I/O itself is out
of scope (SURVEY.md section 2 row 8), so `synthetic_fsos_episodes` provides loader-shaped synthetic episodes.  The
model argument is anything with the reference `forward(ss_data, ss_labels, query_data)` signature: the CUDA `TRXOS`
of this package scores every batch through `arx_score_episodes`, in batched-episode passes on both tensor-core routes
(T=16 pairs: 256 episodes per pass; the tiled kernels, e.g. the T=32 cfg4 shape: as many episodes as keep the support
pool within 1 GiB) and one episode at a time on the fp32 route.
"""
from __future__ import annotations

import numpy as np
import torch


def synthetic_fsos_episodes(n_batches: int, batch: int = 28, way: int = 5, seq_len: int = 16, n_joints: int = 30,
                            n_classes: int = 17, p_known: float = 0.6, noise: float = 0.05, seed: int = 0):
    """Loader-shaped episode batches (dataloader.py:189-199 after default collation).  Every class has one exemplar
    sequence `0.17*N(0,1)` (sigma of the reference's saved support set); an episode draws `way` support classes, and a
    target that is a noisy copy of the exemplar of either one of them (known) or of another class (unknown)."""
    rng = np.random.default_rng(seed)
    exemplars = (0.17 * rng.standard_normal((n_classes, seq_len, n_joints * 3))).astype(np.float32)
    for _ in range(n_batches):
        sup_cls = np.stack([rng.permutation(n_classes)[:way] for _ in range(batch)])            # (b,W)
        known = rng.random(batch) < p_known
        tgt = np.empty(batch, dtype=np.int64)
        for i in range(batch):
            if known[i]:
                tgt[i] = sup_cls[i, rng.integers(0, way)]
            else:
                others = np.setdiff1d(np.arange(n_classes), sup_cls[i])
                tgt[i] = others[rng.integers(0, len(others))]
        target = exemplars[tgt] + (noise * rng.standard_normal((batch, seq_len, n_joints * 3))).astype(np.float32)
        yield {"support_set": {"sk": torch.from_numpy(exemplars[sup_cls])},                     # (b,W,T,3J)
               "target_set": {"sk": torch.from_numpy(target)},                                  # (b,T,3J)
               "support_classes": torch.from_numpy(sup_cls),
               "target_class": torch.from_numpy(tgt),
               "known": torch.from_numpy(known)}


@torch.no_grad()
def evaluate_fsos(model, loader, way: int, device=None) -> dict:
    """compute_fsos.py:84-133 for one repetition.  Returns {'FSOS-ACC','FS-ACC','OS-ACC','episodes','known'}
    (-1 for an accuracy with no samples, like the reference)."""
    fs_score, os_score, fsos_score = [], [], []
    n_known = 0
    for elem in loader:
        support_set = {t: elem["support_set"][t].float() for t in elem["support_set"].keys()}
        target_set = {t: elem["target_set"][t].float() for t in elem["target_set"].keys()}
        if device is not None:
            support_set = {t: v.to(device) for t, v in support_set.items()}
            target_set = {t: v.to(device) for t, v in target_set.items()}
        b = target_set["sk"].shape[0]
        support_labels = torch.arange(way).repeat(b).reshape(b, way).int()                       # compute_fsos.py:93
        if device is not None:
            support_labels = support_labels.to(device)
        known = elem["known"].bool()
        target = torch.argmax((elem["support_classes"] == elem["target_class"][..., None]).int(), dim=1)

        out = model(support_set, support_labels, target_set)
        fs_pred = out["logits"].detach().cpu()
        os_pred = out["is_true"].detach().cpu()

        true_os = (os_pred > 0.5) == known.unsqueeze(-1)                                          # compute_fsos.py:101
        os_score.append(true_os.numpy())
        fs_pred = torch.argmax(fs_pred, dim=1)
        true_fs = fs_pred == target                                                               # meaningless for unknown targets
        fs_score.append(true_fs[known].numpy())
        kn = torch.logical_and(known, true_fs)
        kn = torch.logical_and(kn.unsqueeze(-1), true_os)
        ukn = torch.logical_and(~known.unsqueeze(-1), true_os)
        fsos_score.append(torch.logical_or(kn, ukn).numpy())
        n_known += int(known.sum())

    def acc(parts):
        if len(parts) == 0:
            return -1
        flat = np.concatenate(parts, axis=0).reshape(-1)
        return float(flat.sum() / flat.size) if flat.size else -1

    n = int(sum(p.shape[0] for p in os_score))
    return {"FSOS-ACC": acc(fsos_score), "FS-ACC": acc(fs_score), "OS-ACC": acc(os_score), "episodes": n, "known": n_known}


def compute_fsos(model, way: int = 5, repetitions: int = 10, n_batches: int = 8, batch: int = 28, seed: int = 0, device=None,
                 **episode_kw) -> dict:
    """The outer loops of compute_fsos.py:62-143: `repetitions` evaluations with freshly drawn support classes; returns the
    reference's results layout {'FSOS-ACC': [...], 'FS-ACC': [...], 'OS-ACC': [...]} (one entry per repetition)."""
    results = {"FSOS-ACC": [], "FS-ACC": [], "OS-ACC": []}
    for r in range(repetitions):
        res = evaluate_fsos(model, synthetic_fsos_episodes(n_batches, batch, way, seed=seed + r, **episode_kw), way, device)
        for k in results:
            results[k].append(res[k])
    return results
