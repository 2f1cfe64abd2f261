"""Independent restatements of exact flat search and of eval.py's sequence-level hit rates (test infrastructure).

``flat_search`` is fp64 brute force; ``sequence_hit_rates`` is a literal per-id, per-length loop over numpy arrays,
deliberately not vectorised, so that it stays a second reading of the rules ``grafp_b200.search.evaluate_sequences``
implements in batched form.
"""
from __future__ import annotations

import numpy as np
import torch

RATES = ("top1_exact", "top1_near", "top3_exact", "top10_exact")


def flat_search(R, Q, k: int, chunk: int = 64):
    """(D, I) of the k nearest rows of R for every row of Q in fp64 squared L2 distance, ascending by (distance, id).

    R, Q: torch tensors (on any one device) or numpy arrays; the result is on R's device (numpy in, torch CPU out)."""
    R = torch.as_tensor(R).double()
    Q = torch.as_tensor(Q).to(R.device).double()
    r2 = (R * R).sum(1)
    Ds, Is = [], []
    for i in range(0, Q.shape[0], chunk):
        q = Q[i:i + chunk]
        d = (q * q).sum(1, keepdim=True) - 2.0 * (q @ R.T) + r2[None]
        vals, idx = torch.sort(d, dim=1, stable=True)   # stable: equal distances keep the lower id
        Ds.append(vals[:, :k])
        Is.append(idx[:, :k])
    return torch.cat(Ds), torch.cat(Is)


def sequence_hit_rates(R: np.ndarray, query: np.ndarray, test_ids, seq_lens, k_probe: int, gt_offset: int = 0,
                       probe_ids: np.ndarray = None, probe_dist: np.ndarray = None) -> dict:
    """eval.py's sequence loop, literally.  ``probe_ids`` / ``probe_dist``: the exact (fp64) top-(k_probe + 1) of every
    query row (computed here with ``flat_search`` when absent); the extra column measures the k_probe boundary gap.

    Returns the four rates (percent per length), the hit flags (n_ids, n_lens), and per (id, length) the smallest
    score gap at a rank boundary the flags depend on (1|2, 3|4, 10|11) and the smallest distance gap at the k_probe
    boundary over the sequence's rows - both in fp64 - so that a caller can tell near-ties from disagreements."""
    R = np.asarray(R, dtype=np.float64)
    query = np.asarray(query, dtype=np.float64)
    if probe_ids is None:
        D, I = flat_search(R, query, k_probe + 1)
        probe_ids, probe_dist = I.numpy(), D.numpy()
    n = R.shape[0]
    ids = np.asarray(test_ids, dtype=np.int64)
    flags = {name: np.zeros((len(ids), len(seq_lens)), dtype=bool) for name in RATES}
    score_gap = np.full((len(ids), len(seq_lens)), np.inf)
    probe_gap = np.full((len(ids), len(seq_lens)), np.inf)
    for a, t in enumerate(ids):
        for b, L in enumerate(seq_lens):
            q = query[t:t + L]
            I = probe_ids[t:t + L, :k_probe].copy()
            for o in range(len(I)):
                I[o, :] -= o
            candidates = np.unique(I[I >= 0])
            scores = np.zeros(len(candidates))
            for ci, c in enumerate(candidates):
                match = R[c:c + L]
                m = min(len(q), len(match))
                scores[ci] = np.mean([np.dot(q[o], match[o]) for o in range(m)])
            order = sorted(range(len(candidates)), key=lambda i: (-scores[i], candidates[i]))
            pred = [int(candidates[i]) for i in order][:10]
            s = [scores[i] for i in order]
            gt = int(t) + gt_offset
            flags["top1_exact"][a, b] = pred[0] == gt
            flags["top1_near"][a, b] = abs(pred[0] - gt) <= 1
            flags["top3_exact"][a, b] = gt in pred[:3]
            flags["top10_exact"][a, b] = gt in pred[:10]
            for r in (0, 2, 9):
                if r + 1 < len(s):
                    score_gap[a, b] = min(score_gap[a, b], s[r] - s[r + 1])
            if probe_dist is not None and probe_dist.shape[1] > k_probe and n > k_probe:
                for o in range(len(q)):
                    probe_gap[a, b] = min(probe_gap[a, b], probe_dist[t + o, k_probe] - probe_dist[t + o, k_probe - 1])
    out = {name: 100.0 * flags[name].mean(0) for name in RATES}
    out.update(hits=flags, score_gap=score_gap, probe_gap=probe_gap)
    return out
