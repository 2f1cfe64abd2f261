"""Exact flat search (grafp_b200.search.FingerprintIndex, the key-sliced K1 kernel + merge) against fp64 brute force,
and evaluate_sequences against the literal eval.py loop of oracle/search_oracle.py."""
import math

import numpy as np
import pytest
import torch

import golden_io as gio
from golden_io import _default_kernel_options, _exact_fp32_library_math  # noqa: F401  (autouse: TF32 off, default options)
from grafp_b200 import search as S
from grafp_b200 import synth
from grafp_b200.search import FingerprintIndex, evaluate_sequences, load_index
from oracle.search_oracle import RATES, flat_search, sequence_hit_rates

pytestmark = pytest.mark.gpu

DEV = torch.device("cuda", 0)


def _sms():
    return torch.cuda.get_device_properties(DEV).multi_processor_count


def _unit(n, d, seed, device=DEV):
    g = torch.Generator(device=device).manual_seed(seed)
    return torch.nn.functional.normalize(torch.randn(n, d, generator=g, device=device), dim=1)


# --- mirror of the host planner: plan_with() and search_plan() in grafp_b200/csrc/knn_tc2.cu ---------------------------
_BM, _BUDGET, _BLOCK = 128, 232448 - (2 * 128 * 4 + 64 + (2 * 8 + 8) * 8 + 1024), 32768


def _plan_with(N, C, qs):
    num_kc = (C + 63) // 64
    def queue(nh):
        return 4 * nh * (qs * 512 if qs > 0 else (3 * 1024 if qs < 0 else 0))
    if N >= 4 * _BM and 4 * num_kc * _BLOCK + queue(4) + 3 * (_BLOCK // 2) <= _BUDGET:
        return 4, 64
    for nh in ((2, 1) if N > _BM else (1,)):
        resident = nh * num_kc * _BLOCK + queue(nh)
        if qs > 0 and resident + 2 * (_BLOCK // 2) <= _BUDGET and resident + 3 * _BLOCK > _BUDGET:
            return nh, 64
        if resident + 2 * _BLOCK > _BUDGET:
            continue
        return nh, 128
    raise AssertionError("no plan")


def search_slices(n_q, n_db, d, k, sms):
    """(key tile, slice length, slice count) that grafp_search_fwd uses."""
    nh, bn = _plan_with(n_q, d, -1 if k <= 3 else 6)
    qblocks = -(-n_q // (_BM * nh))
    want = -(-2 * sms // qblocks)
    length = -(-n_db // want)
    length = min(max(-(-length // bn) * bn, 2 * bn), 1 << 26)
    return bn, length, -(-n_db // length)


def group_maxima_slices(index, n_q, k):
    """Per slice: whether the kernel ranks it with the group maxima (k <= 3 and |y|^2 within 1e-4 of 1, spread <= 1e-6)."""
    _, length, count = search_slices(n_q, index.ntotal, index.d, k, _sms())
    sq = index._sq[:index.ntotal]
    out = []
    for s in range(count):
        v = sq[s * length:(s + 1) * length]
        mn, mx = float(v.min()), float(v.max())
        out.append(k <= 3 and mn >= 1 - 1e-4 and mx <= 1 + 1e-4 and mx - mn <= 1e-6)
    return out


def check_exact(R, Q, D, I, k, what):
    """Zero hard mismatches against fp64, ascending lists, distances within the fp32 band; returns the tie count."""
    d = R.shape[1]
    band = 4 * math.sqrt(d) * 2.0 ** -23
    Dref, Iref = flat_search(R, Q, k)
    assert D.shape == I.shape == (Q.shape[0], k) and I.dtype == torch.int64 and D.dtype == torch.float32
    assert bool((I >= 0).all()) and bool((I < R.shape[0]).all()), what
    ours64 = ((Q.double()[:, None, :] - R.double()[I]) ** 2).sum(-1)
    differ = I != Iref
    gap = (ours64 - Dref).abs()
    hard = int((differ & (gap > band)).sum())
    assert hard == 0, f"{what}: {hard} hard mismatches (max gap {float(gap[differ].max()):.3e}, band {band:.3e})"
    assert bool((D[:, 1:] >= D[:, :-1]).all()), f"{what}: lists not ascending"
    err = float((D.double() - ours64).abs().max())
    assert err <= band, f"{what}: distance error {err:.3e} > band {band:.3e}"
    assert all(len(set(row)) == k for row in I.tolist()[:64]), f"{what}: repeated ids"
    return int(differ.sum())


CASES = [  # n_db, n_q, k, d
    (3, 7, 3, 64), (17, 1, 17, 256), (128, 7, 128, 128), (127, 129, 8, 128), (128, 1, 1, 256), (129, 1000, 17, 64),
    (4097, 129, 20, 128), (4097, 7, 128, 256), (4097, 1000, 64, 64), (4097, 1, 16, 128),
    (1_000_003, 1000, 20, 128), (1_000_003, 1, 3, 128), (1_000_003, 129, 16, 64), (1_000_003, 7, 128, 256),
]


@pytest.mark.parametrize("n_db,n_q,k,d", CASES)
def test_search_is_exact_against_fp64(n_db, n_q, k, d):
    R = _unit(n_db, d, n_db + d)
    Q = _unit(n_q, d, 7 * n_q + k)
    index = FingerprintIndex(d, DEV)
    index.add(R)
    D, I = index.search(Q, k)
    ties = check_exact(R, Q, D, I, k, f"n_db={n_db} n_q={n_q} k={k} d={d}")
    gm = group_maxima_slices(index, n_q, k)
    print(f"search n_db={n_db} n_q={n_q} k={k} d={d}: slices {len(gm)} (group maxima on {sum(gm)}), tie-order "
          f"differences {ties} of {n_q * k}")


def test_exact_ties_and_both_selection_paths():
    d, n = 128, 4096
    base = _unit(n, d, 11)
    # duplicated rows: rows 100, 1100, 2100, 3100 are one vector; the lower ids come first, bit-exactly
    R = base.clone()
    R[[1100, 2100, 3100]] = R[100].clone()
    index = FingerprintIndex(d, DEV)
    index.add(R)
    q = torch.cat([R[100:101], R[7:8]])
    for k in (1, 3, 4, 20):
        D, I = index.search(q, k)
        want = [100, 1100, 2100, 3100][:k]
        assert I[0, :len(want)].tolist() == want, (k, I[0].tolist())
        assert len(set(D[0, :len(want)].tolist())) == 1
        assert I[1, 0].item() == 7, "a query equal to a database row finds that row first"
    assert all(group_maxima_slices(index, 2, 1)), "unit rows at k <= 3 take the group maxima"
    # zero rows and rows of norm < 1: the vote-gated scan (k <= 3) and the queues, same exactness
    R2 = base.clone()
    R2[::5] *= 0.5
    R2[3::7] = 0.0
    index2 = FingerprintIndex(d, DEV)
    index2.add(R2)
    Q = torch.cat([_unit(60, d, 12), R2[3:4], R2[5:6]])
    assert not any(group_maxima_slices(index2, Q.shape[0], 1)), "non-unit rows must not take the group maxima"
    for k in (1, 3, 8, 20):
        D, I = index2.search(Q, k)
        check_exact(R2, Q, D, I, k, f"non-unit rows k={k}")
    D, I = index2.search(R2[3:4], 3)
    assert I[0].tolist() == [3, 10, 17] and float(D[0, 0]) == 0.0, "zero query: distance 0 to the zero rows, lowest ids first"
    # unit rows with a ragged last slice (n_db % 32 != 0): group maxima on every slice, exact
    R3 = _unit(50_001, d, 13)
    index3 = FingerprintIndex(d, DEV)
    index3.add(R3)
    Q3 = _unit(129, d, 14)
    assert all(group_maxima_slices(index3, 129, 3))
    for k in (1, 3):
        D, I = index3.search(Q3, k)
        check_exact(R3, Q3, D, I, k, f"ragged group maxima k={k}")


def test_results_do_not_depend_on_the_batch_or_the_slicing():
    d, n_db = 128, 200_000
    index = FingerprintIndex(d, DEV)
    index.add(_unit(n_db, d, 21))
    big = _unit(80_000, d, 22)
    sms = _sms()
    for k in (1, 5, 20, 128):
        plans = {n: search_slices(n, n_db, d, k, sms) for n in (1, 1000, 80_000)}
        counts = [p[2] for p in plans.values()]
        assert counts[0] > counts[1] > 1 == counts[2], (k, plans, "the shapes must cover many slices, fewer, and one")
        assert all(p[1] >= 2 * p[0] for p in plans.values()), (k, plans, "at least two key tiles per slice")
        D_big, I_big = index.search(big, k)
        D_mid, I_mid = index.search(big[:1000], k)
        for j in (0, 17, 999):
            D1, I1 = index.search(big[j:j + 1], k)
            assert torch.equal(I1[0], I_mid[j]) and torch.equal(D1[0], D_mid[j]), (k, j)
            assert torch.equal(I1[0], I_big[j]) and torch.equal(D1[0], D_big[j]), (k, j)
        assert torch.equal(I_mid, I_big[:1000]) and torch.equal(D_mid, D_big[:1000]), k
        print(f"invariance k={k}: alone == batch of 1000 == batch of 80000 (slices {counts})")


def test_ids_beyond_2_pow_24_come_back_exactly():
    d, n_db, n_q = 64, (1 << 24) + 4096, 64
    R = _unit(n_db, d, 31)
    Q = _unit(n_q, d, 32)
    first = (1 << 24) + 1 + 2 * torch.arange(n_q, device=DEV)         # odd ids: not representable in fp32
    second = first + 1 + 2 * n_q
    R[first] = Q
    R[second] = torch.nn.functional.normalize(Q + 0.05 * _unit(n_q, d, 33), dim=1)
    index = FingerprintIndex(d, DEV)
    index.add(R)
    del R
    for k in (1, 3, 20):
        _, I = index.search(Q, k)
        assert torch.equal(I[:, 0], first), k
        if k > 1:
            assert torch.equal(I[:, 1], second), k


def test_errors_raise_before_anything_launches():
    d = 64
    for bad_d in (48, 60, 512):
        with pytest.raises(ValueError):
            FingerprintIndex(bad_d, DEV)
    with pytest.raises(RuntimeError):
        FingerprintIndex(d, "cpu")
    index = FingerprintIndex(d, DEV)
    R = _unit(300, d, 41)
    index.add(R)
    over = R[:5].clone()
    over[2] *= 1.001
    with pytest.raises(ValueError):
        index.add(over)
    assert index.ntotal == 300
    with pytest.raises(ValueError):
        index.search(over, 1)
    with pytest.raises(ValueError):
        index.search(R[:2], 301)
    with pytest.raises(ValueError):
        index.search(R[:2], 0)
    with pytest.raises(RuntimeError):
        index.search(R[:2].cpu(), 1)
    nan = R[:1].clone()
    nan[0, 0] = float("nan")
    with pytest.raises(ValueError):
        index.add(nan)
    assert index.ntotal == 300


def test_load_index_from_writer_files_equals_one_add(tmp_path, monkeypatch):
    from grafp_b200.inference import FingerprintWriter
    monkeypatch.setattr(S, "_STAGING_ROWS", 1000)          # several staging chunks per file
    d = 128
    dummy, db = _unit(3001, d, 51), _unit(4999, d, 52)
    for name, rows, cuts in (("dummy_db", dummy, (0, 700, 701, 3001)), ("db", db, (0, 1234, 4000, 4999))):
        with FingerprintWriter(str(tmp_path), name, rows.shape[0], d) as w:
            for a, b in zip(cuts[:-1], cuts[1:]):
                w.append(rows[a:b])
    loaded = load_index([(str(tmp_path), "dummy_db"), (str(tmp_path), "db")], DEV)
    direct = FingerprintIndex(d, DEV)
    direct.add(torch.cat([dummy, db]))
    assert loaded.ntotal == direct.ntotal == 8000
    assert torch.equal(loaded.rows, direct.rows)
    assert torch.equal(loaded._hi[:8000], direct._hi[:8000]) and torch.equal(loaded._sq[:8000], direct._sq[:8000])
    q = _unit(33, d, 53)
    for k in (1, 20):
        a, b = loaded.search(q, k), direct.search(q, k)
        assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])
    # numpy input and CPU tensors take the same staging path
    host = FingerprintIndex(d, DEV)
    host.add(dummy.cpu().numpy())
    host.add(db.cpu())
    assert torch.equal(host.rows, direct.rows)


def track_fixture(d=128, n_dummy=2000, n_track=3000, n_query=1000, step=0.15, noise=2.0, seed=5):
    """Dummy rows (independent unit vectors), then a track: a normalised random walk, so that neighbouring rows are
    similar and the +-1 "near" hit means something.  Queries: track rows 0 .. n_query - 1 plus noise (gt_offset =
    n_dummy).  Built on the CPU from a seed."""
    g = torch.Generator().manual_seed(seed)
    dummy = torch.nn.functional.normalize(torch.randn(n_dummy, d, generator=g), dim=1)
    x = torch.nn.functional.normalize(torch.randn(d, generator=g), dim=0)
    track = []
    for _ in range(n_track):
        track.append(x)
        x = torch.nn.functional.normalize(x + step * torch.randn(d, generator=g) / math.sqrt(d), dim=0)
    track = torch.stack(track)
    query = torch.nn.functional.normalize(track[:n_query] + noise * torch.randn(n_query, d, generator=g) / math.sqrt(d), dim=1)
    return torch.cat([dummy, track]), query, n_dummy


def test_evaluate_sequences_matches_the_oracle_loop():
    R, query, gt_offset = track_fixture()
    seq_lens, k_probe = (1, 3, 5, 9, 11, 19), 20
    ids = np.sort(np.random.default_rng(6).choice(len(query) - max(seq_lens), 150, replace=False))
    index = FingerprintIndex(R.shape[1], DEV)
    index.add(R)
    got = evaluate_sequences(index, query.to(DEV), ids, seq_lens, k_probe, gt_offset, chunk=64)
    D, I = flat_search(R.to(DEV), query.to(DEV), k_probe + 1)
    want = sequence_hit_rates(R.numpy(), query.numpy(), ids, seq_lens, k_probe, gt_offset, I.cpu().numpy(), D.cpu().numpy())
    noise = 1e-5   # fp32 scores of <= 19 products of unit rows: far below this
    near_tie = (want["score_gap"] < noise) | (want["probe_gap"] < 4 * math.sqrt(R.shape[1]) * 2.0 ** -23)
    disagree = {name: got["hits"][name] != want["hits"][name] for name in RATES}
    n_dis = sum(int(v.sum()) for v in disagree.values())
    print(f"evaluate_sequences: {len(ids)} ids x {len(seq_lens)} lengths, near-ties {int(near_tie.sum())}, "
          f"flag disagreements {n_dis} (all at near-ties)")
    for name in RATES:
        print(f"  {name}: ours {np.round(got[name], 2).tolist()} oracle {np.round(want[name], 2).tolist()}")
        assert not (disagree[name] & ~near_tie).any(), name
        np.testing.assert_array_equal(got[name], want[name], err_msg=name)
    # every length and every rate is exercised: not all hit, not all missed, and the 1-segment top-1 rate rises
    assert 0 < want["top1_exact"][0] < 90 and want["top1_exact"][-1] > want["top1_exact"][0]
    for name in RATES:
        assert (want[name] > 0).all(), name
    assert (want["top1_near"] > want["top1_exact"]).any()
    # "all" resolves and runs through the same path
    every = evaluate_sequences(index, query.to(DEV), "all", (1, 3), k_probe, gt_offset)
    assert len(every["test_ids"]) == len(query) - 3 and every["hits"]["top1_exact"].shape == (len(query) - 3, 2)


def test_real_fingerprints_top1_matches_the_golden_reference():
    """configs[4] at size (the setup of test_fingerprint_generation_at_size_matches_the_reference_on_the_same_gpu):
    index.search(q, 1) gives the reference's top-1 ids up to its recorded near-ties (margin < 0.02)."""
    from grafp_b200.encoder.graph_encoder import GraphEncoder
    from grafp_b200.inference import generate_fingerprints
    from grafp_b200.simclr.simclr import SimCLR
    gold = gio.load("fingerprints")
    cfg = dict(synth.DEFAULT_CFG)
    n_db, n_q = 10_000, 1_000
    torch.manual_seed(0)
    model = SimCLR(cfg, GraphEncoder(cfg=cfg, in_channels=cfg["n_filters"], k=3))
    sd = model.state_dict()
    keep = {k: v for k, v in sd.items() if k.endswith("relative_pos")}
    model.load_state_dict(synth.synth_state_dict({k: v.shape for k, v in sd.items()}, 303, keep))
    db_specs, _ = synth.synth_spec(n_db, 7)
    sd = model.state_dict()
    for key in gold:
        if key.startswith("buf."):
            sd[key[4:]] = gio.t(gold[key])
    model.load_state_dict(sd)
    model.to(DEV).eval()
    pick = torch.randperm(n_db, generator=torch.Generator().manual_seed(8))[:n_q]
    q_specs = db_specs[pick] + 0.02 * torch.randn(n_q, 64, 32, generator=torch.Generator().manual_seed(9))

    def fingerprints(specs):
        with torch.no_grad():
            h = generate_fingerprints(model.encoder, model.peak_extractor(specs.to(DEV)), chunk=128)
            return torch.nn.functional.normalize(model.projector(h), p=2)

    db, q = fingerprints(db_specs), fingerprints(q_specs)
    index = FingerprintIndex(db.shape[1], DEV)
    index.add(db)
    _, I = index.search(q, 1)
    top1, top1_ref, margin = I[:, 0].cpu(), gio.t(gold["top1"]).long(), gio.t(gold["margin"])
    differs = top1 != top1_ref
    print(f"real fingerprints: top-1 differing from the reference {int(differs.sum())} / {n_q}")
    assert int(differs.sum()) <= n_q // 200 and bool((margin[differs] < 0.02).all())
