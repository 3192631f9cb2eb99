"""CPU: the oracle against the reference's own code on seeded random inputs.  The reference's results on these
inputs are stored in tests/golden/oracle_ref_cases.npz (tests/golden/make_golden.py)."""
import numpy as np
import pytest

from conftest import reference_knn, sha256_of
from oracle import cpu_oracle as O


@pytest.mark.parametrize("seed,S,Q,K", [(0, 500, 300, 16), (1, 2000, 100, 1), (2, 64, 64, 32),
                                        (3, 5, 9, 8), (4, 3000, 700, 4)])
def test_knn_random(oracle_ref_golden, seed, S, Q, K):
    rs = np.random.RandomState(seed)
    sup = rs.randn(2, S, 3).astype(np.float32)
    qry = rs.randn(2, Q, 3).astype(np.float32)
    got = O.knn_batch(sup, qry, K)
    want = reference_knn(oracle_ref_golden, "random%d" % seed, got)
    ok, ndiff, _, msg = O.knn_matches(sup, qry, got, want)
    assert ok and ndiff == 0, msg


def test_knn_surface_frame(oracle_ref_golden):
    from ffb6d_b200.synthetic import make_frame
    fr = make_frame(9, n_points=3072)
    cld = fr["cld"][None]
    got = O.knn_batch(cld, cld, 16)
    assert np.array_equal(got, reference_knn(oracle_ref_golden, "surface", got))


@pytest.mark.parametrize("n_points", [4096, 40960, 131072])
def test_knn_stress_sweep_sizes(oracle_ref_golden, n_points):
    """BASELINE configs[4] sizes: the port still equals the reference's KD-tree on the big clouds
    (self search K = 16 on level 1, image -> cloud K = 1 and cloud -> image K = 32 on level 2)."""
    from ffb6d_b200.synthetic import make_frame
    fr = make_frame(21, n_points=n_points)
    lvl1 = fr["cld"][None, : n_points // 4]
    lvl2 = fr["cld"][None, : n_points // 16]
    img = np.ascontiguousarray(fr["dpt_xyz"][::4, ::4].reshape(1, -1, 3))
    # dense clouds do produce the odd exact fp32 distance tie (seen: one row of 10240 at N0 = 40960), and
    # the hole pixels of the image level are exact duplicates: rows may then differ in ORDER only
    for j, (sup, qry, k) in enumerate(((lvl1, lvl1, 16), (lvl2, img, 1), (img, lvl2, 32))):
        got = O.knn_batch(sup, qry, k)
        want = reference_knn(oracle_ref_golden, "stress%d_%d" % (n_points, j), got)
        ok, ndiff, nties, msg = O.knn_matches(sup, qry, got, want)
        assert ok and ndiff == nties, msg
        assert ndiff <= max(4, got.shape[1] // 1000) or sup is img, msg


def test_torch_ops_random(oracle_ref_golden):
    import torch
    want = oracle_ref_golden["torch"]
    g = torch.Generator().manual_seed(7)
    feat = torch.randn(3, 17, 211, 1, generator=g)
    idx = torch.randint(0, 211, (3, 50, 16), generator=g)
    got = O.random_sample(feat.numpy(), idx.numpy())
    assert got.shape == (3, 17, 50, 1) and sha256_of(got) == str(want["random_sample"])
    idx1 = torch.randint(0, 211, (3, 400, 1), generator=g)
    got = O.nearest_interpolation(feat.numpy(), idx1.numpy())
    assert got.shape == (3, 17, 400, 1) and sha256_of(got) == str(want["nearest_interpolation"])
    pc = torch.randn(2, 90, 6, generator=g)
    nidx = torch.randint(0, 90, (2, 90, 16), generator=g)
    got = O.gather_neighbour(pc.numpy(), nidx.numpy())
    assert got.shape == (2, 90, 16, 6) and sha256_of(got) == str(want["gather_neighbour"])


def test_grid_random(oracle_ref_golden):
    rs = np.random.RandomState(5)
    pts = (rs.randn(4000, 3) * 0.5).astype(np.float32)
    feats = rs.rand(4000, 3).astype(np.float32)
    op, of, _ = O.grid_sub_sampling(pts, feats, None, 0.07)
    o = np.lexsort((op[:, 2], op[:, 1], op[:, 0]))
    assert sha256_of(op[o]) == str(oracle_ref_golden["grid"]["points"])
    assert sha256_of(of[o]) == str(oracle_ref_golden["grid"]["features"])


def test_wrap_padded_frame_tie_order_differs_but_gathers_agree(oracle_ref_golden):
    """A frame padded with repeated pixels (np.pad 'wrap', ycb_dataset.py:230): thousands of index rows differ
    between the reference's KD-tree order and the (distance, index) order -- within the tie contract -- yet every
    gather of the forward pass returns the same values, because tied points are duplicates with identical features."""
    from conftest import frame_point_sets
    from ffb6d_b200.synthetic import make_frame
    from ffb6d_b200.tables import gather_schedule, knn_schedule
    n = 3072
    fr = make_frame(11, n_points=n)
    rs = np.random.RandomState(5)
    keep = fr["choose"][0][: n * 5 // 8]
    choose = np.pad(keep, (0, n - len(keep)), "wrap")[rs.permutation(n)]
    fr = dict(fr, cld=fr["dpt_xyz"].reshape(-1, 3)[choose])
    sets = frame_point_sets(fr, n)
    ref, ours, differing = {}, {}, 0
    for key, s, q, kk in knn_schedule(n):
        ours[key] = O.knn_search(sets[s][None], sets[q][None], kk)
        ref[key] = reference_knn(oracle_ref_golden, "wrap_" + key, ours[key])
        ok, _, _, msg = O.knn_matches(sets[s][None], sets[q][None], ours[key], ref[key])
        assert ok, (key, msg)
        differing += int((ref[key] != ours[key]).any(axis=2).sum())
    assert differing > 1000
    for d in (ref, ours):
        d.update({"cld_sub_idx%d" % i: d["cld_nei_idx%d" % i][:, : n // 4 ** (i + 1)] for i in range(4)})
    support_of = {key: s for key, s, q, kk in knn_schedule(n)}
    for op, key, C, S, Q, K in gather_schedule(n):
        if op == "choose":
            continue
        pts = sets[support_of[key.replace("cld_sub_idx", "cld_nei_idx")]]
        w = rs.normal(size=(min(C, 16), 3)).astype(np.float32)
        feat = np.sin(pts @ w.T * 7.0).T[None, :, :, None].astype(np.float32).copy()     # features = f(xyz)
        f = O.random_sample if op == "random_sample" else O.nearest_interpolation
        assert np.array_equal(f(feat, ref[key].astype(np.int64)), f(feat, ours[key].astype(np.int64))), key
