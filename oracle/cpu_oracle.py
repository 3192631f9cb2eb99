"""oracle/cpu_oracle.py -- TEST INFRASTRUCTURE ONLY. NOT A PRODUCT PATH.

numpy / C restatements ("port") of the reference ops on the fusion hot path.  Each
function cites the reference lines it follows (relative to /root/reference/ffb6d/).
KNN and grid subsampling call the C restatements in liboracle.so (knn_oracle.c,
grid_oracle.c); the gather ops are closed-form numpy selections.

Pinned against the reference itself: tests/golden/ holds the outputs of the
reference's own code (oracle/_ref + AST-extracted torch functions) on seeded
inputs, and tests/test_oracle_golden.py / tests/test_oracle_vs_ref.py compare every
function here with them.
"""
import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = os.path.join(_HERE, "liboracle.so")


def build():
    """Compile liboracle.so (our C restatements) with the flags of oracle/Makefile."""
    subprocess.check_call(["make", "-s", "-C", _HERE, "all"])


def _load():
    if not os.path.exists(_LIB):
        build()
    lib = C.CDLL(_LIB)
    lib.oracle_knn_batch.restype = None
    lib.oracle_knn_batch.argtypes = [C.c_void_p, C.c_size_t, C.c_size_t, C.c_void_p, C.c_size_t,
                                     C.c_size_t, C.c_void_p, C.c_void_p]
    lib.oracle_sqdist_of_indices.restype = None
    lib.oracle_sqdist_of_indices.argtypes = [C.c_void_p, C.c_size_t, C.c_size_t, C.c_void_p,
                                             C.c_size_t, C.c_size_t, C.c_void_p, C.c_void_p]
    lib.oracle_grid_subsampling.restype = C.c_long
    lib.oracle_grid_subsampling.argtypes = [C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t,
                                            C.c_void_p, C.c_size_t, C.c_float, C.c_void_p,
                                            C.c_void_p, C.c_void_p, C.c_void_p]
    return lib


_lib = None


def lib():
    global _lib
    if _lib is None:
        _lib = _load()
    return _lib


# ----------------------------------------------------------------------------- KNN
def knn_batch(support, query, k, return_dist=False):
    """``nearest_neighbors.knn_batch`` (NN/knn.pyx:71-109 -> NN/knn_.cxx:72-135):
    support [B,S,3], query [B,Q,3] -> int64 [B,Q,k] (and fp32 squared distances)."""
    sup = np.ascontiguousarray(support, dtype=np.float32)
    qry = np.ascontiguousarray(query, dtype=np.float32)
    B, S, _ = sup.shape
    Q = qry.shape[1]
    idx = np.zeros((B, Q, k), dtype=np.int64)
    dist = np.zeros((B, Q, k), dtype=np.float32) if return_dist else None
    lib().oracle_knn_batch(sup.ctypes.data, B, S, qry.ctypes.data, Q, k, idx.ctypes.data,
                           dist.ctypes.data if return_dist else None)
    return (idx, dist) if return_dist else idx


def knn_search(support_pts, query_pts, k):
    """``DataProcessing.knn_search`` (models/RandLA/helper_tool.py:160-170): int32 result."""
    return knn_batch(support_pts, query_pts, k).astype(np.int32)


def subset_nn_from_knn(knn_idx, n_sub, support, query):
    """What ``ffb6d_knn_subset_nn`` must return, stated on the reference's own data flow: ``cld_interp_idx`` =
    ``knn_search(sub_pts, cld, 1)`` with ``sub_pts = cld[:N//4]`` (datasets/ycb/ycb_dataset.py:278-282), given
    ``knn_idx = knn_search(cld, cld, K)`` (:275-277, one frame, ``[Q,K]``): the first entry of a row that lies in the
    prefix ``[0, n_sub)``, a K = 1 search of the prefix for the rows that have none.  Returns ``([Q,1], #searched)``."""
    knn_idx = np.asarray(knn_idx)
    out = np.empty((len(knn_idx), 1), knn_idx.dtype)
    missed = []
    for q, row in enumerate(knn_idx):
        hit = row[row < n_sub]
        if len(hit):
            out[q, 0] = hit[0]
        else:
            missed.append(q)
    if missed:
        out[missed] = knn_search(np.asarray(support)[None], np.asarray(query)[missed][None], 1)[0]
    return out, len(missed)


def sqdist_of_indices(support, query, idx):
    """Reference-arithmetic squared distances of given neighbour indices [B,Q,K] (-1 when an
    index is out of range)."""
    sup = np.ascontiguousarray(support, dtype=np.float32)
    qry = np.ascontiguousarray(query, dtype=np.float32)
    ii = np.ascontiguousarray(idx, dtype=np.int64)
    B, S, _ = sup.shape
    Q, K = ii.shape[1], ii.shape[2]
    out = np.empty((B, Q, K), np.float32)
    lib().oracle_sqdist_of_indices(sup.ctypes.data, B, S, qry.ctypes.data, Q, K, ii.ctypes.data,
                                   out.ctypes.data)
    return out


def knn_matches(support, query, got_idx, want_idx):
    """The parity contract for neighbour indices (DESIGN.md "tie contract").

    Rows must be bit-identical, except rows whose reference-arithmetic distances contain an
    exact tie inside the first K+1 neighbours: there the SORTED DISTANCES must still be
    bit-identical (same multiset of fp32 distances; order among equals is a traversal
    artefact of the reference's KD-tree, SURVEY.md App. B).  Returns (ok, n_rows_differing,
    n_rows_excused_by_ties, message)."""
    got = np.asarray(got_idx).astype(np.int64)
    want = np.asarray(want_idx).astype(np.int64)
    if got.shape != want.shape:
        return False, -1, 0, "shape %s vs %s" % (got.shape, want.shape)
    diff_rows = np.argwhere((got != want).any(axis=2))
    if len(diff_rows) == 0:
        return True, 0, 0, "bit-exact"
    S = np.asarray(support).shape[1]
    if got.min() < 0 or got.max() >= max(S, 1):
        return False, len(diff_rows), 0, "index out of range"
    dg = sqdist_of_indices(support, query, got)
    dw = sqdist_of_indices(support, query, want)
    K = got.shape[2]
    for b, q in diff_rows:
        a, w = dg[b, q], dw[b, q]
        # A differing index with a bit-identical distance at the same rank IS an exact tie:
        # two distinct support points at the same fp32 distance from the query.
        distinct = len(set(got[b, q, :min(K, S)].tolist())) == min(K, S)
        if not (distinct and np.array_equal(a, w)):
            return False, len(diff_rows), 0, (
                "row (b=%d,q=%d) differs beyond ties: got %s (d=%s) want %s (d=%s)"
                % (b, q, got[b, q], a, want[b, q], w))
    n = len(diff_rows)
    return True, n, n, "%d rows differ, all by exact-distance ties" % n


# ----------------------------------------------------------------------------- gathers
def random_sample(feature, pool_idx):
    """``FFB6D.random_sample`` (models/ffb6d.py:159-177): feature [B,C,S,1] or [B,C,S],
    pool_idx [B,Q,K] -> [B,C,Q,1]; out[b,c,q] = max_k feature[b,c,idx[b,q,k]]."""
    f = np.asarray(feature)
    if f.ndim > 3:
        f = f.squeeze(3)
    idx = np.asarray(pool_idx).astype(np.int64)
    B, Cc, _ = f.shape
    Q, K = idx.shape[1], idx.shape[2]
    out = np.empty((B, Cc, Q, 1), f.dtype)
    for b in range(B):
        g = f[b][:, idx[b].reshape(-1)].reshape(Cc, Q, K)     # torch.gather(dim=2)
        out[b, :, :, 0] = g.max(axis=2)                        # .max(dim=3)
    return out


def nearest_interpolation(feature, interp_idx):
    """``FFB6D.nearest_interpolation`` (models/ffb6d.py:179-194): feature [B,C,S,1],
    interp_idx [B,Q,1] -> [B,C,Q,1]; out[b,c,q] = feature[b,c,idx[b,q,0]]."""
    f = np.asarray(feature).squeeze(3)
    idx = np.asarray(interp_idx).astype(np.int64)
    B, up = idx.shape[0], idx.shape[1]
    idx = idx.reshape(B, up)
    out = np.stack([f[b][:, idx[b]] for b in range(B)])
    return out[..., None]


def choose_gather(rgb_emb, choose):
    """models/ffb6d.py:309-312: rgb_emb [B,C,H,W], choose [B,1,N] -> [B,C,N]."""
    f = np.asarray(rgb_emb)
    B, Cc = f.shape[:2]
    f = f.reshape(B, Cc, -1)
    ch = np.asarray(choose).astype(np.int64).reshape(B, -1)
    return np.stack([f[b][:, ch[b]] for b in range(B)])


def gather_neighbour(pc, neighbor_idx):
    """``Building_block.gather_neighbour`` (models/RandLA/RandLANet.py:225-234):
    pc [B,N,d], idx [B,N,K] -> [B,N,K,d]."""
    pc = np.asarray(pc)
    idx = np.asarray(neighbor_idx).astype(np.int64)
    B, N, K = idx.shape
    return np.stack([pc[b][idx[b].reshape(-1)].reshape(N, K, pc.shape[2]) for b in range(B)])


def relative_pos_encoding(xyz, neigh_idx):
    """``Building_block.relative_pos_encoding`` (RandLANet.py:216-223), fp32:
    [ sqrt(sum(rel^2)), rel, xyz_tile, neighbor_xyz ] -> [B,N,K,10]."""
    xyz = np.asarray(xyz, dtype=np.float32)
    nb = gather_neighbour(xyz, neigh_idx)
    tile = np.repeat(xyz[:, :, None, :], nb.shape[2], axis=2)
    rel = tile - nb
    sq = rel * rel
    dis = np.sqrt((sq[..., 0] + sq[..., 1]) + sq[..., 2])[..., None]
    return np.concatenate([dis, rel, tile, nb], axis=-1).astype(np.float32)


def gather_max_backward(feature3, idx, grad_out):
    """Autograd of gather+max (SURVEY.md §8a note): grad routed to the arg-max neighbour
    (first maximal k), accumulated in float64 then cast -- tolerance-level oracle."""
    f = np.asarray(feature3)
    idx = np.asarray(idx).astype(np.int64)
    g = np.asarray(grad_out)
    B, Cc, S = f.shape
    Q, K = idx.shape[1], idx.shape[2]
    gf = np.zeros((B, Cc, S), np.float64)
    for b in range(B):
        vals = f[b][:, idx[b].reshape(-1)].reshape(Cc, Q, K)
        am = vals.argmax(axis=2)                               # first max
        src = np.take_along_axis(np.broadcast_to(idx[b][None], (Cc, Q, K)), am[..., None], 2)[..., 0]
        for c in range(Cc):
            np.add.at(gf[b, c], src[c], g[b, c].astype(np.float64))
    return gf.astype(np.float32)


# ----------------------------------------------------------------------------- grid subsampling
def grid_sub_sampling(points, features=None, labels=None, grid_size=0.1):
    """``DataProcessing.grid_sub_sampling`` (helper_tool.py:199-219 ->
    GS/cpp_subsampling/grid_subsampling/grid_subsampling.cpp:5-106).  Rows by ascending
    voxel key.  Returns (points[, features][, labels], keys)."""
    pts = np.ascontiguousarray(points, dtype=np.float32)
    N = pts.shape[0]
    feats = None if features is None else np.ascontiguousarray(features, dtype=np.float32)
    cls = None if labels is None else np.ascontiguousarray(labels, dtype=np.int32)
    fdim = 0 if feats is None else feats.shape[1]
    ldim = 0 if cls is None else (1 if cls.ndim == 1 else cls.shape[1])
    sp = np.empty((N, 3), np.float32)
    sf = np.empty((N, max(fdim, 1)), np.float32)
    sc = np.empty((N, max(ldim, 1)), np.int32)
    keys = np.empty((N,), np.uint64)
    M = lib().oracle_grid_subsampling(pts.ctypes.data, N,
                                      feats.ctypes.data if feats is not None else None, fdim,
                                      cls.ctypes.data if cls is not None else None, ldim,
                                      float(grid_size), sp.ctypes.data, sf.ctypes.data,
                                      sc.ctypes.data, keys.ctypes.data)
    if M < 0:
        raise RuntimeError("oracle_grid_subsampling failed")
    out = [sp[:M].copy()]
    if feats is not None:
        out.append(sf[:M, :fdim].copy())
    if cls is not None:
        out.append(sc[:M, :ldim].copy())
    out.append(keys[:M].copy())
    return tuple(out)
