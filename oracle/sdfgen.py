"""CPU restatement of the reference's GT-SDF generator -- TEST INFRASTRUCTURE ONLY (never imported by the product).

Follows /root/reference/ext/sdfgen/sdf_from_points.cu line by line (the only native code of the reference tree,
built by ext/__init__.py:18-23; call sites dataset/av_gt_geometry.py:63-78 and models/loss.py:85):

  :150-166  kd-tree over ref_xyz; adaptive_knn > 0: ref_std[i] = mean over the adaptive_knn nearest reference points
            (the point itself included, distance 0) of the distance                                     (:158-166)
  :168-175  the nb_points nearest reference points of every query, nearest first
  :92-147   ComputeSDFKernel: d_k = <n_k, x - p_k>;  nearest neighbour (k = 0): |x - p_0| < stdv * ref_std[p_0] ?
            sdf = |d_0|, grad = sign(d_0) n_0  :  sdf = |x - p_0|, grad = (x - p_0)/|x - p_0|; sign = + iff more than
            nb_points/2 (integer division) of the d_k are > 0                                            (:118-146)
  :33-90    ComputeIMLSKernel: w_k = exp(-|x - p_k|^2/stdv^2 + min_k |x - p_k|^2/stdv^2), sdf = sum d_k w_k / sum w_k,
            grad = sum n_k w_k / sum w_k

Unlike the rest of oracle/, this restatement is PINNED: oracle/Makefile.ref compiles the unmodified reference sources
into oracle/_ref/nksr_sdfgen_ref.so, tests/golden/sdfgen/sdf_from_points_reference.npz holds that binary's output at a
sample of the queries, and tests/test_gpu_sdfgen.py checks both this file and the CUDA kernel against it on the GPU.
The k-NN search is exact (tinyflann eps = 0, ext/common/kdtree_cuda.cuh:34); scipy's cKDTree stands in.
"""
from __future__ import annotations

import numpy as np
from scipy.spatial import cKDTree


def sdf_from_points(queries, ref_xyz, ref_normal, nb_points, stdv, compute_grad=False, imls=False, adaptive_knn=0):
    q = np.asarray(queries, np.float32)
    p = np.asarray(ref_xyz, np.float32)
    nrm = np.asarray(ref_normal, np.float32)
    n_ref = p.shape[0]
    tree = cKDTree(p.astype(np.float64))
    ref_std = np.ones(n_ref, np.float32)
    if adaptive_knn > 0:
        d, _ = tree.query(p.astype(np.float64), k=adaptive_knn)
        ref_std = d.reshape(n_ref, -1).astype(np.float32).mean(axis=1)
    _, idx = tree.query(q.astype(np.float64), k=nb_points)
    idx = idx.reshape(q.shape[0], -1)
    ray = q[:, None, :] - p[idx]                                   # (M, k, 3)  x - p_k
    d = np.einsum('mkc,mkc->mk', nrm[idx], ray)                    # <n_k, x - p_k>
    if imls:
        e = np.einsum('mkc,mkc->mk', ray, ray) / np.float32(stdv * stdv)
        w = np.exp(-e + e.min(axis=1, keepdims=True))
        ws = w.sum(axis=1)
        sdf = (d * w).sum(axis=1) / ws
        grad = (nrm[idx] * w[:, :, None]).sum(axis=1) / ws[:, None]
    else:
        r0 = ray[:, 0, :]
        l0 = np.linalg.norm(r0, axis=1)
        near = l0 < np.float32(stdv) * ref_std[idx[:, 0]]
        mag = np.where(near, np.abs(d[:, 0]), l0)
        with np.errstate(divide='ignore', invalid='ignore'):
            g = np.where(near[:, None], np.where((d[:, 0] > 0)[:, None], nrm[idx[:, 0]], -nrm[idx[:, 0]]),
                         r0 / l0[:, None])
        pos = (d > 0).sum(axis=1) > (nb_points // 2)
        sdf = np.where(pos, mag, -mag)
        grad = np.where(pos[:, None], g, -g)
    out = [sdf.astype(np.float32)]
    if compute_grad:
        out.append(grad.astype(np.float32))
    return out


def decision_margins(queries, ref_xyz, ref_normal, nb_points, stdv, adaptive_knn=0):
    """how far every query is from the discontinuities of the non-IMLS rule (tests skip the queries that sit on one):
    (a) | |x - p_0| - stdv * ref_std | relative, (b) min_k |d_k| (a vote about to flip), (c) gap between the k-th and
    (k+1)-th neighbour distances (the neighbour SET about to change)"""
    q = np.asarray(queries, np.float64)
    p = np.asarray(ref_xyz, np.float64)
    tree = cKDTree(p)
    ref_std = np.ones(p.shape[0])
    if adaptive_knn > 0:
        d, _ = tree.query(p, k=adaptive_knn)
        ref_std = d.reshape(p.shape[0], -1).mean(axis=1)
    dist, idx = tree.query(q, k=nb_points + 1)
    dk = np.einsum('mkc,mkc->mk', np.asarray(ref_normal, np.float64)[idx[:, :nb_points]], q[:, None, :] - p[idx[:, :nb_points]])
    thr = stdv * ref_std[idx[:, 0]]
    a = np.abs(dist[:, 0] - thr) / np.maximum(thr, 1e-30)
    b = np.abs(dk).min(axis=1)
    c = dist[:, nb_points] - dist[:, nb_points - 1]
    return a, b, c
