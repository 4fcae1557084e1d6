"""CPU check of the derivation pcc_rift_batched relies on: one (d2, index)-sorted radius pass at R = max(r_n, r_g, r_r) over the
union of the clusters, with neighbours restricted to the query's own cluster, yields every stage row set of per-cluster processRIFT.
A stage's row is the prefix with d2 < float(r^2); for the gradient and RIFT stages the neighbours with a non-finite normal are then
removed and the rows of such queries are empty.  Filtering renumbers points in increasing order, so the rows keep their order.  The
derived rows must equal the directly searched per-cluster rows, and the descriptors computed on them must be bit-identical to
descriptor_oracle.process_rift on each cluster alone."""
import numpy as np

import descriptor_oracle as D
import oracle
from conftest import bits
from pointcloudcomparator_b200 import synth

RN, RG, RR = 0.03, 0.03, 0.05


def _patch(n, radius, seed):
    base = (synth.room(60000, seed)[:, :3] * 0.12).astype(np.float32)
    return np.ascontiguousarray(base[np.flatnonzero(np.linalg.norm(base - base[0], axis=1) < radius)[:n]])


def _batch():
    """two clusters interleaved in space, a third overlapping them, a sparse cluster (drops at the normals and for NaN gradients),
    a 2-point cluster and an empty cluster"""
    a = _patch(700, 0.12, 41)
    b = _patch(700, 0.12, 45) + np.float32([0.05, 0, 0])
    lab = np.random.default_rng(62).integers(0, 3, a.shape[0])
    sparse = _patch(3000, 0.3, 47)[::9]
    clusters = [a[lab == 0], a[lab == 1], b, sparse, a[:2], np.empty((0, 3), np.float32)]
    rgbs = [synth.rgb_for(c * 8, 43 + i) for i, c in enumerate(clusters)]
    off = np.concatenate([[0], np.cumsum([c.shape[0] for c in clusters])]).astype(np.int64)
    return clusters, rgbs, np.concatenate(clusters).astype(np.float32), np.concatenate(rgbs).astype(np.uint8), off


def _stage_rows(mo, mi, md, seg, r, keep):
    """rows at radius r from the master rows (mo, mi, md): the prefix d2 < float(r^2), neighbours with keep[] only, empty rows for
    queries without keep[]"""
    r2 = np.float32(r * r)
    n = mo.size - 1
    off = np.zeros(n + 1, np.int64)
    nbr, d2 = [], []
    for q in range(n):
        sl = slice(mo[q], mo[q + 1])
        i, d = mi[sl], md[sl]
        assert (seg[i] == seg[q]).all()
        p = int(np.searchsorted(d, r2, side="left"))                 # sorted by d2: the prefix below r2
        assert (d[:p] < r2).all() and (d[p:] >= r2).all()
        m = keep[i[:p]] if keep[q] else np.zeros(p, bool)
        nbr.append(i[:p][m]), d2.append(d[:p][m])
        off[q + 1] = off[q] + int(m.sum())
    return off, np.concatenate(nbr).astype(np.int32), np.concatenate(d2).astype(np.float32)


def _same_rows(derived, direct, rows, local):
    """derived rows of `rows` (global indices, renumbered by `local`) == the directly searched rows"""
    o, i, d = derived
    wo, wi, wd = direct
    got_off = np.concatenate([[0], np.cumsum(o[rows + 1] - o[rows])]).astype(np.int64)
    assert np.array_equal(got_off, wo)
    gi = np.concatenate([i[o[q]:o[q + 1]] for q in rows] + [np.empty(0, np.int32)])
    gd = np.concatenate([d[o[q]:o[q + 1]] for q in rows] + [np.empty(0, np.float32)])
    assert np.array_equal(local[gi], wi) and np.array_equal(bits(gd), bits(wd))


def test_one_sorted_pass_yields_every_stage_of_every_cluster():
    clusters, rgbs, xyz, rgb, off = _batch()
    n = xyz.shape[0]
    seg = np.repeat(np.arange(off.size - 1), np.diff(off))
    # the master pass: every row at R, restricted to the query's cluster, sorted by (d2, index) as the oracle's radius rows are
    mo, mi, md = oracle.KdTree(xyz).radius(xyz, max(RN, RG, RR))
    rows = [], [], []
    for q in range(n):
        sl = slice(mo[q], mo[q + 1])
        m = seg[mi[sl]] == seg[q]
        rows[0].append(mi[sl][m]), rows[1].append(md[sl][m]), rows[2].append(int(m.sum()))
    mo = np.concatenate([[0], np.cumsum(rows[2])]).astype(np.int64)
    mi, md = np.concatenate(rows[0]).astype(np.int32), np.concatenate(rows[1]).astype(np.float32)

    on = _stage_rows(mo, mi, md, seg, RN, np.ones(n, bool))
    nrm = oracle.normals_from_lists(xyz, xyz, on[0], on[1])
    keep = np.isfinite(nrm[:, :3]).all(1)
    og = _stage_rows(mo, mi, md, seg, RG, keep)
    orr = _stage_rows(mo, mi, md, seg, RR, keep)
    grad = D.intensity_gradient(xyz, og[0], og[1], D.rgb_to_intensity(rgb), nrm)
    desc = D.rift(xyz, xyz, orr[0], orr[1], orr[2], grad, RR)
    ok = keep & np.isfinite(desc).all(1)

    drops = []
    for c, (x, r) in enumerate(zip(clusters, rgbs)):
        b, e = int(off[c]), int(off[c + 1])
        if b == e:
            assert not ok[b:e].any()
            continue
        st = {}
        dw, kw = D.process_rift(x, r, stages=st)
        # normals stage: the cluster's own rows at r_n
        local = np.full(n, -1, np.int64)
        local[b:e] = np.arange(e - b)
        _same_rows(on, oracle.KdTree(x).radius(x, RN), np.arange(b, e), local)
        # gradient and RIFT stages: the rows of the cluster's filtered cloud, renumbered
        k1 = st["kept_normals"]
        assert np.array_equal(k1, np.flatnonzero(keep[b:e]))
        local = np.full(n, -1, np.int64)
        local[b + k1] = np.arange(k1.size)
        x1 = np.ascontiguousarray(x[k1])
        t1 = oracle.KdTree(x1)
        _same_rows(og, t1.radius(x1, RG), b + k1, local)
        _same_rows(orr, t1.radius(x1, RR), b + k1, local)
        # descriptors and kept rows, bit for bit
        kg = np.flatnonzero(ok[b:e])
        assert np.array_equal(kg, kw)
        assert np.array_equal(bits(desc[b:e][kg]), bits(dw))
        drops.append((e - b - k1.size, k1.size - kw.size))
    # the sparse cluster drops rows at both stages, and some of its dropped points lie within r_r of kept ones
    assert drops[3][0] > 0 and drops[3][1] > 0
    b, e = int(off[3]), int(off[4])
    dropped = ~keep[b:e]
    near = oracle.KdTree(xyz[b:e][dropped]).radius(xyz[b:e][keep[b:e]], RR)[0]
    assert near[-1] > 0
