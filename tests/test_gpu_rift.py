"""GPU parity of the descriptor-stage consumers (pcc_intensity_gradient, pcc_rift, process_rift) against the CPU oracle
(descriptor_oracle/ over oracle.KdTree radius rows), plus the C++ mirror self-test.  Bars: gradients bit-identical (only
correctly rounded fp32 operations, same order on both sides); RIFT bins <= 1e-5 absolute (acosf is not correctly rounded on
either side), identical NaN / zero rows.  Run on the B200 box with `-m gpu`."""
import os
import subprocess

import numpy as np
import pytest

import descriptor_oracle as D
import oracle
from conftest import bits
from pointcloudcomparator_b200 import synth

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def torch_cuda():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch


@pytest.fixture(scope="module")
def room():
    xyz = synth.room(100000, 31)[:, :3].copy()
    xyz[::997] = np.nan                                             # non-finite rows: skipped by the index, NaN output rows
    inten = synth.rgb_for(np.nan_to_num(xyz), 32)
    from pointcloudcomparator_b200.search import rgb_to_intensity
    inten = rgb_to_intensity(inten)
    tree = oracle.KdTree(xyz)
    q = synth.noisy_copy(np.nan_to_num(xyz), 34, 0.004)[:, :3][:20000].copy()
    far = np.array([[50.0, 50.0, 50.0], [-3.0, 1.0, 1.0]], np.float32)        # no neighbour at all
    return xyz, inten, tree, np.vstack([q, far]).astype(np.float32)


def same(a, b):
    """bit-identical, NaN payloads aside (the C oracle's NAN and CUDA's differ in payload only)"""
    a, b = np.asarray(a, np.float32), np.asarray(b, np.float32)
    na, nb = np.isnan(a), np.isnan(b)
    return a.shape == b.shape and np.array_equal(na, nb) and np.array_equal(bits(np.where(na, 0, a)), bits(np.where(nb, 0, b)))


def _oracle_gradient(xyz, inten, tree, qpts, normals, r):
    off, idx, _ = tree.radius(qpts, r)
    return D.intensity_gradient(xyz, off, idx, inten, normals), off


def test_intensity_gradient_bit_identical(torch_cuda, room):
    from pointcloudcomparator_b200.search import GridSearch
    xyz, inten, tree, q = room
    r = 0.03
    s = GridSearch().setInputCloud(xyz, cell_hint=r)
    # self (q == NULL): oracle normals of every input row (NaN rows for the skipped points)
    off0, idx0, _ = tree.radius(xyz, r)
    nrm_self = oracle.normals_from_lists(np.nan_to_num(xyz), np.nan_to_num(xyz), off0, idx0)
    want, off = _oracle_gradient(xyz, inten, tree, xyz, nrm_self, r)
    bad = ~np.isfinite(xyz).all(1)
    want[bad, :3] = np.nan
    got = s.intensityGradient(None, r, inten, nrm_self)
    assert same(got, want)
    assert np.isnan(got[bad, :3]).all() and (got[:, 3] == 0).all()
    counts = np.diff(off)
    assert (counts[~bad] < 3).any() and (counts[~bad] >= 3).any()
    # external noisy queries, host and device memory; rows with 0 / 1 / 2 neighbours are NaN
    offq, idxq, _ = tree.radius(q, r)
    nrm_q = oracle.normals_from_lists(np.nan_to_num(xyz), q, offq, idxq)
    nrm_q = np.where(np.isfinite(nrm_q), nrm_q, np.float32(0.0)).astype(np.float32)
    wq = D.intensity_gradient(xyz, offq, idxq, inten, nrm_q)
    cq = np.diff(offq)
    assert {0, 1, 2} <= set(cq.tolist())
    gh = s.intensityGradient(q, r, inten, nrm_q)
    assert same(gh, wq)
    torch = torch_cuda
    sd = GridSearch().setInputCloud(torch.as_tensor(xyz, device="cuda"), cell_hint=r)
    gd = sd.intensityGradient(torch.as_tensor(q, device="cuda"), r, torch.as_tensor(inten, device="cuda"), torch.as_tensor(nrm_q, device="cuda"))
    torch.cuda.synchronize()
    assert same(gd.cpu().numpy(), wq)
    assert np.isnan(gh[cq < 3, :3]).all()


@pytest.mark.parametrize("nd,ng", [(4, 8), (3, 7)])
def test_rift_matches_oracle(torch_cuda, room, nd, ng):
    from pointcloudcomparator_b200.search import GridSearch
    xyz, inten, tree, q = room
    r = 0.05
    rng = np.random.default_rng(35)
    grad = rng.normal(0, 50, (xyz.shape[0], 4)).astype(np.float32)
    grad[:, 3] = 0
    grad[::5, :3] = 0                                               # zero gradients: weight 0, NaN angle -> 0
    grad[::4001, :3] = np.nan                                       # NaN gradients poison the bins they reach, as in PCL
    s = GridSearch().setInputCloud(xyz, cell_hint=r)
    fin = np.isfinite(xyz).all(1)
    for qq in (None, q):
        qp = np.nan_to_num(xyz) if qq is None else qq
        off, idx, d2 = tree.radius(qp, r)
        want = D.rift(np.nan_to_num(xyz), qp, off, idx, d2, grad, r, nd, ng)
        if qq is None:
            want[~fin] = np.nan
        got = s.rift(qq, r, grad, nd, ng)
        assert got.shape == want.shape
        nan_g, nan_w = np.isnan(got), np.isnan(want)
        assert np.array_equal(nan_g, nan_w)
        # unit-norm rows: 1e-5 absolute per bin.  A NaN gradient in the neighbourhood leaves NaN bins and skips the normalisation
        # (its squared norm is NaN), so the other bins of such a row are raw weighted sums of gradient magnitudes: there the bar
        # is 1e-5 relative to the row's largest bin (processRIFT drops these rows as non-finite anyway).
        poisoned = nan_w.any(1) & ~nan_w.all(1)
        clean = ~nan_w.any(1)
        assert np.abs(got[clean] - want[clean]).max() <= 1e-5
        if poisoned.any():
            err = np.abs(np.where(nan_w, 0, got - want))[poisoned].max(1)
            scale = np.abs(np.where(nan_w, 0, want))[poisoned].max(1)
            assert (err <= 1e-5 * np.maximum(scale, 1.0)).all()
        zero_w = (np.where(nan_w, 1, want) == 0).all(1)
        assert np.array_equal((np.where(nan_g, 1, got) == 0).all(1), zero_w)
        assert np.isnan(want).all(1).any()                          # rows without neighbours (skipped self rows / far queries)
    torch = torch_cuda
    sd = GridSearch().setInputCloud(torch.as_tensor(xyz, device="cuda"), cell_hint=r)
    gd = sd.rift(torch.as_tensor(q, device="cuda"), r, torch.as_tensor(grad, device="cuda"), nd, ng)
    torch.cuda.synchronize()
    gh = s.rift(q, r, grad, nd, ng)
    assert same(gd.cpu().numpy(), gh)


def test_rift_rejects_more_than_32_bins(torch_cuda):
    from pointcloudcomparator_b200._lib import PccError
    from pointcloudcomparator_b200.search import GridSearch
    xyz = synth.room(2000, 36)[:, :3]
    s = GridSearch().setInputCloud(xyz)
    with pytest.raises(PccError):
        s.rift(None, 0.05, np.zeros((xyz.shape[0], 4), np.float32), 4, 9)


def _near_boundary(ref, qry, dims, thr=0.05, margin=1e-4):
    """queries whose oracle best distance is within margin of the threshold, or whose second best is within margin of the best"""
    a, b = np.asarray(ref, np.float64)[:, :dims], np.asarray(qry, np.float64)[:, :dims]
    d = ((b[:, None, :] - a[None, :, :]) ** 2).sum(-1)
    s = np.sort(d, axis=1)
    second = s[:, 1] if s.shape[1] > 1 else np.full(len(s), np.inf)
    return (np.abs(s[:, 0] - thr) < margin) | (second - s[:, 0] < margin)


def test_process_rift_end_to_end(torch_cuda):
    from pointcloudcomparator_b200.search import descriptor_nn, match_rift_features_knn, process_rift
    base = (synth.room(60000, 41)[:, :3] * 0.12).astype(np.float32)
    sel = np.flatnonzero(np.linalg.norm(base - base[0], axis=1) < 0.12)[:700]
    a = base[sel]
    b = synth.noisy_copy(a, 42, 0.0008)[:, :3]
    rgb = synth.rgb_for(a * 8, 43)                                   # the copy keeps its points' colours
    out = []
    for xyz in (a, b):
        dg, kg = process_rift(xyz, rgb)
        do, ko = D.process_rift(xyz, rgb)
        assert dg.shape == do.shape and np.array_equal(kg, ko), (dg.shape, do.shape)
        diff = float(np.abs(dg - do).max()) if dg.size else 0.0
        print(f"process_rift: {dg.shape[0]} descriptors of {xyz.shape[0]} points, max per-bin |gpu - oracle| = {diff:.3g}")
        out.append((dg, do))
    (ga, oa), (gb, ob) = out
    assert ga.shape[0] > 100
    for dims in (3, 32):
        okq = ~_near_boundary(oa, ob, dims)
        ig, dg2 = descriptor_nn(ga, gb, dims=dims)
        io, do2 = oracle.descriptor_nn(oa, ob, dims)
        acc_g, acc_o = (ig >= 0) & (dg2 < np.float32(0.05)), (io >= 0) & (do2 < np.float32(0.05))
        # the correspondence vectors of match_rift_features_knn, restricted to the queries away from the threshold and from ties
        assert [0] + ig[okq & acc_g].tolist() == [0] + io[okq & acc_o].tolist(), dims
        cg = match_rift_features_knn(ga, gb, match_dims=dims)
        print(f"match_dims={dims}: {len(cg) - 1} correspondences on the GPU, {int((~okq).sum())} boundary queries excluded")


@pytest.mark.gpu
def test_cpp_rift_mirror(torch_cuda):
    exe = os.path.join(ROOT, "tests", "cpp", "test_rift")
    assert os.path.exists(exe), "run __graft_entry__.build() first"
    out = subprocess.run([exe], capture_output=True, text=True, timeout=300)
    assert out.returncode == 0 and "PASS" in out.stdout, out.stdout + out.stderr
