"""The NumPy restatement of the MRF stage (tests/mrf_util.py) against exact dynamic programming on chains, and its
winner-take-all limit on the oracle's own peak lists.  CPU only."""
import numpy as np
import pytest

from stereoreconstruction_b200 import types as T
import mrf_util as M


class Mrf:
    """Duck-typed sr_mrf_params."""

    def __init__(self, iterations=16, unknown_cost=1.0, smooth_weight=0.05, smooth_trunc=8.0, unknown_pair=0.3):
        self.iterations, self.unknown_cost, self.smooth_weight = iterations, unknown_cost, smooth_weight
        self.smooth_trunc, self.unknown_pair = smooth_trunc, unknown_pair


P = T.default_params(True, 420.0, 580.0, 64)


@pytest.mark.parametrize("shape", [(1, 23), (31, 1), (1, 2), (1, 1)])
@pytest.mark.parametrize("seed", [0, 1, 2])
def test_bp_on_a_chain_reaches_viterbi(shape, seed):
    rng = np.random.RandomState(seed)
    h, w = shape
    lists = M.random_lists(h, w, rng, P, adversarial=False)
    mask = np.full(shape, 255, np.uint8)
    mp = Mrf(iterations=max(h, w) + 1, smooth_weight=0.3, smooth_trunc=6.0, unknown_pair=0.5, unknown_cost=0.8)
    lab, _, _, _, e = M.mrf_select(lists, mask, P, mp)
    unary, zs = M.prepare(lists, P)
    best, vlab = M.viterbi_chain(unary.reshape(M.K, -1), zs.reshape(M.K, -1), mp)
    assert e >= best * (1 - 1e-12)
    assert (lab.reshape(-1) == vlab).all() or abs(e - best) <= 1e-6 * abs(best), (e, best)


@pytest.mark.parametrize("seed", [3, 4])
def test_viterbi_energy_is_the_energy_of_its_labelling(seed):
    rng = np.random.RandomState(seed)
    lists = M.random_lists(1, 17, rng, P)
    mp = Mrf(smooth_weight=0.2, unknown_pair=0.4)
    unary, zs = M.prepare(lists, P)
    best, vlab = M.viterbi_chain(unary.reshape(M.K, -1), zs.reshape(M.K, -1), mp)
    e = M.energy(vlab.reshape(1, -1), unary, zs, np.ones((1, 17), bool), mp)
    assert e == pytest.approx(best, rel=1e-12)


@pytest.mark.parametrize("mp", [Mrf(unknown_cost=1e30, smooth_weight=0.0, unknown_pair=0.0),
                                Mrf(unknown_cost=1e30, iterations=0)])
def test_huge_unknown_cost_without_smoothing_is_the_wta(mp):
    """Sorted lists: slot 8 (the largest (ncc, depth) pair) wherever there is a candidate, U elsewhere."""
    rng = np.random.RandomState(5)
    lists = M.random_lists(13, 11, rng, P, adversarial=False)
    mask = np.where(rng.rand(13, 11) < 0.9, 255, 0).astype(np.uint8)
    lab, depth, best, index, _ = M.mrf_select(lists, mask, P, mp)
    inm = mask == 255
    cand = lists[..., 8, 1] != -1.0
    assert (lab[inm & cand] == 8).all() and (lab[inm & ~cand] == M.U).all()
    assert (depth[inm] == np.where(cand, lists[..., 8, 1], -1.0)[inm]).all()
    assert (best[inm] == np.where(cand, lists[..., 8, 0], 0.0)[inm]).all()
    assert (index[inm] == np.where(cand, 8, M.SR_INDEX_NONE)[inm]).all()
    assert np.isnan(depth[~inm]).all()


def test_oracle_peaks_wta_limit():
    """On the oracle's peak lists of a real (small) scene, in label and curve mode, the WTA limit of the model is
    the oracle's depth map."""
    from oracle import oracle_api as O
    from scene_util import refractive_arc_scene
    cams, imgs, ms, _ = refractive_arc_scene(V=3, w=96, h=64, masks=True)
    sc = O.Scene(cams, imgs, ms)
    Q = T.default_params(True, 420.0, 580.0, 32)
    nbrs = sc.select_neighbours(2)
    for curve in (False, True):
        depth, index, best, _, peaks = sc.mvs_view(Q, 0, nbrs[0], curve_mode=curve, want_peaks=True)
        _, d, b, _, _ = M.mrf_select(peaks, ms[0], Q, Mrf(unknown_cost=1e30, iterations=0), depth, best, index)
        inm = ms[0] == 255
        found = inm & (depth != -1.0)  # (the oracle's curve mode leaves the index at -1)
        assert found.sum() > 0.5 * inm.sum()
        assert (d[found] == depth[found]).all() and (b[found] == best[found]).all()
        assert (d[inm & ~found] == -1.0).all()


def test_half_sweep_writes_only_into_the_other_colour():
    rng = np.random.RandomState(6)
    lists = M.random_lists(9, 10, rng, P)
    unary, zs = M.prepare(lists, P)
    inmask = np.ones((9, 10), bool)
    msg = np.zeros((4, M.L, 9, 10), np.float32)
    M.half_sweep(msg, unary, zs, inmask, 0, Mrf(smooth_weight=0.3))
    yy, xx = np.mgrid[0:9, 0:10]
    even = ((yy + xx) & 1) == 0
    assert (msg[:, :, even] == 0).all()
    assert (msg[:, :, ~even] != 0).any()
    assert (msg >= 0).all() and np.isfinite(msg).all()
