"""Pin the ranking oracle (oracle/rank_oracle.c) to the reference: golden vectors produced by the
reference's evaluate_rank (tests/golden/make_golden.py) and the reference's own compiled rank_cy on larger
dataset-shaped inputs: its recorded outputs (tests/golden/fresh_rank_cy.npz) or, when built, oracle/_ref itself."""
import os

import numpy as np
import pytest

from conftest import GOLDEN, golden_files
from oracle import rank as orank
from oracle import synth


def _load(name):
    return dict(np.load(os.path.join(GOLDEN, name), allow_pickle=False))


@pytest.mark.parametrize('fname', golden_files('rank_'))
def test_market1501_port_matches_reference_golden(fname):
    g = _load(fname)
    args = (g['distmat'], g['q_pids'], g['g_pids'], g['q_camids'], g['g_camids'], int(g['max_rank']))
    if 'cy_error' in g:
        with pytest.raises(AssertionError):
            orank.market1501_port(*args)
        return
    cmc, mAP = orank.market1501_port(*args)
    assert cmc.dtype == np.float32 and cmc.shape == g['cy_cmc'].shape
    assert np.array_equal(cmc.view(np.uint32), g['cy_cmc'].view(np.uint32))        # bit-exact
    assert np.float32(mAP).view(np.uint32) == g['cy_mAP'].view(np.uint32)
    assert mAP == float(g['cy_mAP_f64'])
    if 'py_cmc' in g:      # the reference's float64 Python evaluator agrees to rounding (SURVEY 8c)
        assert np.array_equal(cmc, g['py_cmc'])
        assert abs(mAP - float(g['py_mAP'])) < 1e-6


@pytest.mark.parametrize('fname', golden_files('rank_'))
def test_mars_port_matches_reference_golden(fname):
    g = _load(fname)
    args = (g['distmat'], g['q_pids'], g['g_pids'], g['q_camids'], g['g_camids'], int(g['max_rank']))
    if 'mars_error' in g:
        exc = ZeroDivisionError if int(g['mars_error']) == 2 else ValueError
        with pytest.raises(exc):
            orank.mars_port(*args)
        return
    cmc, mAP = orank.mars_port(*args)
    assert cmc.dtype == np.float64
    assert np.array_equal(cmc.view(np.uint64), g['mars_cmc'].view(np.uint64))      # bit-exact
    assert np.float64(mAP).view(np.uint64) == g['mars_mAP'].view(np.uint64)


@pytest.mark.parametrize('n', [0, 1, 5, 8, 9, 127, 128, 129, 1000, 1980, 4099])
def test_pairwise_sum_is_numpys(n):
    x = np.random.RandomState(n).rand(n) * 3 - 1
    assert orank.pairwise_sum_f64(x) == (np.add.reduce(x) if n else 0.0)


FRESH_CY = 'fresh_rank_cy.npz'          # rank_cy's outputs on the inputs below (tests/golden/make_golden.py rank_cy)
FRESH_CY_CASES = [('dukev', 0, False), ('dukev', 1, True), ('ilidsvid', 2, False), ((200, 3000, 40, 5), 3, True)]


def fresh_cy_inputs(shape, seed, ties):
    """(key, distmat, q_pids, q_camids, g_pids, g_camids, checksum) of one case, regenerated from its seed."""
    qp, qc, gp, gc = synth.eval_labels(shape, seed=seed)
    nq, ng = len(qp), len(gp)
    if ties:
        d = synth.quantised_distmat(nq, ng, seed=seed)
    else:
        d = np.random.RandomState(seed).randn(nq, ng).astype(np.float32)
    key = '%s_%d_%d' % (shape if isinstance(shape, str) else 'x'.join(map(str, shape)), seed, ties)
    checksum = np.float64(d.astype(np.float64).sum() + sum((i + 2) * x.astype(np.float64).sum()
                                                           for i, x in enumerate((qp, qc, gp, gc))))
    return key, d, qp, qc, gp, gc, checksum


@pytest.mark.skipif(not os.path.exists(os.path.join(GOLDEN, FRESH_CY)) and orank.reference_rank_cy() is None,
                    reason='no stored outputs of the reference rank_cy (tests/golden/%s) and oracle/_ref not built' % FRESH_CY)
@pytest.mark.parametrize('shape,seed,ties', FRESH_CY_CASES)
def test_port_vs_compiled_reference_rank_cy(shape, seed, ties):
    key, d, qp, qc, gp, gc, checksum = fresh_cy_inputs(shape, seed, ties)
    cmc, mAP = orank.market1501_port(d, qp, gp, qc, gc, 50)
    if os.path.exists(os.path.join(GOLDEN, FRESH_CY)):
        g = _load(FRESH_CY)
        assert g[key + '_checksum'] == checksum, 'regenerated inputs drifted from the recorded ones'
        rcmc, rmAP = g[key + '_cmc'], float(g[key + '_mAP'])
    else:
        rcmc, rmAP = orank.reference_evaluate_cy(d, qp, gp, qc, gc, 50)
    assert np.array_equal(cmc.view(np.uint32), np.asarray(rcmc).view(np.uint32))
    assert mAP == rmAP
