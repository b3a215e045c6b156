#!/usr/bin/env python
"""Regenerate tests/golden/*.npz by RUNNING THE REFERENCE ITSELF (imported from /root/reference).

Run in the build container only (the GPU box has no /root/reference):

    make -C oracle ref && python tests/golden/make_golden.py

What is recorded
    rank_*.npz       inputs + outputs of the reference's evaluate_rank for the market1501 metric
                     (Cython rank_cy, compiled unmodified into oracle/_ref, AND the pure-Python
                     eval_market1501) and for the MARS metric (evaluate_mars), numpy.argsort forced
                     to kind='stable' (tie order is otherwise undefined in the reference).
    distance_*.npz   inputs + outputs of the reference's compute_distance_matrix (CPU tensors).
    head_*.npz       outputs of the reference's GSTA.forward (vmgn.py:292-321) with featuremaps()
                     replaced by seeded synthetic maps; inputs are NOT stored (regenerated from
                     oracle.synth with the recorded seeds; a float64 checksum guards RNG drift).

Harness-side shims only (reference files untouched): sklearn.metrics.base alias (rank.py:242),
model_zoo.load_url stub (vmgn.py:225,365 downloads ImageNet weights), rank_cy injected from oracle/_ref.
"""
import contextlib
import io
import os
import sys

sys.dont_write_bytecode = True
HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
REF = os.environ.get('AGRL_REFERENCE', '/root/reference')
sys.path.insert(0, ROOT)

import numpy as np
import torch
import torch.utils.model_zoo as mz
import sklearn.metrics._base as _skb

from oracle import rank as orank
from oracle import synth

sys.modules['sklearn.metrics.base'] = _skb
mz.load_url = lambda *a, **k: {}
ref_cy = orank.reference_rank_cy()
assert ref_cy is not None, 'run `make -C oracle ref` first'
sys.path.insert(0, REF)
import torchreid.metrics.rank_cylib as _rcl          # noqa: E402  (package exists in the reference)
sys.modules['torchreid.metrics.rank_cylib.rank_cy'] = ref_cy
_rcl.rank_cy = ref_cy
from torchreid import metrics as ref_metrics          # noqa: E402
from torchreid.metrics import rank as ref_rank        # noqa: E402
from torchreid.models.vmgn import vmgn as ref_vmgn    # noqa: E402

assert ref_rank.IS_CYTHON_AVAI


def quiet(fn, *a, **k):
    with contextlib.redirect_stdout(io.StringIO()):
        return fn(*a, **k)


# ------------------------------------------------------------------------------------------ rank
def rank_case(name, distmat, qp, qc, gp, gc, max_rank):
    out = dict(distmat=distmat.astype(np.float32), q_pids=qp, q_camids=qc, g_pids=gp, g_camids=gc,
               max_rank=np.int64(max_rank))
    with orank.stable_argsort():
        try:
            cmc, mAP = quiet(ref_metrics.evaluate_rank, distmat, qp, gp, qc, gc, max_rank=max_rank,
                             use_metric_market1501=True, use_cython=True)
            out['cy_cmc'], out['cy_mAP'] = np.asarray(cmc), np.float32(mAP)
            assert out['cy_cmc'].dtype == np.float32
            out['cy_mAP_f64'] = np.float64(mAP)       # the python float rank_cy returns
        except AssertionError:
            out['cy_error'] = np.int64(1)
        try:
            cmc, mAP = quiet(ref_metrics.evaluate_rank, distmat, qp, gp, qc, gc, max_rank=max_rank,
                             use_metric_market1501=True, use_cython=False)
            out['py_cmc'], out['py_mAP'] = np.asarray(cmc), np.float64(mAP)
        except (AssertionError, ValueError, AttributeError):
            pass                                       # ragged cmc rows / np.bool in old code paths
        try:
            cmc, mAP = quiet(ref_metrics.evaluate_rank, distmat, qp, gp, qc, gc, max_rank=max_rank,
                             use_metric_mars=True)
            out['mars_cmc'], out['mars_mAP'] = np.asarray(cmc), np.float64(mAP)
            assert out['mars_cmc'].dtype == np.float64
        except ZeroDivisionError:
            out['mars_error'] = np.int64(2)
        except ValueError:
            out['mars_error'] = np.int64(3)
    np.savez_compressed(os.path.join(HERE, 'rank_%s.npz' % name), **out)
    print('rank_%s' % name, {k: (v.shape if hasattr(v, 'shape') and v.shape else v) for k, v in out.items()
                             if k not in ('distmat', 'q_pids', 'q_camids', 'g_pids', 'g_camids')})


def make_rank():
    rng = np.random.RandomState(7)
    # (1) the shape of the reference's own timing script (rank_cylib/test_cython.py:29-37)
    nq, ng = 30, 300
    qp, qc, gp, gc = synth.eval_labels((nq, ng, 12, 3), seed=1)
    rank_case('testcython_shape', (rng.rand(nq, ng) * 20).astype(np.float32), qp, qc, gp, gc, 5)
    # (2) heavy exact ties
    nq, ng = 40, 400
    qp, qc, gp, gc = synth.eval_labels((nq, ng, 10, 4), seed=2)
    rank_case('ties', synth.quantised_distmat(nq, ng, seed=3, levels=16), qp, qc, gp, gc, 50)
    # (3) distractors (pid == -1) + queries without any gallery identity (skipped by rank_cy)
    nq, ng = 48, 700
    qp, qc, gp, gc = synth.eval_labels((nq, ng, 20, 6), seed=4, distractor_frac=0.2)
    qp2 = qp.copy()
    qp2[:5] = 10_000 + np.arange(5)                   # identities absent from the gallery
    d = rng.randn(nq, ng).astype(np.float32)
    rank_case('distractors', d, qp, qc, gp, gc, 50)
    rank_case('absent_ids', d, qp2, qc, gp, gc, 50)    # MARS metric -> ZeroDivisionError
    # (4) tiny gallery: max_rank clamps to num_g and kept < max_rank -> rank_cy's stale cmc tail
    nq, ng = 25, 12
    qp, qc, gp, gc = synth.eval_labels((nq, ng, 4, 2), seed=5)
    rank_case('tiny_gallery', rng.rand(nq, ng).astype(np.float32), qp, qc, gp, gc, 50)
    # (5) iLIDS/PRID style: one gallery item per id, other camera
    qp, qc, gp, gc = synth.eval_labels('prid2011', seed=0)
    qf, gf = synth.eval_features(qp, gp, 64, seed=6, clustered=True)
    d = ref_metrics.compute_distance_matrix(qf, gf, 'euclidean').numpy()
    rank_case('prid_shape', d, qp, qc, gp, gc, 50)
    # (6) special values: -0.0/+0.0 ties, inf, and a query with no valid identity at all
    nq, ng = 16, 128
    qp, qc, gp, gc = synth.eval_labels((nq, ng, 6, 3), seed=8)
    d = rng.randn(nq, ng).astype(np.float32)
    d[:, ::7] = 0.0
    d[:, 3::14] = -0.0
    d[:, 5::31] = np.inf
    d[:, 6::37] = -np.inf
    rank_case('special_values', d, qp, qc, gp, gc, 20)
    # (7) every query invalid -> AssertionError in rank_cy
    rank_case('all_invalid', d, qp + 1000, qc, gp, gc, 20)


# -------------------------------------------------------------------------------------- distance
def make_distance():
    g = torch.Generator().manual_seed(11)
    for name, (m, n, d) in {'small': (37, 53, 200), 'odd': (5, 131, 77), 'wide': (16, 24, 4096)}.items():
        a = torch.randn(m, d, generator=g)
        b = torch.randn(n, d, generator=g)
        if name == 'odd':
            b[3] = 0.0                                  # zero row: cosine eps clamp
            a[1] = b[7]                                 # identical pair: euclid ~ 0, cosine ~ 0
        out = dict(a=a.numpy(), b=b.numpy())
        for metric in ('euclidean', 'cosine'):
            out[metric] = ref_metrics.compute_distance_matrix(a, b, metric).numpy()
        np.savez_compressed(os.path.join(HERE, 'distance_%s.npz' % name), **out)
        print('distance_%s' % name, out['euclidean'].shape)


# ------------------------------------------------------------------------------------------ head
def make_head():
    torch.manual_seed(0)
    model = quiet(ref_vmgn, num_classes=625, loss={'xent', 'htri'}, last_stride=1, num_split=4,
                  num_gb=2, num_scale=1, pyramid_part=True, use_pose=True, learn_graph=True).eval()
    cases = {
        # name: (B, w, maps seed, scale, adj mode, weights seed, randomise_bn)
        'pose': (2, 2, 21, 1.0, 'pose', 31, True),
        'zeros_adj': (1, 1, 22, 1.0, 'zeros', 32, True),
        'ones_adj': (1, 1, 23, 1.0, 'ones', 33, False),
        'scaled': (2, 1, 24, 20.0, 'pose', 34, True),     # exp(d) and the 1e-12 clamp get exercised
    }
    for name, (B, w, mseed, scale, mode, wseed, rbn) in cases.items():
        S, C, h = 8, 2048, 16
        x4_1, x4_2 = synth.feature_maps(B, S, C, h, w, seed=mseed, scale=scale)
        adj = synth.pose_adjacency(B, S, 7, seed=mseed, mode=mode)
        wts = synth.head_weights(C, 2, seed=wseed, randomise_bn=rbn)
        sd = model.state_dict()
        for k, v in wts.items():
            assert sd[k].shape == v.shape, k
            sd[k].copy_(v)
        model.featuremaps = lambda x, a=x4_1, b=x4_2: (a, b)      # everything after :295 is the reference
        with torch.no_grad():
            out = model(torch.zeros(B, S, 3, 4, 4), adj)
        rec = dict(out=out.numpy(), B=np.int64(B), w=np.int64(w), maps_seed=np.int64(mseed),
                   scale=np.float64(scale), weights_seed=np.int64(wseed), randomise_bn=np.int64(rbn),
                   adj_mode=np.array(mode),
                   checksum=np.float64(x4_1.double().sum() + 3 * x4_2.double().sum() + 7 * adj.double().sum()
                                       + sum(v.double().sum() for v in wts.values())))
        np.savez_compressed(os.path.join(HERE, 'head_%s.npz' % name), **rec)
        print('head_%s' % name, out.shape, float(out.abs().max()))


if __name__ == '__main__':
    which = sys.argv[1:] or ['rank', 'distance', 'head']
    if 'rank' in which:
        make_rank()
    if 'distance' in which:
        make_distance()
    if 'head' in which:
        make_head()


# ------------------------------------------------------------------------------------ full model
def make_full_model():
    """Whole reference VMGN (random-init ResNet-50 under seed 0, eval) on one synthetic tracklet,
    CPU fp32 -- used for the end-to-end check through the stock cuDNN backbone -- and the list of
    state_dict keys/shapes the drop-in module must reproduce (SURVEY.md section 5, checkpoint row)."""
    import json
    torch.manual_seed(0)
    model = quiet(ref_vmgn, num_classes=625, loss={'xent', 'htri'}, last_stride=1, num_split=4,
                  num_gb=2, num_scale=1, pyramid_part=True, use_pose=True, learn_graph=True).eval()
    sd = model.state_dict()
    with open(os.path.join(HERE, 'vmgn_state_dict_keys.json'), 'w') as f:
        json.dump([[k, list(v.shape)] for k, v in sd.items()], f)
    g = torch.Generator().manual_seed(77)
    x = torch.randn(2, 8, 3, 256, 128, generator=g)
    adj = synth.pose_adjacency(2, 8, 7, seed=77)
    with torch.no_grad():
        out = model(x, adj)
        x4_1, x4_2 = model.featuremaps(x.view(16, 3, 256, 128))
    np.savez_compressed(os.path.join(HERE, 'full_model.npz'), out=out.numpy(), input_seed=np.int64(77),
                        model_seed=np.int64(0), x_checksum=np.float64(x.double().sum()),
                        map_absmax=np.float64(max(x4_1.abs().max(), x4_2.abs().max())),
                        conv1_checksum=np.float64(sd['conv1.weight'].double().sum()))
    print('full_model', out.shape, float(out.abs().max()), float(x4_1.abs().max()))


if __name__ == '__main__' and ('full' in sys.argv[1:] or not sys.argv[1:]):
    make_full_model()


# ------------------------------------------------------------------------------------ pose graph
def make_pose():
    """The reference's own generate_graph (dataset_loader.py:218-343 -> adj_graph :345-388) on synthetic OpenPose
    detections: MARS-style paths, a pose dict with some frames missing (KeyError -> empty sets), integer image sizes.
    Stored: the detections and the (56, 56) adjacency per tracklet (bit-packed)."""
    from torchreid.dataset_loader import generate_graph as ref_generate_graph
    B, S = 24, 8
    kp, heights, valid = synth.pose_keypoints(B, S, seed=21)
    kp[1, :, :, 2] = 0.0                         # a tracklet without a single confident keypoint -> all-zero graph
    valid[2] = 0                                 # a tracklet whose pose file has no entry at all
    kp[3, 2] = np.nan                            # NaN coordinates / confidences in one frame
    heights[4] = 7.0                             # tiny boxes: np.arange yields MORE than num_split + 1 boundaries below h = 4 only
    heights[5, :3] = [1.0, 2.0, 3.0]             # ... exercised here
    adjs = []
    for b in range(B):
        paths = ['data/mars/bbox_test/%04d/%04dC1T%04dF%03d.jpg' % (b, b, b, s) for s in range(S)]
        poses = {p.split('/')[-1]: kp[b, s] for s, p in enumerate(paths) if valid[b, s]}
        sizes = [(128, int(heights[b, s])) for s in range(S)]
        adj = ref_generate_graph([None] * S, im_paths=paths, im_sizes=sizes, poses=poses, num_split=4, num_parts=3,
                                 num_scale=1, pyramid_part=True)
        adjs.append(adj.numpy())
    adjs = np.stack(adjs)
    assert adjs.shape == (B, 56, 56) and set(np.unique(adjs)) <= {0.0, 1.0}
    np.savez_compressed(os.path.join(HERE, 'pose_graph.npz'), keypoints=kp, heights=heights, valid=valid,
                        adj_bits=np.packbits(adjs.astype(np.uint8), axis=-1), density=np.float64(adjs.mean()))
    print('pose_graph', adjs.shape, 'density %.3f' % adjs.mean(), 'empty graphs', int((adjs.sum((1, 2)) == 0).sum()))


if __name__ == '__main__' and ('pose' in sys.argv[1:] or not sys.argv[1:]):
    make_pose()


# ------------------------------------------------------------------------------------ re-ranking
def make_rerank():
    """The reference's own re_ranking() (utils/re_ranking.py:30-94) as test() calls it (train_vidreid_xent_htri.py:
    523-527: the three distance matrices come from compute_distance_matrix), numpy.argsort forced stable."""
    from torchreid.utils.re_ranking import re_ranking as ref_re_ranking
    cases = {
        'clustered': dict(nq=40, ng=260, nid=12, d=64, metric='euclidean', k1=20, k2=6, lam=0.3),
        'cosine': dict(nq=25, ng=150, nid=8, d=48, metric='cosine', k1=20, k2=6, lam=0.3),
        'tiny': dict(nq=3, ng=9, nid=2, d=16, metric='euclidean', k1=20, k2=6, lam=0.3),     # N < k1 + 1
        'k2_one': dict(nq=20, ng=120, nid=6, d=32, metric='euclidean', k1=10, k2=1, lam=0.5),
        'ties': dict(nq=16, ng=100, nid=5, d=8, metric='euclidean', k1=7, k2=3, lam=0.3, quantise=True),
    }
    for name, c in cases.items():
        qp, qc, gp, gc = synth.eval_labels((c['nq'], c['ng'], c['nid'], 3), seed=31)
        qf, gf = synth.eval_features(qp, gp, c['d'], seed=32, clustered=True)
        if c.get('quantise'):
            qf, gf = torch.round(qf), torch.round(gf)                  # integer features -> many exact distance ties
        qg = ref_metrics.compute_distance_matrix(qf, gf, c['metric']).numpy()
        qq = ref_metrics.compute_distance_matrix(qf, qf, c['metric']).numpy()
        gg = ref_metrics.compute_distance_matrix(gf, gf, c['metric']).numpy()
        with orank.stable_argsort():
            out = ref_re_ranking(qg, qq, gg, k1=c['k1'], k2=c['k2'], lambda_value=c['lam'])
        assert out.shape == (c['nq'], c['ng']) and out.dtype == np.float32
        np.savez_compressed(os.path.join(HERE, 'rerank_%s.npz' % name), q_g=qg, q_q=qq, g_g=gg, out=out,
                            k1=np.int64(c['k1']), k2=np.int64(c['k2']), lam=np.float64(c['lam']))
        print('rerank_%s' % name, out.shape, float(out.min()), float(out.max()))


if __name__ == '__main__' and ('rerank' in sys.argv[1:] or not sys.argv[1:]):
    make_rerank()


# ------------------------------------------------------------------------------- rank_cy on dataset shapes
def make_rank_cy_fresh():
    """The reference's compiled rank_cy (numpy.argsort forced stable) on the dataset-shaped inputs of
    tests/test_oracle_rank.py::test_port_vs_compiled_reference_rank_cy: cmc and mAP per case, and a checksum of the
    inputs (they are regenerated from their seeds, not stored)."""
    sys.path.insert(0, os.path.dirname(HERE))
    from test_oracle_rank import FRESH_CY, FRESH_CY_CASES, fresh_cy_inputs
    out = {}
    for case in FRESH_CY_CASES:
        key, d, qp, qc, gp, gc, checksum = fresh_cy_inputs(*case)
        cmc, mAP = orank.reference_evaluate_cy(d, qp, gp, qc, gc, 50)
        out[key + '_cmc'], out[key + '_mAP'], out[key + '_checksum'] = np.asarray(cmc), np.float64(mAP), checksum
        assert out[key + '_cmc'].dtype == np.float32
    np.savez_compressed(os.path.join(HERE, FRESH_CY), **out)
    print(FRESH_CY, sorted(out))


if __name__ == '__main__' and ('rank_cy' in sys.argv[1:] or not sys.argv[1:]):
    make_rank_cy_fresh()
