"""oracle/qe.py against a literal float32 transcription of FastReID's ``aqe`` (fastreid/evaluation/query_expansion.py),
on inputs whose margin (each row's k-th minus (k+1)-th similarity) exceeds 1e-4 at every iteration, so that
np.argpartition picks the same neighbours as the oracle's stable order."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import qe as oqe


def fastreid_aqe(query_feat, gallery_feat, qe_times=1, qe_k=10, alpha=3.0):
    """fastreid/evaluation/query_expansion.py, as it is written there"""
    num_query = query_feat.shape[0]
    all_feat = torch.cat((query_feat, gallery_feat), dim=0)
    norm_feat = F.normalize(all_feat, p=2, dim=1)
    all_feat = all_feat.numpy()
    for i in range(qe_times):
        all_feat_list = []
        sims = torch.mm(norm_feat, norm_feat.t()).data.cpu().numpy()
        for sim in sims:
            init_rank = np.argpartition(-sim, range(1, qe_k + 1))
            weights = np.power(sim[init_rank[:qe_k]].reshape((-1, 1)), alpha)
            all_feat_list.append(np.mean(all_feat[init_rank[:qe_k], :] * weights, axis=0))
        all_feat = np.stack(all_feat_list, axis=0)
        norm_feat = F.normalize(torch.from_numpy(all_feat), p=2, dim=1)
    return torch.from_numpy(all_feat[:num_query]), torch.from_numpy(all_feat[num_query:])


def near(got, ref, tol=1e-5):
    """every row within tol of the reference, relative to the reference row's norm"""
    err = np.abs(got - ref).max(axis=1)
    scale = np.maximum(np.linalg.norm(ref, axis=1), 1e-30)
    return float((err / scale).max())


@pytest.mark.parametrize('qe_times', [1, 2, 3])
@pytest.mark.parametrize('alpha', [0.0, 1.0, 3.0, 0.5])
@pytest.mark.parametrize('shape', [(12, 48, 16, 5, 0.3), (7, 23, 9, 3, 0.3), (30, 90, 64, 10, 0.5)])
def test_oracle_equals_fastreid(qe_times, alpha, shape):
    nq, ng, dim, k, spread = shape              # (7, 23, 9, 3): lists that cross the groups
    qf, gf = oqe.grouped_features(nq, ng, dim, k, seed=nq + k, spread=spread)
    q, g, lists, sims, margins = oqe.aqe(qf, gf, k, qe_times, alpha)
    assert len(lists) == qe_times
    for m in margins:
        assert m.min() > 1e-4, m.min()
    rq, rg = fastreid_aqe(qf, gf, qe_times, k, alpha)
    assert near(rq.numpy(), q) < 1e-5 and near(rg.numpy(), g) < 1e-5


def test_lists_are_stable_and_include_the_row_itself():
    x = torch.tensor([[1., 0.], [1., 0.], [0., 1.], [2., 0.], [0., 3.], [1., 1.]])
    _, _, lists, sims, margins = oqe.aqe(x[:2], x[2:], 3, 1, 3.0)
    # rows 0, 1 and 3 are the same direction: every list of one of them is [0, 1, 3] (ties to the lower index)
    for r in (0, 1, 3):
        assert lists[0][r].tolist() == [0, 1, 3] and margins[0][r] > 0.29
    assert lists[0][2].tolist() == [2, 4, 5]
    assert np.allclose(sims[0][5], [1.0, np.sqrt(0.5), np.sqrt(0.5)])
    assert lists[0][5].tolist() == [5, 0, 1]                  # a tie of four at 1/sqrt(2): the two lowest indices


def test_mean_expansion_and_negative_similarity():
    x = torch.tensor([[1., 0.], [-1., 0.1], [0., 1.]])
    q, g, lists, sims, _ = oqe.aqe(x[:1], x[1:], 3, 1, 0.0)
    assert np.allclose(np.concatenate([q, g]), x.double().mean(0).numpy())      # alpha 0: plain mean of all three
    q, g, _, sims, _ = oqe.aqe(x[:1], x[1:], 3, 1, 0.5)
    neg = (sims[0] < 0).any(axis=1)                                            # np.power(negative, 0.5) = NaN
    assert neg.tolist() == [True, True, False]
    assert np.array_equal(np.isnan(np.concatenate([q, g])).all(axis=1), neg)
    q, g, _, _, margins = oqe.aqe(x[:1], x[1:], 3, 1, 3.0)
    assert np.isfinite(np.concatenate([q, g])).all() and np.isinf(margins[0]).all()   # N == k: no (k+1)-th
