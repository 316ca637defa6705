"""bindsnet_b200.evaluation against the reference's evaluation functions (evaluation/evaluation.py:8-61,
99-180; their results stored under tests/golden/live) on the CPU, from rasters and from the per-sample counts the window
kernels deliver."""
import importlib

import torch

from live import REF, stored


def ref_eval():
    return importlib.import_module("bindsnet.evaluation.evaluation")   # needs sklearn


def test_label_assignment_and_readout_match_the_reference():
    from bindsnet_b200 import evaluation as ev

    g = torch.Generator().manual_seed(3)
    S, T, n, L = 60, 30, 50, 10
    spikes = (torch.rand(S, T, n, generator=g) < 0.1 * torch.rand(1, 1, n, generator=g) + 0.02).byte()
    labels = torch.randint(0, L - 1, (S,), generator=g)            # the last class never occurs (n_labeled == 0 branch)
    a_ref, p_ref, r_ref = stored("assign_labels", lambda: ref_eval().assign_labels(spikes.float(), labels, L))
    a, p, r = ev.assign_labels(spikes, labels, L)
    assert torch.equal(a, a_ref) and torch.allclose(p, p_ref, atol=1e-6) and torch.allclose(r, r_ref, atol=1e-6)
    # from counts (what SpikeCounter hands over), second batch with the running rates and alpha
    spikes2 = (torch.rand(S, T, n, generator=g) < 0.08).byte()
    a_ref2, p_ref2, r_ref2 = stored("assign_labels/rates", lambda: ref_eval().assign_labels(spikes2.float(), labels, L, rates=r_ref.clone(), alpha=0.9))
    a2, p2, r2 = ev.assign_labels(spikes2.sum(1).int(), labels, L, rates=r.clone(), alpha=0.9)
    assert torch.equal(a2, a_ref2) and torch.allclose(p2, p_ref2, atol=1e-6) and torch.allclose(r2, r_ref2, atol=1e-6)
    assert torch.equal(ev.all_activity(spikes2.sum(1).int(), a2, L), stored("all_activity", lambda: ref_eval().all_activity(spikes2.float(), a_ref2, L)))
    assert torch.equal(ev.proportion_weighting(spikes2, a2, p2, L),
                       stored("proportion_weighting", lambda: ref_eval().proportion_weighting(spikes2.float(), a_ref2, p_ref2, L)))


def test_ngram_scores_and_predictions_match_the_reference():
    """evaluation.py:183-258: dictionaries of per-class counts keyed by firing sequences, and the class read from them."""
    from bindsnet_b200 import evaluation as ev

    g = torch.Generator().manual_seed(12)
    S, T, n_neurons, L = 14, 12, 9, 4
    spikes = (torch.rand(S, T, n_neurons, generator=g) < 0.12).byte()
    spikes[3] = 0                                                    # a silent example
    labels = torch.randint(0, L, (S,), generator=g)
    for n in (2, 3):
        a = stored(f"update_ngram_scores/{n}", lambda: ref_eval().update_ngram_scores(spikes, labels, L, n, {}))
        b = ev.update_ngram_scores(spikes, labels, L, n, {})
        assert sorted(a) == sorted(b) and len(a) > 10
        assert all(torch.equal(a[k], b[k]) for k in a)
        # second batch accumulates into the same dictionary
        more = (torch.rand(S, T, n_neurons, generator=g) < 0.1).byte()
        a = stored(f"update_ngram_scores/{n}/more", lambda: ref_eval().update_ngram_scores(more, labels, L, n, a))
        b = ev.update_ngram_scores(more, labels, L, n, b)
        assert sorted(a) == sorted(b) and all(torch.equal(a[k], b[k]) for k in a)
        pa, pb = stored(f"ngram/{n}", lambda: ref_eval().ngram(spikes, a, L, n)), ev.ngram(spikes, b, L, n)
        assert pa.dtype == pb.dtype and torch.equal(pa, pb)
        assert len(set(pb.tolist())) > 1


def test_logreg_wrappers_match_the_reference():
    from sklearn.linear_model import LogisticRegression

    from bindsnet_b200 import evaluation as ev

    g = torch.Generator().manual_seed(13)
    labels = torch.randint(0, 3, (40,), generator=g)
    x = torch.rand(40, 6, generator=g) + torch.nn.functional.one_hot(labels, 6).float() * 2.0
    fresh = LogisticRegression(max_iter=200)
    assert torch.equal(ev.logreg_predict(x, fresh), stored("logreg_predict/fresh", lambda: ref_eval().logreg_predict(x, fresh)))
    assert int(ev.logreg_predict(x, fresh)[0]) == -1
    b = ev.logreg_fit(x, labels, LogisticRegression(max_iter=200))
    pa = stored("logreg_predict", lambda: ref_eval().logreg_predict(x, ref_eval().logreg_fit(x, labels, LogisticRegression(max_iter=200))))
    pb = ev.logreg_predict(x, b)
    assert pa.dtype == pb.dtype and torch.equal(pa, pb) and float((pb == labels).float().mean()) > 0.9
