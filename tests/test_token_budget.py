"""CPU: the token-budget rule of oracle/token_budget.py and the drop-in's validation of model.token_budget."""
import numpy as np
import pytest
import torch

from oracle import token_budget as TB

P = 196


def brute_force_mask(s, k, mode, mt):
    """Python's stable sort: descending score, NaN after every number, ties (and NaNs) by token index."""
    order = sorted(range(len(s)), key=lambda t: (1, 0.0) if np.isnan(s[t]) else (0, -float(s[t])))
    top = set(order[:k])
    keep = [t in top and (mode == "exact" or (not np.isnan(s[t]) and s[t] >= np.float32(mt))) for t in range(len(s))]
    return np.array([True] + keep)


def quantised_scores(rng, B, levels=16, nan_frac=0.0):
    s = (rng.integers(0, levels, size=(B, P)) / levels).astype(np.float32)
    if nan_frac:
        s[rng.random((B, P)) < nan_frac] = np.nan
    return s


@pytest.mark.parametrize("mode", TB.MODES)
@pytest.mark.parametrize("levels, nan_frac", [(8, 0.0), (64, 0.0), (1 << 20, 0.0), (16, 0.1)])
def test_rule_matches_stable_sort(mode, levels, nan_frac):
    rng = np.random.default_rng(levels + int(nan_frac * 100))
    s = quantised_scores(rng, 6, levels, nan_frac)
    for k in (0, 1, 13, 49, 98, 195, 196):
        got = TB.budget_mask(s, k, mode, 0.5)
        for b in range(s.shape[0]):
            assert np.array_equal(got[b], brute_force_mask(s[b], k, mode, 0.5)), (mode, levels, k, b)


def test_ranks_are_a_permutation_with_ties_to_the_lower_index():
    s = np.full((1, P), 0.25, dtype=np.float32)
    assert np.array_equal(TB.ranks(s)[0], np.arange(P))
    s[0, 100] = 0.75
    r = TB.ranks(s)[0]
    assert r[100] == 0 and r[0] == 1 and r[99] == 100 and r[101] == 101
    rng = np.random.default_rng(0)
    s = quantised_scores(rng, 4, 4, 0.2)
    for row in TB.ranks(s):
        assert sorted(row) == list(range(P))


def test_edge_budgets():
    rng = np.random.default_rng(1)
    s = rng.random((5, P), dtype=np.float32)
    cls_only = TB.budget_mask(s, 0, "exact")
    assert cls_only[:, 0].all() and not cls_only[:, 1:].any()
    assert TB.budget_mask(s, P, "exact").all()                  # k = N-1 keeps everything
    assert np.array_equal(TB.budget_mask(s, P, "cap", 0.5)[:, 1:], s >= 0.5)
    assert (TB.budget_mask(s, 49, "exact").sum(1) == 50).all()


@pytest.mark.parametrize("k", [0, 10, 64, 150, 196])
def test_cap_is_the_top_of_the_threshold_set(k):
    rng = np.random.default_rng(k)
    s = quantised_scores(rng, 8, 32)
    thr = s >= 0.5
    cap = TB.budget_mask(s, k, "cap", 0.5)[:, 1:]
    assert not (cap & ~thr).any()                                # CAP is a subset of the threshold set
    assert np.array_equal(cap.sum(1), np.minimum(k, thr.sum(1)))
    for b in range(s.shape[0]):                                   # ... made of its highest scores
        if cap[b].any() and (thr[b] & ~cap[b]).any():
            assert s[b][cap[b]].min() >= s[b][thr[b] & ~cap[b]].max()


def test_nan_ordering():
    s = np.linspace(0.9, 0.1, P).astype(np.float32)[None].copy()
    s[0, [3, 7, 50]] = np.nan
    r = TB.ranks(s)[0]
    assert list(r[[3, 7, 50]]) == [P - 3, P - 2, P - 1]         # below every number, by index
    exact = TB.budget_mask(s, P - 1, "exact")[0, 1:]
    assert not exact[50] and exact[3] and exact[7]
    assert not TB.budget_mask(s, P, "cap", 0.0)[0, 1:][[3, 7, 50]].any()   # NaN never passes the threshold


def test_near_cut_flags_close_kth_scores():
    s = np.linspace(0.9, 0.1, P).astype(np.float32)[None].repeat(2, 0)
    s[1, 10] = s[1, 9] + 5e-5
    s[1, 9], s[1, 10] = s[1, 10], s[1, 9]
    near = TB.near_cut(s, 10, "exact")
    assert not near[0] and near[1]


def _model():
    import model_utils
    from transformers.models.vit.modeling_vit import ViTConfig
    cfg = ViTConfig(hidden_size=384, num_attention_heads=6, intermediate_size=1536, num_hidden_layers=12)
    cfg.num_labels = 10
    return model_utils.ModifiedViTModel(cfg, 0.9, 0.5, 0)


@pytest.mark.parametrize("budget, mode", [
    (-1, "exact"), (197, "exact"), (1.5, "exact"), (True, "exact"), ("49", "exact"),
    ([49] * 11, "exact"), ([49] * 11 + [197], "cap"), (49, "topk"),
])
def test_drop_in_rejects_malformed_budgets(budget, mode):
    model = _model()
    model.token_budget, model.token_budget_mode = budget, mode
    with pytest.raises(ValueError):
        model(torch.zeros(1, 3, 224, 224))


def test_drop_in_budget_setting():
    model = _model()
    assert model._token_budget_setting() is None
    model.token_budget = 49
    assert model._token_budget_setting() == ("exact", (49,) * 12)
    model.token_budget, model.token_budget_mode = [0] * 6 + [196] * 6, "cap"
    assert model._token_budget_setting() == ("cap", (0,) * 6 + (196,) * 6)
    model.token_budget = np.array([3] * 12).tolist()
    assert model._token_budget_setting() == ("cap", (3,) * 12)
