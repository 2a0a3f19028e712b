"""The numpy extraction oracle against the committed golden vectors produced by the reference's own code."""
import os

import numpy as np
import pytest

from oracle import extract_np
from tests.helpers import GOLDEN, KEYS, injected_sampler, load_random_cases, reference_case_tag


def test_toy_appendix_b():
    z = np.load(os.path.join(GOLDEN, "toy_appendix_b.npz"))
    import scipy.sparse as ssp
    g = extract_np.RatingCSR(ssp.csr_matrix(z["M"]))
    for h in (1, 2):
        sub = extract_np.extract_subgraph(g, 0, 0, h=h)
        for k in KEYS:
            assert np.array_equal(sub[k], z["h%d_%s" % (h, k)]), (h, k)
        d = extract_np.construct_graph(sub, 5.0, h)
        assert np.array_equal(d["edge_index"], z["h%d_edge_index" % h])
        assert np.array_equal(d["edge_type"], z["h%d_edge_type" % h])
        assert np.array_equal(d["x"], z["h%d_x" % h])
    # literal known answers of SURVEY.md Appendix B (h=1)
    sub = extract_np.extract_subgraph(g, 0, 0, h=1)
    assert sub["u"].tolist() == [0, 0, 1, 1, 2, 2, 2]
    assert sub["v"].tolist() == [4, 5, 3, 5, 3, 4, 5]
    assert sub["r"].tolist() == [2, 0, 3, 0, 0, 0, 4]
    assert sub["node_labels"].tolist() == [0, 2, 2, 1, 3, 3]


@pytest.mark.parametrize("group", load_random_cases(), ids=lambda g: g["tag"])
def test_golden_random(group):
    g = extract_np.RatingCSR(group["A"])
    pu, pv, pl = group["pairs"]
    for c, case in enumerate(group["cases"]):
        sub = extract_np.extract_subgraph(g, pu[c], pv[c], group["h"], group["ratio"], group["mnph"],
                                          sampler=injected_sampler(case))
        for k in KEYS:
            assert np.array_equal(sub[k], case[k]), (group["tag"], c, k)
        assert case["y"] == group["cv"][pl[c]]


def test_edge_cases_present():
    """the golden set really contains the edge cases SURVEY Appendix B lists"""
    seen_empty, seen_noedge, seen_cap_equal = False, False, False
    for group in load_random_cases():
        for case in group["cases"]:
            if len(case["u_nodes"]) == 1 and len(case["v_nodes"]) == 1:
                seen_empty = True
            if len(case["u"]) == 0:
                seen_noedge = True
    assert seen_empty and seen_noedge


def test_mnph_strict_less():
    """a fringe of exactly mnph nodes is NOT sampled (reference util_functions.py:226,228)"""
    import scipy.sparse as ssp
    M = np.zeros((4, 6), np.float32)
    M[0, :5] = 1
    M[1:, 0] = 2
    g = extract_np.RatingCSR(ssp.csr_matrix(M))
    called = []
    sub = extract_np.extract_subgraph(g, 0, 0, 1, 1.0, 4, sampler=lambda c, k, s, h: called.append((s, k)) or c[:k])
    assert called == [(1, 4)] or called == []  # only the item side (4 < 4 is false -> no call at all)
    sub = extract_np.extract_subgraph(g, 0, 0, 1, 1.0, 3, sampler=lambda c, k, s, h: called.append((s, k)) or c[:k])
    assert (1, 3) in called


def test_hash_sampler_uniform():
    """chi-square of the counter-hash sampler: each candidate picked with prob k/n"""
    n, k, trials = 40, 10, 4000
    cands = np.arange(100, 100 + n)
    cnt = np.zeros(n)
    for t in range(trials):
        sel = extract_np.hash_sample(cands, k, seed=12345, pair_id=t, side=0, hop=1)
        assert len(sel) == k and len(set(sel.tolist())) == k
        cnt[sel - 100] += 1
    exp = trials * k / n
    chi2 = ((cnt - exp) ** 2 / (exp * (1 - k / n))).sum()
    assert chi2 < 80.0, chi2  # 39 dof, p ~ 1e-4 at 80


@pytest.mark.parametrize("h,mnph", [(1, None), (1, 6), (2, None), (2, 3)])
def test_live_reference(h, mnph):
    """40 pairs of a seeded 50x45 matrix: the oracle against the reference's own extraction of the same pairs
    (stored in tests/golden/reference_cases.npz by tests/golden/make_golden.py), the reference's draw injected"""
    from igmc_b200.data import build_adj
    z = np.load(os.path.join(GOLDEN, "reference_cases.npz"))
    tag = reference_case_tag(h, mnph)
    u, v, lab = z[tag + "__coo"]
    A = build_adj(u, v, lab, 50, 45)
    g = extract_np.RatingCSR(A)
    for c in range(40):
        canon = {k: z["%s__%s" % (tag, k)][z["%s__%s_off" % (tag, k)][c]:z["%s__%s_off" % (tag, k)][c + 1]]
                 for k in KEYS}
        canon["y"] = float(z[tag + "__y"][c])
        sub = extract_np.extract_subgraph(g, u[c], v[c], h, 1.0, mnph, sampler=injected_sampler(canon))
        for k in KEYS:
            assert np.array_equal(sub[k], canon[k]), (c, k)
        # PyG-layout arrays: same multiset of (src, dst, type) after relabelling is implied by the
        # canonical equality above; check sizes and x one-hot
        d = extract_np.construct_graph(sub, canon["y"], h)
        assert tuple(z[tag + "__x_shape"][c]) == d["x"].shape
        assert z[tag + "__n_edges"][c] == d["edge_index"].shape[1]
        # the label of the reference's PyG Data, stored apart from the extraction's y that construct_graph was given
        assert z[tag + "__data_y"][c] == d["y"][0]


def test_flixster_real_data_golden():
    """REAL flixster ratings (fixture built from the reference's raw_data by tests/golden/make_flixster_fixture.py):
    the oracle reproduces what the reference's own extraction returned for 64 pairs (40 train incl. the target-edge
    removal, 24 test), RNG-free because max_nodes_per_hop=10000 exceeds every degree."""
    from tests.helpers import load_flixster_cases
    ds, pairs, cases = load_flixster_cases()
    assert ds["adj_train"].shape == (3000, 3000) and ds["adj_train"].nnz == 23556 and ds["num_relations"] == 10
    assert len(ds["test"][0]) == 2617
    g = extract_np.RatingCSR(ds["adj_train"])
    for c, want in enumerate(cases):
        sub = extract_np.extract_subgraph(g, pairs[0, c], pairs[1, c], 1, 1.0, 10000)
        for k in ("u_nodes", "v_nodes", "u", "v", "r", "node_labels"):
            assert np.array_equal(np.asarray(sub[k], np.int64), want[k]), (c, k)
        assert float(ds["class_values"][pairs[2, c]]) == want["y"]
