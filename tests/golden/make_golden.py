"""Generate tests/golden/*.npz from the UNMODIFIED reference extraction code.

Needs the reference's code: oracle/_ref/ as build() leaves it, or ``IGMC_REFERENCE_DIR`` naming a checkout
(``oracle/ref_shim.py``):

    python tests/golden/make_golden.py

Every vector is produced by the reference's own ``subgraph_extraction_labeling`` +
``construct_pyg_graph`` (util_functions.py:208-297) through ``oracle/ref_shim.py``
(PyG stubbed, ``random.sample`` made set-tolerant) and relabelled into canonical
form (SURVEY.md §8c).  For sampled cases the reference's own draw is recorded as
the per-graph node lists, so the GPU/oracle paths can be checked with the fringe
injected.
"""
import os
import random
import sys

import numpy as np
import scipy.sparse as ssp

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))

from oracle import ref_shim  # noqa: E402
from igmc_b200.data import synth_ratings, build_adj  # noqa: E402
from tests.helpers import reference_case_tag  # noqa: E402

KEYS = ("u_nodes", "v_nodes", "u", "v", "r", "node_labels")


def pack(cases):
    """list of canonical dicts -> flat arrays + offsets (npz friendly)."""
    out = {}
    for k in KEYS:
        out[k] = np.concatenate([np.asarray(c[k], np.int64) for c in cases]) if cases else np.zeros(0, np.int64)
        out[k + "_off"] = np.cumsum([0] + [len(c[k]) for c in cases]).astype(np.int64)
    out["y"] = np.array([c["y"] for c in cases], np.float64)
    return out


def run_cases(A, pairs_u, pairs_v, labels, cv, h, ratio, mnph, seed):
    idx = ref_shim.make_indexers(A)
    random.seed(seed)
    cases = []
    for i, j, l in zip(pairs_u, pairs_v, labels):
        canon, raw = ref_shim.extract_ref_canonical(A, int(i), int(j), int(l), cv, h, ratio, mnph, idx)
        # the PyG Data built by the reference must agree with the canonical arrays up to order
        data = raw[-1]
        assert data.edge_index.shape[1] == 2 * len(canon["u"])
        cases.append(canon)
    return cases


def main():
    # ---- 1. SURVEY Appendix B toy matrix -------------------------------------------
    M = np.array([[5, 3, 0, 1], [4, 0, 0, 1], [1, 1, 0, 5], [0, 0, 5, 4], [0, 1, 5, 4]], np.float32)
    A = ssp.csr_matrix(M)
    cv = np.array([1, 2, 3, 4, 5], np.float64)
    toy = {}
    for h in (1, 2):
        c, raw = ref_shim.extract_ref_canonical(A, 0, 0, 4, cv, h)
        for k in KEYS:
            toy["h%d_%s" % (h, k)] = np.asarray(c[k], np.int64)
        toy["h%d_y" % h] = np.float64(c["y"])
        d = raw[-1]
        toy["h%d_edge_index" % h] = d.edge_index.numpy()
        toy["h%d_edge_type" % h] = d.edge_type.numpy()
        toy["h%d_x" % h] = d.x.numpy()
    toy["M"] = M
    np.savez_compressed(os.path.join(HERE, "toy_appendix_b.npz"), **toy)

    # ---- 2. seeded random matrices: edge cases + sampling ---------------------------
    rnd = {}
    specs = [
        # tag, users, items, nnz, R, h, ratio, mnph
        ("a_h1", 40, 30, 300, 5, 1, 1.0, None),
        ("a_h1_m5", 40, 30, 300, 5, 1, 1.0, 5),
        ("a_h2", 40, 30, 120, 5, 2, 1.0, None),
        ("a_h2_m4", 40, 30, 120, 5, 2, 1.0, 4),
        ("b_h1_r10", 70, 90, 500, 10, 1, 1.0, None),
        ("b_h1_ratio", 70, 90, 500, 10, 1, 0.5, None),
        ("c_h1_m20", 200, 150, 6000, 5, 1, 1.0, 20),
        ("c_h3", 30, 30, 60, 3, 3, 1.0, None),
    ]
    for tag, nu, nv, nnz, R, h, ratio, mnph in specs:
        seed = abs(hash(tag)) % 1000 if False else sum(map(ord, tag))
        u, v, lab = synth_ratings(nu, nv, nnz, R, seed)
        A = build_adj(u, v, lab, nu, nv)
        cvv = np.arange(1, R + 1, dtype=np.float64) * 0.5
        rng = np.random.default_rng(seed + 7)
        # pairs: 24 train pairs (in the matrix) + 8 pairs NOT in the matrix + degenerate ones
        pick = rng.choice(nnz, 24, replace=False)
        pu, pv, pl = list(u[pick]), list(v[pick]), list(lab[pick])
        dense = A.toarray()
        cnt = 0
        while cnt < 8:
            i, j = int(rng.integers(nu)), int(rng.integers(nv))
            if dense[i, j] == 0:
                pu.append(i); pv.append(j); pl.append(int(rng.integers(R))); cnt += 1
        # a user with an empty row / an item with an empty column if any exist
        er = np.where(np.diff(A.indptr) == 0)[0]
        ec = np.where(np.diff(A.tocsc().indptr) == 0)[0]
        if len(er) and len(ec):
            pu.append(int(er[0])); pv.append(int(ec[0])); pl.append(0)
        if len(er):
            pu.append(int(er[0])); pv.append(int(v[0])); pl.append(1)
        if len(ec):
            pu.append(int(u[0])); pv.append(int(ec[0])); pl.append(2)
        cases = run_cases(A, pu, pv, pl, cvv, h, ratio, mnph, seed)
        P = pack(cases)
        for k, val in P.items():
            rnd["%s__%s" % (tag, k)] = val
        rnd[tag + "__coo_u"], rnd[tag + "__coo_v"], rnd[tag + "__coo_l"] = u, v, lab
        rnd[tag + "__shape"] = np.array([nu, nv, R, h, -1 if mnph is None else mnph], np.int64)
        rnd[tag + "__ratio"] = np.float64(ratio)
        rnd[tag + "__pairs"] = np.array([pu, pv, pl], np.int64)
        rnd[tag + "__cv"] = cvv
    rnd["tags"] = np.array([s[0] for s in specs])
    np.savez_compressed(os.path.join(HERE, "random_cases.npz"), **rnd)
    write_live_cases()
    print("wrote", os.listdir(HERE))


def write_live_cases():
    """reference_cases.npz: 40 pairs per (h, mnph) of tests/test_oracle_extract.py::test_live_reference, with the
    reference's canonical subgraphs and the shapes / label of the PyG Data it built."""
    out = {}
    for h, mnph in LIVE_SPECS:
        tag = reference_case_tag(h, mnph)
        u, v, lab = synth_ratings(50, 45, 420, 5, seed=99 + h)
        A = build_adj(u, v, lab, 50, 45)
        cv = np.array([1, 2, 3, 4, 5.0])
        idx = ref_shim.make_indexers(A)
        random.seed(5)
        cases, x_shape, n_edges, y = [], [], [], []
        for c in range(40):
            canon, raw = ref_shim.extract_ref_canonical(A, int(u[c]), int(v[c]), int(lab[c]), cv, h, 1.0, mnph, idx)
            data = raw[-1]
            cases.append(canon)
            x_shape.append(tuple(data.x.shape))
            n_edges.append(data.edge_index.shape[1])
            y.append(float(data.y))      # the label as the reference's PyG Data carries it
        for k, val in pack(cases).items():
            out["%s__%s" % (tag, k)] = val
        out[tag + "__coo"] = np.array([u, v, lab], np.int64)
        out[tag + "__x_shape"] = np.array(x_shape, np.int64)
        out[tag + "__n_edges"] = np.array(n_edges, np.int64)
        out[tag + "__data_y"] = np.array(y, np.float64)
    np.savez_compressed(os.path.join(HERE, "reference_cases.npz"), **out)


LIVE_SPECS = ((1, None), (1, 6), (2, None), (2, 3))


if __name__ == "__main__":
    main()
