"""Shared loaders for tests/golden."""
import os

import numpy as np

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
KEYS = ("u_nodes", "v_nodes", "u", "v", "r", "node_labels")


def load_random_cases():
    """Yield dict(tag, A (scipy csr), pairs, cv, h, ratio, mnph, cases=[canonical dicts])."""
    from igmc_b200.data import build_adj
    z = np.load(os.path.join(GOLDEN, "random_cases.npz"))
    out = []
    for tag in z["tags"]:
        tag = str(tag)
        nu, nv, R, h, mnph = [int(x) for x in z[tag + "__shape"]]
        A = build_adj(z[tag + "__coo_u"], z[tag + "__coo_v"], z[tag + "__coo_l"], nu, nv)
        n = z[tag + "__pairs"].shape[1]
        cases = []
        for c in range(n):
            d = {}
            for k in KEYS:
                off = z["%s__%s_off" % (tag, k)]
                d[k] = z["%s__%s" % (tag, k)][off[c]:off[c + 1]]
            d["y"] = float(z[tag + "__y"][c])
            cases.append(d)
        out.append(dict(tag=tag, A=A, pairs=z[tag + "__pairs"], cv=z[tag + "__cv"], h=h,
                        ratio=float(z[tag + "__ratio"]), mnph=None if mnph < 0 else mnph,
                        R=R, cases=cases))
    return out


def injected_sampler(case):
    """sampler(cands, k, side, hop) returning the reference's recorded draw for a golden case."""
    n_u = len(case["u_nodes"])
    labels = case["node_labels"]
    ud, vd = labels[:n_u] // 2, (labels[n_u:] - 1) // 2

    def smp(cands, k, side, hop):
        nodes, dist = (case["u_nodes"], ud) if side == 0 else (case["v_nodes"], vd)
        sel = nodes[dist == hop]
        assert len(sel) == k and set(sel.tolist()) <= set(np.asarray(cands).tolist())
        return sel
    return smp


def oracle_collated(group, sampler_from_cases=True, seed=0):
    """numpy-oracle collate of every pair of a golden group (h must be 1)."""
    from oracle import extract_np
    g = extract_np.RatingCSR(group["A"])
    pu, pv, pl = group["pairs"]
    smp = None
    if sampler_from_cases:
        samplers = [injected_sampler(c) for c in group["cases"]]
        smp = lambda k, cands, kk, side, hop: samplers[k](cands, kk, side, hop)  # noqa: E731
    return extract_np.extract_batch(g, pu, pv, pl, group["cv"].astype(np.float32), group["h"], group["ratio"],
                                    group["mnph"], sampler=smp, seed=seed)


def inject_arrays(cases, cap):
    """golden canonical node lists -> padded [B,cap] int32 arrays for SubgraphExtractor.extract(inject=...)."""
    B = len(cases)
    nu = np.zeros((B, cap), np.int32)
    nv = np.zeros((B, cap), np.int32)
    cu = np.zeros(B, np.int32)
    cvv = np.zeros(B, np.int32)
    for k, c in enumerate(cases):
        cu[k], cvv[k] = len(c["u_nodes"]), len(c["v_nodes"])
        nu[k, :cu[k]] = c["u_nodes"]
        nv[k, :cvv[k]] = c["v_nodes"]
    return nu, nv, cu, cvv


def batch_equal(b, ob):
    """compare an igmc_b200 Batch with an oracle collated dict, bit-exact on every integer field."""
    import torch
    out = {}
    out["x"] = np.array_equal(b.x.cpu().numpy(), ob["x"])
    out["edge_index"] = np.array_equal(b.edge_index.cpu().numpy(), ob["edge_index"])
    out["edge_type"] = np.array_equal(b.edge_type.cpu().numpy(), ob["edge_type"])
    out["batch"] = np.array_equal(b.batch.cpu().numpy(), ob["batch"])
    out["y"] = np.array_equal(b.y.cpu().numpy(), ob["y"].astype(np.float32))
    out["node_label"] = np.array_equal(b.node_label.cpu().numpy().astype(np.int64), ob["node_labels"])
    return out


def reference_case_tag(h, mnph):
    """key prefix of one (h, max_nodes_per_hop) group in tests/golden/reference_cases.npz"""
    return "h%d_m%s" % (h, "none" if mnph is None else mnph)


def load_flixster_cases():
    """(dataset dict, pairs [3,n], list of canonical dicts) of tests/golden/flixster_cases.npz: outputs of the
    reference's own subgraph_extraction_labeling on 64 pairs of the REAL flixster split (h=1, no sampling)."""
    from igmc_b200.data import load_flixster
    ds = load_flixster()
    z = np.load(os.path.join(GOLDEN, "flixster_cases.npz"))
    cases = []
    for c in range(z["pairs"].shape[1]):
        d = {k: z[k][z[k + "_off"][c]:z[k + "_off"][c + 1]] for k in KEYS}
        d["y"] = float(z["y"][c])
        cases.append(d)
    return ds, z["pairs"], cases
