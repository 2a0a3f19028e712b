"""Import the UNMODIFIED reference extraction code (container only).

/root/reference/util_functions.py needs ``torch_geometric.data`` (line 13) for
three class names only; we register a stub module before importing it.  On
Python >= 3.11 ``random.sample`` refuses sets (reference line 223-229 passes
sets), so calls are wrapped to pass ``tuple(population)`` which is what
CPython <= 3.10 did internally.  Nothing else is changed.

This module is used by the generators under ``tests/golden/`` (which store
the reference's outputs for the tests) and by the CPU arm of ``bench.py``.
"""
import importlib.util
import os
import random
import sys
import types

# the copy build() places under oracle/_ref/ (oracle/make_ref.py); without it, a reference checkout named by
# IGMC_REFERENCE_DIR (for the golden-data generators run before a build)
_VENDORED = os.path.join(os.path.dirname(os.path.abspath(__file__)), "_ref")
REF_DIR = _VENDORED
if not os.path.isfile(os.path.join(_VENDORED, "util_functions.py")) and os.environ.get("IGMC_REFERENCE_DIR"):
    REF_DIR = os.environ["IGMC_REFERENCE_DIR"]


def available():
    return os.path.isfile(os.path.join(REF_DIR, "util_functions.py"))


def _install_pyg_stub():
    if "torch_geometric" in sys.modules:
        return
    tg = types.ModuleType("torch_geometric")
    tgd = types.ModuleType("torch_geometric.data")

    class Data(object):
        def __init__(self, x=None, edge_index=None, edge_type=None, y=None, **kw):
            self.x, self.edge_index, self.edge_type, self.y = x, edge_index, edge_type, y
            for k, v in kw.items():
                setattr(self, k, v)

        @property
        def num_nodes(self):
            return self.x.size(0)

    class Dataset(object):
        def __init__(self, root=None, *a, **kw):
            self.root = root

    class InMemoryDataset(Dataset):
        pass

    tgd.Data, tgd.Dataset, tgd.InMemoryDataset = Data, Dataset, InMemoryDataset
    tg.data = tgd
    sys.modules["torch_geometric"] = tg
    sys.modules["torch_geometric.data"] = tgd


_ref = None


def load():
    """Return the reference ``util_functions`` module object."""
    global _ref
    if _ref is not None:
        return _ref
    if not available():
        raise RuntimeError("reference checkout not present at %s" % REF_DIR)
    _install_pyg_stub()
    spec = importlib.util.spec_from_file_location(
        "_igmc_reference_util_functions", os.path.join(REF_DIR, "util_functions.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)

    class _Random(object):
        """``random`` facade whose sample() accepts sets (py<=3.10 behaviour)."""

        def __getattr__(self, name):
            return getattr(random, name)

        @staticmethod
        def sample(population, k):
            if isinstance(population, (set, frozenset)):
                population = tuple(population)
            return random.sample(population, k)

    mod.random = _Random()
    _ref = mod
    return mod


def extract_ref(A_csr, i, j, label, class_values, h=1, sample_ratio=1.0, max_nodes_per_hop=None,
                indexers=None):
    """Run the reference's own extraction + graph construction for one pair.

    Returns the raw reference outputs as numpy/torch objects:
    (u, v, r, node_labels, max_node_label, y, data) where ``data`` is the
    ``construct_pyg_graph`` result.  ``indexers`` may carry (Arow, Acol) to
    avoid rebuilding them per call.
    """
    m = load()
    if indexers is None:
        indexers = (m.SparseRowIndexer(A_csr), m.SparseColIndexer(A_csr.tocsc()))
    Arow, Acol = indexers
    out = m.subgraph_extraction_labeling((i, j), Arow, Acol, h, sample_ratio, max_nodes_per_hop,
                                         None, None, class_values, label)
    data = m.construct_pyg_graph(*out)
    return out + (data,)


def make_indexers(A_csr):
    m = load()
    return m.SparseRowIndexer(A_csr), m.SparseColIndexer(A_csr.tocsc())


class _RecordingMatrix(object):
    """Wraps the csr returned by ``Arow[u_nodes]`` to see the ``[:, v_nodes]`` key."""

    def __init__(self, mat, log):
        self._mat, self._log = mat, log

    @property
    def indices(self):
        return self._mat.indices

    def __getitem__(self, key):
        if isinstance(key, tuple) and len(key) == 2:
            self._log["v_nodes"] = list(key[1])
        return self._mat[key]


class _RecordingRows(object):
    """Wraps the reference's SparseRowIndexer: records the row selector of every call
    (the last one is ``u_nodes``, reference util_functions.py:236)."""

    def __init__(self, inner, log):
        self._inner, self._log, self.shape = inner, log, inner.shape

    def __getitem__(self, rows):
        self._log["u_nodes"] = list(rows)
        return _RecordingMatrix(self._inner[rows], self._log)


def extract_ref_canonical(A_csr, i, j, label, class_values, h=1, sample_ratio=1.0,
                          max_nodes_per_hop=None, indexers=None):
    """Reference extraction of one pair, relabelled into canonical form.

    The reference function is called unmodified; only the indexer argument is a
    recording proxy so that we learn its (set-ordered) ``u_nodes``/``v_nodes``.
    Returns (canonical dict, raw reference tuple incl. Data).
    """
    from . import extract_np
    m = load()
    if indexers is None:
        indexers = make_indexers(A_csr)
    log = {}
    Arow = _RecordingRows(indexers[0], log)
    out = m.subgraph_extraction_labeling((i, j), Arow, indexers[1], h, sample_ratio,
                                         max_nodes_per_hop, None, None, class_values, label)
    u, v, r, node_labels, max_node_label, y, feats = out
    canon = extract_np.canonicalize_reference(u, v, r, node_labels, log["u_nodes"], log["v_nodes"])
    canon["y"] = float(y)
    canon["max_node_label"] = int(max_node_label)
    data = m.construct_pyg_graph(*out)
    return canon, out + (data,)
