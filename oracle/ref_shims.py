"""TEST INFRASTRUCTURE — import shims that let the UNMODIFIED reference run in this container.

Only `oracle/make_golden.py`, `tests/test_oracle_vs_reference.py` and the reference arm of `bench.py`
(`--impl reference`) use this file, on the reference named by REFERENCE_ROOT below.  It never travels into the
product path.

The reference imports three packages that are absent here (SURVEY.md Appendix A):
`matplotlib` (import only), `torch_scatter` (training loss only) and `dgl` — pinned `dgl==1.1.2+cu117`
in the reference's requirements:16, not vendored.  The dgl surface the hot path touches is restated
from DGL's published semantics:

* `dgl.from_networkx(g, device=)` (python/dgl/convert.py): nodes relabelled with
  `nx.convert_node_labels_to_integers(g, ordering='sorted')`, then `to_directed()` — both directions
  of every undirected edge; the returned graph exposes `.ndata` (call sites models/agc.py:704-707,
  models/gmatcher.py:244-249, 268-269).
* `dgl.nn.SAGEConv(in, out, 'mean')` (python/dgl/nn/pytorch/conv/sageconv.py): `fc_neigh`, `fc_self`
  are `nn.Linear(bias=False)`, a separate `bias` parameter; `h_neigh` = mean of source features over
  in-edges (0 for in-degree 0); `fc_neigh` is applied BEFORE aggregation iff in_feats > out_feats;
  `rst = fc_self(h) + h_neigh + bias`.

The shim's SAGE/from_networkx restatement is itself unpinned against real DGL ("parity unpinned",
SURVEY.md §8c).
"""
import os
import sys
import types

# a checkout of songxf1024/GIMS named by GIMS_REFERENCE_ROOT, else the copy of its modules that
# __graft_entry__.install_reference() leaves in the git-ignored oracle/_ref; the repository itself does not contain it
REFERENCE_ROOT = os.environ.get('GIMS_REFERENCE_ROOT') or os.path.join(os.path.dirname(os.path.abspath(__file__)), '_ref')


def reference_available():
    return os.path.isfile(os.path.join(REFERENCE_ROOT, 'models', 'gmatcher.py'))


def _install_stubs():
    import networkx as nx
    import torch
    import torch.nn as nn

    if 'matplotlib' not in sys.modules:
        try:
            import matplotlib  # noqa: F401
            import matplotlib.pyplot  # noqa: F401
        except Exception:
            mpl = types.ModuleType('matplotlib')
            plt = types.ModuleType('matplotlib.pyplot')
            mpl.pyplot = plt
            mpl.use = lambda *a, **k: None
            sys.modules['matplotlib'] = mpl
            sys.modules['matplotlib.pyplot'] = plt
    if 'torch_scatter' not in sys.modules:
        try:
            import torch_scatter  # noqa: F401
        except Exception:
            sys.modules['torch_scatter'] = types.ModuleType('torch_scatter')
    if 'dgl' in sys.modules:
        return
    try:
        import dgl  # noqa: F401
        return
    except Exception:
        pass

    class ShimGraph:
        def __init__(self, src, dst, num_nodes):
            self.src, self.dst, self._n = src, dst, num_nodes
            self.ndata = {}

        def num_nodes(self):
            return self._n

        number_of_nodes = num_nodes

        def num_edges(self):
            return int(self.src.numel())

        def edges(self):
            return self.src, self.dst

    def from_networkx(g, device=None, **_):
        g2 = nx.convert_node_labels_to_integers(g, ordering='sorted').to_directed()
        e = list(g2.edges())
        src = torch.tensor([a for a, _ in e], dtype=torch.int64, device=device)
        dst = torch.tensor([b for _, b in e], dtype=torch.int64, device=device)
        return ShimGraph(src, dst, g2.number_of_nodes())

    class SAGEConv(nn.Module):
        def __init__(self, in_feats, out_feats, aggregator_type, bias=True, **_):
            super().__init__()
            assert aggregator_type == 'mean'
            self._in, self._out = in_feats, out_feats
            self.fc_neigh = nn.Linear(in_feats, out_feats, bias=False)
            self.fc_self = nn.Linear(in_feats, out_feats, bias=False)
            self.bias = nn.Parameter(torch.zeros(out_feats))
            gain = nn.init.calculate_gain('relu')
            nn.init.xavier_uniform_(self.fc_self.weight, gain=gain)
            nn.init.xavier_uniform_(self.fc_neigh.weight, gain=gain)

        def forward(self, graph, feat):
            h_self = feat
            lin_before_mp = self._in > self._out
            msg = self.fc_neigh(feat) if lin_before_mp else feat
            n = graph.num_nodes()
            agg = torch.zeros(n, msg.shape[1], dtype=msg.dtype, device=msg.device)
            agg.index_add_(0, graph.dst, msg[graph.src])
            deg = torch.zeros(n, dtype=msg.dtype, device=msg.device)
            deg.index_add_(0, graph.dst, torch.ones_like(graph.dst, dtype=msg.dtype))
            h_neigh = agg / deg.clamp(min=1).unsqueeze(1)
            if not lin_before_mp:
                h_neigh = self.fc_neigh(h_neigh)
            return self.fc_self(h_self) + h_neigh + self.bias

    dgl = types.ModuleType('dgl')
    dgl_nn = types.ModuleType('dgl.nn')
    dgl.from_networkx = from_networkx
    dgl.DGLGraph = ShimGraph
    dgl.graph = lambda *a, **k: (_ for _ in ()).throw(NotImplementedError('dead code path'))
    dgl_nn.SAGEConv = SAGEConv
    dgl.nn = dgl_nn
    sys.modules['dgl'] = dgl
    sys.modules['dgl.nn'] = dgl_nn


_REF = None


def load_reference():
    """Import models/{agc,gmatcher}.py of REFERENCE_ROOT unchanged; returns (agc_module, gmatcher_module)."""
    global _REF
    if _REF is not None:
        return _REF
    if not reference_available():
        raise RuntimeError('reference tree not present at %s (set GIMS_REFERENCE_ROOT)' % REFERENCE_ROOT)
    _install_stubs()
    if REFERENCE_ROOT not in sys.path:
        sys.path.insert(0, REFERENCE_ROOT)
    import importlib
    # `models/__init__.py` may import matching.py -> utils.common (cv2, requests, torchvision: present)
    agc = importlib.import_module('models.agc')
    gm = importlib.import_module('models.gmatcher')
    _REF = (agc, gm)
    return _REF
