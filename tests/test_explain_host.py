"""Argument checks of Explainer that must raise before any device work (no GPU)."""
from types import SimpleNamespace

import numpy as np
import pytest
import torch


class _HostPairSet:
    """The host fields of a PairSet that Explainer reads before it touches the device."""

    def __init__(self, n, F=8):
        self.n_h = np.full(n, 5, dtype=np.int64)
        self.e_h = np.full(n, 8, dtype=np.int64)
        self.graph = SimpleNamespace(F=F, device=torch.device("cpu"))

    def __len__(self):
        return len(self.n_h)


def _explainer(n=10, F=8, B=4):
    """An Explainer with its host state only (no engine): explain() must reject bad arguments before it needs one."""
    from npi_gnn_b200 import Explainer
    ex = Explainer.__new__(Explainer)
    ex.ps, ex.params, ex.B, ex.P, ex.index = _HostPairSet(n, F), None, B, n, None
    ex.n_rows, ex.device, ex.engine = ex.ps.n_h, torch.device("cpu"), None
    return ex


@pytest.mark.parametrize("index", [[], np.zeros(0, dtype=np.int64)])
def test_empty_view_is_rejected(index):
    from npi_gnn_b200 import Explainer
    with pytest.raises(ValueError, match="nothing to explain"):
        Explainer(_HostPairSet(10), None, index=index)
    with pytest.raises(ValueError, match="nothing to explain"):
        Explainer(_HostPairSet(0), None)


def test_index_out_of_range_and_bad_batch_size_are_rejected():
    from npi_gnn_b200 import Explainer
    for index in ([0, 10], [-1], [3, 4, 11]):
        with pytest.raises(ValueError, match="index"):
            Explainer(_HostPairSet(10), None, index=index)
    with pytest.raises(ValueError, match="batch_size"):
        Explainer(_HostPairSet(10), None, batch_size=0)


@pytest.mark.parametrize("target", [2, -1, "1", None, 1.5])
def test_target_outside_the_two_classes_is_rejected(target):
    with pytest.raises(ValueError, match="target"):
        _explainer().explain(target=target)


@pytest.mark.parametrize("wrt", ["p", "log", None, "PROB"])
def test_unknown_wrt_is_rejected(wrt):
    with pytest.raises(ValueError, match="wrt"):
        _explainer().explain(wrt=wrt)


def test_full_gradient_that_does_not_fit_is_rejected_with_its_size(monkeypatch):
    ex = _explainer(n=10, F=8)
    need = 10 * 5 * 8 * 4
    monkeypatch.setattr(torch.cuda, "mem_get_info", lambda device=None: (need - 1, 1 << 40))
    with pytest.raises(ValueError, match="%d bytes" % need):
        ex.explain(full=True)


@pytest.mark.parametrize("k", [0, -3, 1025])
def test_top_nodes_rejects_k(k):
    from npi_gnn_b200 import Explainer
    res = dict(node_attr=torch.zeros(4), node_ptr=torch.tensor([0, 4]), node=torch.zeros(4, dtype=torch.int32))
    with pytest.raises(ValueError, match="k"):
        Explainer.top_nodes(res, k)


@pytest.mark.parametrize("order", [None, [3], [7, 2, 9], np.arange(10)[::-1], [1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1]])
def test_batch_caps_of_a_view_sums_each_batch_of_the_view(order):
    """PairSet.batch_caps over an ``order`` of any length (the Scorer and Explainer views) against plain per-batch sums."""
    from npi_gnn_b200.graph import PairSet
    ps, B = _HostPairSet(10), 4
    ps.n_h = np.arange(10, dtype=np.int64) + 2
    ps.e_h = 3 * np.arange(10, dtype=np.int64)[::-1] + 1
    idx = np.arange(10) if order is None else np.asarray(order)
    batches = [idx[i:i + B] for i in range(0, len(idx), B)]
    want = (max(int(ps.n_h[b].sum()) for b in batches), max(int(ps.e_h[b].sum()) for b in batches), int(ps.n_h[idx].max()))
    assert PairSet.batch_caps(ps, B, order) == want
