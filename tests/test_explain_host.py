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
