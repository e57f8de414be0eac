"""CPU: the decay table of ema.ModelEMA, its argument checks, the averaged copy's structure and the store without
optimizer buffers."""
import math

import numpy as np
import pytest
import torch

from snn_object_detectionddp_b200 import kernels as K
from snn_object_detectionddp_b200.ema import ModelEMA, _averaged_copy, decay_table


@pytest.mark.parametrize("decay,tau", [(0.9999, 2000), (0.999, 100), (0.5, 3)])
def test_decay_table_rows_are_ultralytics_lambda_and_saturate(decay, tau):
    t = decay_table(decay, tau)
    assert t.dtype == torch.float32 and t.dim() == 2 and t.shape[1] == 2
    ks = np.arange(1, t.shape[0] + 1)
    d = np.array([decay * (1 - math.exp(-k / tau)) for k in ks])             # ultralytics' lambda, in double
    assert np.array_equal(t[:, 0].numpy(), d.astype(np.float32))
    assert np.array_equal(t[:, 1].numpy(), (1 - d).astype(np.float32))
    # the last row is the first at which both columns reach their fp32 limits, and every later update rounds to it
    lim = np.float32(decay), np.float32(1 - decay)
    assert (t[-1, 0].item(), t[-1, 1].item()) == (float(lim[0]), float(lim[1]))
    if t.shape[0] > 1:
        assert (t[-2, 0].item(), t[-2, 1].item()) != (float(lim[0]), float(lim[1]))
    for k in (t.shape[0] + 1, t.shape[0] + 7, 10 * t.shape[0], 10 ** 9):
        dk = decay * (1 - math.exp(-k / tau))
        assert (np.float32(dk), np.float32(1 - dk)) == lim, k


def test_default_table_size():
    t = decay_table()
    assert 50_000 < t.shape[0] < 60_000 and t.numel() * 4 < 512 * 1024
    assert t[0, 0].item() == float(np.float32(0.9999 * (1 - math.exp(-1 / 2000))))


@pytest.mark.parametrize("kw", [dict(decay=0.0), dict(decay=1.0), dict(decay=-0.1), dict(decay=1.5), dict(tau=0),
                                dict(tau=-5.0)])
def test_arguments_are_validated(kw):
    args = dict(decay=0.9999, tau=2000)
    args.update(kw)
    with pytest.raises(ValueError):
        decay_table(**args)
    with pytest.raises(ValueError):
        ModelEMA(None, **args)                     # rejected before the model is looked at


def _model():
    from snn_object_detectionddp_b200.model import TemporalUNet, YOLOTemporalUNet
    torch.manual_seed(0)
    net = YOLOTemporalUNet(num_classes=4, neuron="lif", extractor_backend="standin")
    net.temporal_unet = TemporalUNet([144, 144, 144], neuron="lif", widths=(16, 32, 64, 128))
    return net


def test_averaged_copy_shares_the_extractor_and_drops_store_and_stats():
    net = _model()
    net.spike_stats = object()
    object.__setattr__(net, "_snn_store", object())
    c = _averaged_copy(net)
    assert c.feature_extractor is net.feature_extractor
    assert c.spike_stats is None and "_snn_store" not in c.__dict__
    assert net.spike_stats is not None and "_snn_store" in net.__dict__
    sa, sb = net.state_dict(), c.state_dict()
    assert list(sa) == list(sb) and all(torch.equal(sa[k], sb[k]) for k in sa)
    pa, pb = dict(net.named_parameters()), dict(c.named_parameters())
    assert all(pa[k] is not pb[k] and pa[k].data_ptr() != pb[k].data_ptr() for k in pa)
    # the state dict's alias of the head (model.0.*) stays an alias in the copy
    assert c.model[0] is c.detection_head


def test_store_without_optimizer_state(monkeypatch):
    from snn_object_detectionddp_b200.params import ParamStore
    monkeypatch.setattr(K, "_EMULATED", True, raising=False)      # let the store live on the CPU for this check
    net = _model()
    st = ParamStore(net)
    st.ensure("cpu", optimizer_state=False)
    assert st.flat_g is None and st.flat_m is None and st.flat_v is None
    assert st.flat_p.numel() == st.total and st.shadow.dtype == torch.bfloat16
    assert all(st._attached(e) for e in st.entries)
    full = ParamStore(_model())
    full.ensure("cpu")
    assert all(t is not None and t.numel() == full.total for t in (full.flat_g, full.flat_m, full.flat_v))

