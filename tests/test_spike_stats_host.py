"""Host side of the spike-activity statistics (no GPU): the fan-out table derived from the module tree and the frame size,
and the rate / SynOps / dense-MAC arithmetic of SpikeStats.compute on a synthetic counter buffer."""
import numpy as np
import pytest

# default widths (128, 256, 512, 1024), 144 feature channels, 256 x 256 frames (no skip resize)
TABLE_256 = {
    "enc1": 576 + 1152, "down1.conv1": 2304, "down1.conv2": 2304,
    "enc2": 1152 + 2304, "down2.conv1": 4608, "down2.conv2": 4608,
    "enc3": 2304 + 4608, "down3.conv1": 9216, "down3.conv2": 36864,
    "bottleneck_conv": 2048,
    "up1.conv1": 4608, "up1.conv2": 1024 + 144,
    "up2.conv1": 2304, "up2.conv2": 512 + 144,
    "up3.conv1": 1152, "up3.conv2": 144,
}


@pytest.fixture(scope="module")
def lif_model():
    from snn_object_detectionddp_b200.model import YOLOTemporalUNet
    return YOLOTemporalUNet(num_classes=8, neuron="lif", extractor_backend="standin")


def _table(model, H, W):
    return model.temporal_unet.spike_fanout(model.feature_extractor.feature_hw(H, W))


def test_fanout_table_at_256(lif_model):
    assert lif_model.feature_extractor.feature_hw(256, 256) == [(32, 32), (16, 16), (8, 8)]
    assert _table(lif_model, 256, 256) == TABLE_256


def test_fanout_table_at_480x640_drops_the_resized_skips(lif_model):
    # 60x80 -> 30x40 -> 15x20; down3 pads 15x20 to 16x20 (transparent), the decoder's 16x20 / 32x40 / 64x80 maps differ
    # from the 15x20 / 30x40 / 60x80 skips, so every skip is resized and none of the skip K-slices counts
    assert lif_model.feature_extractor.feature_hw(480, 640) == [(60, 80), (30, 40), (15, 20)]
    want = dict(TABLE_256, enc1=576, enc2=1152, enc3=2304)
    assert _table(lif_model, 480, 640) == want


def test_fanout_equals_dense_conv_macs_per_element(lif_model):
    """For even maps F is kernels._conv_flops / 2 of each consuming K-slice over the slice's elements."""
    from snn_object_detectionddp_b200 import kernels as K
    u = lif_model.temporal_unet
    nb = 3
    # (layer, H, W, C of its spike map, [(geom, Cout of the consumer)])
    s1, s2, k1, t2 = K.GEOM_3x3_S1, K.GEOM_3x3_S2, K.GEOM_1x1, K.GEOM_T2x2_S2
    consumers = {
        "enc1": (32, 128, [(s2, 256), (s1, 128)]), "down1.conv1": (16, 256, [(s1, 256)]), "down1.conv2": (16, 256, [(s1, 256)]),
        "enc2": (16, 256, [(s2, 512), (s1, 256)]), "down2.conv1": (8, 512, [(s1, 512)]), "down2.conv2": (8, 512, [(s1, 512)]),
        "enc3": (8, 512, [(s2, 1024), (s1, 512)]), "down3.conv1": (4, 1024, [(s1, 1024)]),
        "down3.conv2": (4, 1024, [(s1, 4096)]), "bottleneck_conv": (4, 1024, [(t2, 512)]),
        "up1.conv1": (8, 512, [(s1, 512)]), "up1.conv2": (8, 512, [(t2, 256), (k1, 144)]),
        "up2.conv1": (16, 256, [(s1, 256)]), "up2.conv2": (16, 256, [(t2, 128), (k1, 144)]),
        "up3.conv1": (32, 128, [(s1, 128)]), "up3.conv2": (32, 128, [(k1, 144)]),
    }
    table = _table(lif_model, 256, 256)
    for name, (hw, c, cons) in consumers.items():
        macs = sum(K._conv_flops(g, nb, hw, hw, c, co) / 2 for g, co in cons)
        assert table[name] == macs / (nb * hw * hw * c), name
    assert set(consumers) == set(table) == {n for n, m in u.named_modules() if getattr(m, "neuron", None) is not None
                                            and hasattr(m, "bn")}


def test_results_arithmetic_on_a_synthetic_buffer(lif_model):
    from snn_object_detectionddp_b200.spikes import SpikeStats
    st = SpikeStats(lif_model, max_T=8)
    assert st.layers == list(TABLE_256)
    assert st.counts.shape == (16, 2, 8)
    st.fanout = dict(TABLE_256)
    L, T = 16, 3
    rng = np.random.default_rng(0)
    buf = np.zeros((L, 2, 8), dtype=np.int64)
    steps = rng.integers(1 << 30, 1 << 33, size=(L, 1)) * np.ones((1, T), dtype=np.int64)
    spikes = (steps * rng.uniform(0, 0.5, size=(L, T))).astype(np.int64)
    buf[:, 0, :T], buf[:, 1, :T] = spikes, steps
    res = st.results(buf)
    assert res["rate_per_t"].shape == (L, T)
    np.testing.assert_array_equal(res["spike_counts"], spikes)
    np.testing.assert_array_equal(res["neuron_steps"], steps)
    np.testing.assert_allclose(res["rate_per_t"], spikes / steps, rtol=1e-15)
    assert res["spikes/rate"] == int(spikes.sum()) / int(steps.sum())
    for i, name in enumerate(st.layers):
        assert res[f"spikes/rate/{name}"] == int(spikes[i].sum()) / int(steps[i].sum())
    synops = sum(TABLE_256[n] * int(spikes[i].sum()) for i, n in enumerate(st.layers))
    dense = sum(TABLE_256[n] * int(steps[i].sum()) for i, n in enumerate(st.layers))
    assert res["spikes/synops"] == synops and res["spikes/dense_macs"] == dense
    assert res["spikes/synops_fraction"] == synops / dense
    empty = st.results(np.zeros((L, 2, 8), dtype=np.int64))
    assert empty["rate_per_t"].shape == (L, 0) and np.isnan(empty["spikes/rate"]) and empty["spikes/synops"] == 0.0


def test_errors_before_any_launch(lif_model):
    from snn_object_detectionddp_b200.model import YOLOTemporalUNet
    from snn_object_detectionddp_b200.spikes import SpikeStats
    with pytest.raises(ValueError, match="LIF"):
        SpikeStats(YOLOTemporalUNet(num_classes=8, neuron="silu", extractor_backend="standin"))
    with pytest.raises(ValueError, match="max_T"):
        SpikeStats(lif_model, max_T=65)
    st = SpikeStats(lif_model, max_T=4)
    u, dev = lif_model.temporal_unet, st.counts.device
    with pytest.raises(ValueError, match="T=5"):
        st.begin_forward(u, 5, lif_model.feature_extractor.feature_hw(256, 256), dev)
    st.begin_forward(u, 4, lif_model.feature_extractor.feature_hw(256, 256), dev)
    st.reset()
    assert st.fanout == TABLE_256                   # the recorded table survives reset()
    with pytest.raises(ValueError, match="fan-out"):
        st.begin_forward(u, 4, lif_model.feature_extractor.feature_hw(480, 640), dev)
    assert not lif_model.spike_stats and "spike_stats" not in str(list(lif_model.state_dict()))
