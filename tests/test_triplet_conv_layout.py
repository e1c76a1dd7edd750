"""Host-only layout and sizing of the conv-encoder training step (no GPU needed)."""
import os

import pytest

from nomad_b200 import _lib


@pytest.fixture(scope="module")
def lib():
    if not os.path.isfile(_lib.LIB_PATH):
        import __graft_entry__
        __graft_entry__.build()
    return _lib.load()


def test_conv_gradient_segments_tile_the_buffer(lib):
    from nomad_b200.triplet import grad_segments
    from nomad_b200.weights import random_state_dict
    sd = random_state_dict(1234)
    segs = grad_segments(conv=True)
    assert [n for n, _, _ in segs] == (
        ["ssl_model.feature_extractor.conv_layers.0.0.weight", "ssl_model.feature_extractor.conv_layers.0.2.weight",
         "ssl_model.feature_extractor.conv_layers.0.2.bias"]
        + [f"ssl_model.feature_extractor.conv_layers.{l}.0.weight" for l in range(1, 7)])
    end = 0
    for name, off, cnt in segs:
        assert off == end and cnt == sd[name].numel(), name
        end = off + cnt
    assert end == lib.nomad_b200_triplet_conv_grad_floats()
    # the frozen step's layout is a separate buffer and does not name the conv encoder
    assert not any("feature_extractor" in n for n, _, _ in grad_segments())


def test_conv_workspace_is_the_frozen_one_plus_scratch(lib):
    for B, N in ((1, 400), (4, 6000), (8, 160000), (32, 32000)):
        frozen = lib.nomad_b200_triplet_workspace_bytes(B, N)
        conv = lib.nomad_b200_triplet_conv_workspace_bytes(B, N)
        assert frozen > 0 and conv > frozen, (B, N)
    assert lib.nomad_b200_triplet_conv_workspace_bytes(2, 399) == 0
    assert lib.nomad_b200_triplet_conv_workspace_bytes(0, 16000) == 0
