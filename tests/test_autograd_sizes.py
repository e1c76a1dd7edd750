"""Host-only sizing of the autograd entry points (no GPU needed)."""
import os

import pytest

from nomad_b200 import _lib


@pytest.fixture(scope="module")
def lib():
    if not os.path.isfile(_lib.LIB_PATH):
        import __graft_entry__
        __graft_entry__.build()
    return _lib.load()


def test_saved_and_backward_workspace_sizes(lib):
    for B, N in ((1, 400), (3, 16384), (32, 32000), (8, 160000)):
        saved = lib.nomad_b200_layers_saved_bytes(B, N)
        bwd = lib.nomad_b200_layers_bwd_workspace_bytes(B, N)
        assert saved > 0 and bwd > 0, (B, N)
        # the saved activations hold at least the 12 per-layer fp32 LayerNorm inputs
        assert saved > 12 * B * lib.nomad_b200_num_frames(N) * 768 * 4
    assert lib.nomad_b200_layers_saved_bytes(8, 32000) > lib.nomad_b200_layers_saved_bytes(4, 32000)


@pytest.mark.parametrize("fn", ["nomad_b200_layers_saved_bytes", "nomad_b200_layers_bwd_workspace_bytes"])
def test_too_short_or_empty_batches_are_rejected(lib, fn):
    assert getattr(lib, fn)(2, 399) == 0
    assert b"at least 400" in lib.nomad_b200_last_error()
    assert getattr(lib, fn)(0, 16000) == 0
