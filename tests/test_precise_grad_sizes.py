"""Host-only sizing of the fp32-class waveform-gradient entry points (no GPU needed): the ``*_mode`` functions give the
existing sizes for mode 0, at least as much for mode 1, and reject what the existing functions reject."""
import os

import pytest

from nomad_b200 import _lib

SHAPES = ((1, 400), (3, 16384), (32, 32000), (8, 160000))


@pytest.fixture(scope="module")
def lib():
    if not os.path.isfile(_lib.LIB_PATH):
        import __graft_entry__
        __graft_entry__.build()
    return _lib.load()


def _sizes(lib, B, N, mode):
    return (lib.nomad_b200_layers_saved_bytes_mode(B, N, mode), lib.nomad_b200_layers_bwd_workspace_bytes_mode(B, N, mode),
            lib.nomad_b200_loss_workspace_bytes_mode(B, N, 1, mode), lib.nomad_b200_loss_workspace_bytes_mode(B, N, 0, mode))


@pytest.mark.parametrize("B,N", SHAPES)
def test_mode0_is_the_existing_size_and_mode1_is_larger(lib, B, N):
    old = (lib.nomad_b200_layers_saved_bytes(B, N), lib.nomad_b200_layers_bwd_workspace_bytes(B, N),
           lib.nomad_b200_loss_workspace_bytes(B, N, 1), lib.nomad_b200_loss_workspace_bytes(B, N, 0))
    assert _sizes(lib, B, N, 0) == old
    fp32 = _sizes(lib, B, N, 1)
    assert all(s > 0 for s in fp32)
    assert all(a >= b for a, b in zip(fp32[:3], old[:3]))
    # the fp32-class saved forward holds at least the 12 per-layer fp32 QKV rows and pre-LayerNorm sums
    T = lib.nomad_b200_num_frames(N)
    assert fp32[0] > 12 * B * T * (3 * 768 + 2 * 768) * 4
    assert fp32[2] > fp32[3]  # the gradient needs its own scratch


@pytest.mark.parametrize("mode", [0, 1])
def test_too_short_or_empty_batches_are_rejected(lib, mode):
    for B, N in ((2, 399), (0, 16000)):
        assert _sizes(lib, B, N, mode) == (0, 0, 0, 0), (B, N)
    lib.nomad_b200_layers_saved_bytes_mode(2, 399, mode)
    assert b"at least 400" in lib.nomad_b200_last_error()
