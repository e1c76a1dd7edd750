"""Host-only parts of parameter gradients through autograd (no GPU needed): the sizing of the parameter entry points,
the flat-buffer-to-checkpoint-name mapping and the keep_state_dict requirement."""
import os
from types import SimpleNamespace

import pytest
import torch

from nomad_b200 import _lib


@pytest.fixture(scope="module")
def lib():
    if not os.path.isfile(_lib.LIB_PATH):
        import __graft_entry__
        __graft_entry__.build()
    return _lib.load()


P, CV = _lib.SAVE_PARAMS, _lib.SAVE_CONV


def test_sizes_grow_with_what_is_saved(lib):
    for B, N in ((1, 400), (3, 16000), (8, 160000)):
        plain = lib.nomad_b200_layers_saved_bytes(B, N)
        assert lib.nomad_b200_layers_saved_bytes_ex(B, N, 0) == plain > 0
        # PARAMS keeps each layer's GELU(fc1) activations: 12 x frames x 3072 16-bit values more
        frames = B * lib.nomad_b200_num_frames(N)
        assert lib.nomad_b200_layers_saved_bytes_ex(B, N, P) >= plain + 12 * frames * 3072 * 2
        assert lib.nomad_b200_layers_saved_bytes_ex(B, N, P | CV) == lib.nomad_b200_layers_saved_bytes_ex(B, N, P)
        bwd = lib.nomad_b200_layers_bwd_workspace_bytes(B, N)
        params = lib.nomad_b200_layers_bwd_params_workspace_bytes(B, N, P)
        conv = lib.nomad_b200_layers_bwd_params_workspace_bytes(B, N, P | CV)
        assert 0 < bwd < params < conv, (B, N, bwd, params, conv)


@pytest.mark.parametrize("fn", ["nomad_b200_layers_saved_bytes_ex", "nomad_b200_layers_bwd_params_workspace_bytes"])
def test_short_or_empty_batches_are_rejected(lib, fn):
    assert getattr(lib, fn)(2, 399, P) == 0
    assert b"at least 400" in lib.nomad_b200_last_error()
    assert getattr(lib, fn)(0, 16000, P | CV) == 0


def test_flat_mapping_covers_every_trainable_key_once(lib):
    from nomad_b200.triplet import POS_G, POS_V, grad_segments, grads_by_name
    from nomad_b200.weights import random_state_dict
    sd = random_state_dict(3)
    conv_names = [n for n, _, _ in grad_segments(conv=True)]
    flat = torch.arange(int(lib.nomad_b200_triplet_grad_floats()), dtype=torch.float32)
    conv = torch.arange(int(lib.nomad_b200_triplet_conv_grad_floats()), dtype=torch.float32)
    g = grads_by_name(flat, 2.0, sd[POS_V], sd[POS_G], conv, {k: sd[k].shape for k in conv_names})
    trainable = [k for k in sd if not k.endswith("mask_emb")]
    assert sorted(g) == sorted(trainable)
    for k in trainable:
        assert g[k].shape == sd[k].shape, k
    # every flat element lands in exactly one tensor (the folded positional-conv weight through its weight norm)
    direct = [k for k in trainable if k not in (POS_V, POS_G)]
    seen = torch.cat([g[k].reshape(-1) * (8.0 if k.endswith("q_proj.weight") or k.endswith("q_proj.bias") else 1.0)
                      for k in direct if "feature_extractor" not in k]) * 2.0
    pos = [o for n, o, c in grad_segments() if n.endswith("folded_weight")][0]
    n_pos = 16 * 48 * 128 * 48
    expect = torch.cat([flat[:pos], flat[pos + n_pos:]])
    assert torch.equal(torch.sort(seen).values, expect)
    assert torch.equal(torch.sort(torch.cat([g[k].reshape(-1) for k in conv_names]) * 2.0).values, conv)


def test_parameters_need_keep_state_dict():
    from nomad_b200.nomad import TripletModel, _ParamStore
    with pytest.raises(ValueError, match="keep_state_dict=True"):
        TripletModel(None).parameters()
    store = _ParamStore(SimpleNamespace(state_dict_ref=None, engine=None))
    with pytest.raises(ValueError, match="keep_state_dict=True"):
        TripletModel(None, store=store).named_parameters()
    assert store.trainable(0) == [] and store.params is None
