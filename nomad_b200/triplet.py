"""Triplet fine-tuning step of the reference (``src/training/train_triplet.py:92-133``) on the B200 path.

``Training.train`` runs, per batch of (anchor, positive, negative) waveforms: three forwards of ``TripletModel``,
``nn.TripletMarginLoss(margin)``, ``loss.backward()`` and an Adam step with lr 1e-5 for the pre-trained network and
``lr`` for the embedding head (``:96-104``), over everything but the conv feature encoder when ``freeze_convnet: True``
(the default of ``src/config/train_triplet.yaml``) and over the encoder too when it is ``False``.  Here the three
forwards, the loss and ALL parameter gradients come from one C-ABI call (``nomad_b200_triplet_fwd_bwd``, or
``nomad_b200_triplet_conv_fwd_bwd`` with the encoder trained: tensor-core forward, dgrad chain, weight-gradient GEMMs);
the optimiser state and the update are host plumbing (``torch.optim.Adam`` on fp32 master tensors on the GPU), after
which the kernel-ready weights are rebuilt on the device from those tensors (``nomad_b200_refresh_weights``, plus
``nomad_b200_refresh_conv_weights`` for a trained encoder).

Deliberate difference from the reference: the network runs in evaluation mode (no dropout / LayerDrop: fairseq's
``Wav2Vec2Model`` applies dropout 0.1 and layerdrop 0.05 under ``model.train()``, which makes the reference's step
stochastic).
"""
from __future__ import annotations

import ctypes as C
import functools
from collections import OrderedDict
from typing import Dict, Optional, Tuple

import torch

from . import _lib
from .engine import Engine, _ptr, _stream_ptr


@functools.lru_cache(maxsize=None)
def grad_segments(conv: bool = False):
    """[(name, offset, numel)] of the flat gradient buffer (``conv``: of the conv-encoder buffer), as the library lays it
    out."""
    lib = _lib.load()
    seg = lib.nomad_b200_triplet_conv_grad_segment if conv else lib.nomad_b200_triplet_grad_segment
    out, i = [], 0
    name = C.create_string_buffer(128)
    off, cnt = C.c_int64(), C.c_int64()
    while seg(i, name, 128, C.byref(off), C.byref(cnt)) == 0:
        out.append((name.value.decode(), int(off.value), int(cnt.value)))
        i += 1
    return out


_DEV_CACHE: Dict = {}


def _device_copy(engine: Engine, state_dict, key: str) -> torch.Tensor:
    """fp32 copy of a (host) checkpoint tensor on the engine's device, cached per source tensor version: the positional
    conv's weight_v is 19 MB, and a pageable H2D copy of it per step cost 1.5 ms."""
    t = state_dict[key]
    if t.is_cuda:
        return t.detach().to(torch.float32).clone()
    tag = (id(t), t._version, engine.device_index)
    hit = _DEV_CACHE.get(key)
    if hit is None or hit[0] != tag:
        _DEV_CACHE[key] = (tag, t.detach().to(engine.device, torch.float32))
    return _DEV_CACHE[key][1].clone()


SHAPES = {"qkv.weight": (2304, 768), "self_attn.out_proj.weight": (768, 768), "fc1.weight": (3072, 768),
          "fc2.weight": (768, 3072), "post_extract_proj.weight": (768, 512), "embedding_layer.1.weight": (256, 768)}


POS_V, POS_G = "ssl_model.encoder.pos_conv.0.weight_v", "ssl_model.encoder.pos_conv.0.weight_g"


def grads_by_name(flat: torch.Tensor, scale, weight_v: torch.Tensor, weight_g: torch.Tensor,
                  conv_flat: Optional[torch.Tensor] = None, conv_shapes=None) -> "OrderedDict[str, torch.Tensor]":
    """The library's flat gradient buffers (``grad_segments()`` and, when ``conv_flat`` is given, ``grad_segments(conv=
    True)``; both times the scale S: a float or a 0-dim tensor on their device) -> {state_dict key: gradient}.  The fused
    q|k|v rows are split (q carries the kernel's head_dim^-0.5), the positional conv's folded-weight gradient goes through
    the weight-norm backward to ``weight_v`` / ``weight_g`` (the values the forward used), ``conv_shapes`` gives the
    checkpoint shapes of the conv tensors."""
    flat = flat / scale
    grads: "OrderedDict[str, torch.Tensor]" = OrderedDict()
    for name, off, cnt in grad_segments():
        g = flat[off:off + cnt]
        leaf = next((k for k in SHAPES if name.endswith(k)), None)
        if leaf is not None:
            g = g.view(SHAPES[leaf])
        if name.endswith("qkv.weight") or name.endswith("qkv.bias"):
            base = name[: -len("qkv.weight")] if name.endswith("weight") else name[: -len("qkv.bias")]
            kind = "weight" if name.endswith("weight") else "bias"
            q, k, v = g[:768], g[768:1536], g[1536:]
            grads[base + f"self_attn.q_proj.{kind}"] = q * 0.125   # the kernel's q rows carry head_dim^-0.5
            grads[base + f"self_attn.k_proj.{kind}"] = k
            grads[base + f"self_attn.v_proj.{kind}"] = v
        elif name.endswith("pos_conv.0.folded_weight"):
            # [g][n][tap][c] -> (out = g * 48 + n, in = c, tap); then through weight_norm(dim=2): w = g * v / ||v||
            dw = g.view(16, 48, 128, 48).permute(0, 1, 3, 2).reshape(768, 48, 128)
            with torch.enable_grad():
                v = weight_v.detach().to(flat.device, torch.float32).requires_grad_(True)
                gg = weight_g.detach().to(flat.device, torch.float32).requires_grad_(True)
                w = gg * v / v.pow(2).sum(dim=(0, 1), keepdim=True).sqrt()
                gv, ggr = torch.autograd.grad(w, (v, gg), dw)
            grads[POS_V] = gv
            grads[POS_G] = ggr
        else:
            grads[name] = g
    if conv_flat is not None:
        conv_flat = conv_flat / scale
        for name, off, cnt in grad_segments(conv=True):   # already in the checkpoint's (out, in, tap) order
            grads[name] = conv_flat[off:off + cnt].view(conv_shapes[name])
    return grads


def triplet_loss_and_grads(engine: Engine, state_dict, anchor: torch.Tensor, positive: torch.Tensor, negative: torch.Tensor,
                           margin: float = 0.2, freeze_convnet: bool = True,
                           feature_grad_mult: float = 0.1) -> Tuple[torch.Tensor, "OrderedDict[str, torch.Tensor]"]:
    """loss (0-dim CUDA tensor) and {state_dict key: gradient} for every trainable tensor.  ``freeze_convnet=False``
    trains the conv feature encoder too: its 9 tensors join the result, with fairseq's GradMultiply of
    ``feature_grad_mult`` on the conv features (the frozen step has no gradient below the conv features for it to scale).
    ``anchor`` / ``positive`` / ``negative``: (B, N) or (B, 1, N) waveforms of one common length."""
    lib = engine.lib
    engine.sync_weights()
    sq = lambda t: (t.squeeze(1) if t.dim() == 3 else t).to(engine.device, torch.float32)
    wav = torch.cat([sq(anchor), sq(positive), sq(negative)]).contiguous()
    B, N = wav.shape[0] // 3, wav.shape[1]
    need = (lib.nomad_b200_triplet_workspace_bytes if freeze_convnet else lib.nomad_b200_triplet_conv_workspace_bytes)(B, N)
    if need == 0:
        raise _lib.NomadB200Error(lib.nomad_b200_last_error().decode())
    wp, wbytes = engine._aligned(engine.workspace(need))
    n_grad = int(lib.nomad_b200_triplet_grad_floats())
    flat = torch.empty((n_grad,), dtype=torch.float32, device=engine.device)
    loss = torch.empty((), dtype=torch.float32, device=engine.device)
    scale = C.c_float()
    with torch.cuda.device(engine.device):
        if freeze_convnet:
            _lib.check(lib.nomad_b200_triplet_fwd_bwd(engine.handle, _ptr(wav), B, N, C.c_float(margin), _ptr(loss), _ptr(flat),
                                                      C.byref(scale), wp, wbytes, _stream_ptr()), "nomad_b200_triplet_fwd_bwd")
        else:
            conv_flat = torch.empty((int(lib.nomad_b200_triplet_conv_grad_floats()),), dtype=torch.float32, device=engine.device)
            _lib.check(lib.nomad_b200_triplet_conv_fwd_bwd(engine.handle, _ptr(wav), B, N, C.c_float(margin),
                                                           C.c_float(feature_grad_mult), _ptr(loss), _ptr(flat), _ptr(conv_flat),
                                                           C.byref(scale), wp, wbytes, _stream_ptr()),
                       "nomad_b200_triplet_conv_fwd_bwd")
    conv_shapes = None if freeze_convnet else {k: state_dict[k].shape for k, _, _ in grad_segments(conv=True)}
    grads = grads_by_name(flat, scale.value, _device_copy(engine, state_dict, POS_V), _device_copy(engine, state_dict, POS_G),
                          None if freeze_convnet else conv_flat, conv_shapes)
    return loss, grads


class TripletTrainer:
    """``Training.train``'s inner step (``train_triplet.py:112-133``) with the optimiser of ``:92-107``.
    ``freeze_convnet=False`` trains the conv feature encoder as well (its tensors are part of ``ssl_model`` and take
    ``lr_pretrained``), with ``nomad.feature_grad_mult`` on the conv features as fairseq applies it."""

    def __init__(self, nomad, lr: float = 1e-4, margin: float = 0.2, lr_pretrained: float = 1e-5,
                 freeze_convnet: bool = True):
        self.nomad = nomad
        self.margin = margin
        self.freeze_convnet = freeze_convnet
        dev = nomad.engine.device
        self.master = OrderedDict((k, v.detach().to(dev, torch.float32).clone()) for k, v in self._state_dict(nomad).items())
        head = ["embedding_layer.1.weight", "embedding_layer.1.bias"]
        train = [k for k in self.master if not k.endswith("mask_emb") and not (freeze_convnet and "feature_extractor" in k)]
        for k in train:
            self.master[k].requires_grad_(True)
        self.optim = torch.optim.Adam([{"params": [self.master[k] for k in train if k not in head], "lr": lr_pretrained},
                                       {"params": [self.master[k] for k in head]}], lr=lr, fused=True)

    @staticmethod
    def _state_dict(nomad):
        sd = getattr(nomad, "state_dict_ref", None)
        if sd is None:
            raise ValueError("TripletTrainer needs the Nomad to be built with keep_state_dict=True")
        return sd

    def step(self, anchor, positive, negative) -> float:
        loss, grads = triplet_loss_and_grads(self.nomad.engine, self.master, anchor, positive, negative, self.margin,
                                             self.freeze_convnet, self.nomad.feature_grad_mult)
        self.optim.zero_grad(set_to_none=True)
        for k, g in grads.items():
            self.master[k].grad = g.reshape(self.master[k].shape).contiguous()
        self.optim.step()
        # rebuild the kernel-ready weights (16-bit copies, q|k|v fusion, transposes, LayerNorm folds, weight-norm fold) from
        # the updated master tensors, on the device
        self.nomad.engine.refresh_weights(self.master)
        if not self.freeze_convnet:
            self.nomad.engine.refresh_conv_weights(self.master)
        return float(loss.item())
