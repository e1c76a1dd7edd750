"""Triplet fine-tuning with the conv feature encoder trained (reference ``src/config/train_triplet.yaml``
``freeze_convnet: False``): the conv gradients against CPU autograd on the oracle, the unchanged frozen outputs, the
device-side rebuild of the conv weights and the trainer.  Every comparison records the error it ACHIEVED."""
import ctypes as C
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

MARGIN = 0.5
CONV_KEYS = (["ssl_model.feature_extractor.conv_layers.0.0.weight", "ssl_model.feature_extractor.conv_layers.0.2.weight",
              "ssl_model.feature_extractor.conv_layers.0.2.bias"]
             + [f"ssl_model.feature_extractor.conv_layers.{l}.0.weight" for l in range(1, 7)])


@pytest.fixture(scope="module")
def sd():
    from nomad_b200.weights import random_state_dict
    return random_state_dict(1234)


def _triplets(B, N, seed):
    g = torch.Generator().manual_seed(seed)
    A = 0.1 * torch.randn(B, N, generator=g)
    P = A + 0.1 * torch.randn(B, N, generator=g)    # positives: the anchor at 0 dB SNR
    Nn = 0.1 * torch.randn(B, N, generator=g)
    return A, P, Nn


def _reference(sd, A, P, Nn, fgm):
    """loss, {key: grad} of every trainable tensor (conv encoder included) by CPU autograd, and the hinge margins."""
    from oracle import w2v_oracle as O
    torch.set_num_threads(os.cpu_count() or 1)
    sdg = {k: (v.clone().requires_grad_(True) if not k.endswith("mask_emb") else v) for k, v in sd.items()}

    def emb(w):
        layers = O.ssl_layers(sdg, w, feature_grad_mult=fgm)
        return O.head(layers[-1], sdg["embedding_layer.1.weight"], sdg["embedding_layer.1.bias"])
    ea, ep, en = emb(A), emb(P), emb(Nn)
    loss = torch.nn.TripletMarginLoss(margin=MARGIN)(ea, ep, en)
    loss.backward()
    hinge = ((ea - ep + 1e-6).norm(dim=1) - (ea - en + 1e-6).norm(dim=1) + MARGIN).detach()
    grads = {k: v.grad for k, v in sdg.items() if torch.is_tensor(v) and v.requires_grad}
    return loss.item(), grads, hinge


def _compare(grads, ref, record, tag, per_tensor=lambda k: True, **extra):
    """The bounds of the frozen step's gradient test (test_triplet_step_gradients_against_autograd): per tensor for the
    tensors ``per_tensor`` selects, all gradients as one vector over every tensor.  Everything is recorded before
    asserting."""
    names = sorted(ref)
    missing = [k for k in names if k not in grads]
    assert not missing, missing
    ours = {k: grads[k].detach().cpu().reshape(-1).double() for k in names}
    refs = {k: ref[k].reshape(-1).double() for k in names}
    med = float(torch.tensor([float(refs[k].norm()) for k in names]).median())
    table, bad = [], []
    for k in names:
        a, b = ours[k], refs[k]
        assert torch.isfinite(a).all(), k
        if k.endswith("k_proj.bias"):   # softmax ignores a constant key shift: exactly zero in exact arithmetic
            assert float(a.norm()) <= 1e-3 * med, (k, float(a.norm()), med)
            continue
        diff = float((a - b).norm())
        cos = float((a @ b) / (a.norm() * b.norm()).clamp_min(1e-30))
        table.append((diff / (3e-2 * float(b.norm()) + 1e-3 * med), cos, k, diff / float(b.norm().clamp_min(1e-30))))
        if per_tensor(k) and not (diff <= 3e-2 * float(b.norm()) + 1e-3 * med and cos >= 0.995):
            bad.append((k, diff, float(b.norm()), cos))
    keep = [k for k in names if not k.endswith("k_proj.bias")]
    va, vb = torch.cat([ours[k] for k in keep]), torch.cat([refs[k] for k in keep])
    g_rel = float((va - vb).norm() / vb.norm())
    g_cos = float((va @ vb) / (va.norm() * vb.norm()))
    conv = [t for t in table if "feature_extractor" in t[2]]
    for rel, cos, k, r in sorted(table, reverse=True)[:8]:
        print(f"GRAD {rel:8.3f} of bound  rel {r:10.3e}  cos {cos:.6f}  {k}")
    record(tag, all_grads_rel_l2=g_rel, all_grads_cosine=g_cos, tensors=len(names),
           tightest_check_fraction_of_bound=max(table)[0], tightest_check_tensor=max(table)[2],
           conv_worst_fraction_of_bound=max(conv)[0], conv_worst_tensor=max(conv)[2],
           conv_worst_rel_l2=max(t[3] for t in conv), conv_min_cosine=min(t[1] for t in conv),
           conv_rel_l2={t[2].split("conv_layers.")[1]: t[3] for t in conv}, **extra)
    assert not bad, (bad, med)
    assert g_rel <= 2.5e-2 and g_cos >= 0.9997, (g_rel, g_cos)


def _check_step(sd, B, N, seed, fgm, record, tag, per_tensor=lambda k: True):
    from nomad_b200.engine import Engine
    from nomad_b200.triplet import triplet_loss_and_grads
    eng = Engine(sd, 0)
    A, P, Nn = _triplets(B, N, seed)
    loss, grads = triplet_loss_and_grads(eng, sd, A, P, Nn, margin=MARGIN, freeze_convnet=False, feature_grad_mult=fgm)
    ref_loss, ref, hinge = _reference(sd, A, P, Nn, fgm)
    # the hinge is a discontinuity of the gradient: every triplet must sit clearly on one side of it
    assert ref_loss > 0.0 and float(hinge.abs().min()) > 0.02, hinge
    assert all(k in grads for k in CONV_KEYS)
    rel_loss = abs(loss.item() - ref_loss) / ref_loss
    _compare(grads, ref, record, tag, per_tensor=per_tensor, B=B, N=N, fgm=fgm, loss=loss.item(), loss_rel_err=rel_loss)
    assert rel_loss <= 1e-3
    return grads, ref


@pytest.mark.parametrize("fgm", [1.0, 0.1])
def test_conv_training_gradients_against_autograd(sd, fgm, record):
    """Every trainable tensor, the 9 conv-encoder tensors included, against the oracle's CPU autograd at 4 x 6000."""
    _check_step(sd, 4, 6000, 31, fgm, record, "triplet_conv_step")


def _vec(g, keys):
    return torch.cat([g[k].detach().cpu().reshape(-1).double() for k in keys if not k.endswith("k_proj.bias")])


def test_conv_training_gradients_long_utterances(sd, record):
    """2 triplets x 10 s: the conv weight gradients split K (up to 24 slices at level 1) and every level has padding rows
    past the utterance's valid frames.  At this length the frozen step's own gradients (the parameters above the conv
    encoder, computed by the unchanged frozen entry point) are 4.7 % off the oracle as one vector on this input, outside
    the bound the 4 x 6000 case uses; the conv gradients are computed from them, so the check here is that the conv
    gradients are no less accurate than those upstream gradients, and that the rest equals the frozen entry's output."""
    from nomad_b200.engine import Engine
    from nomad_b200.triplet import triplet_loss_and_grads
    eng = Engine(sd, 0)
    A, P, Nn = _triplets(2, 160000, 32)
    loss, grads = triplet_loss_and_grads(eng, sd, A, P, Nn, margin=MARGIN, freeze_convnet=False, feature_grad_mult=0.1)
    _, frozen = triplet_loss_and_grads(eng, sd, A, P, Nn, margin=MARGIN)
    ref_loss, ref, hinge = _reference(sd, A, P, Nn, 0.1)
    assert ref_loss > 0.0 and float(hinge.abs().min()) > 0.02, hinge
    rest = list(frozen)
    ref_conv, ours_conv = _vec(ref, CONV_KEYS), _vec(grads, CONV_KEYS)
    ref_rest, ours_rest = _vec(ref, rest), _vec(frozen, rest)
    rel = lambda a, b: float((a - b).norm() / b.norm())
    cos = lambda a, b: float((a @ b) / (a.norm() * b.norm()))
    per_conv = {k.split("conv_layers.")[1]: rel(_vec(grads, [k]), _vec(ref, [k])) for k in CONV_KEYS}
    same = max(float((frozen[k] - grads[k]).norm() / frozen[k].norm()) for k in rest if not k.endswith("k_proj.bias"))
    rel_loss = abs(loss.item() - ref_loss) / ref_loss
    record("triplet_conv_step_long", B=2, N=160000, fgm=0.1, loss_rel_err=rel_loss, conv_rel_l2=rel(ours_conv, ref_conv),
           conv_cosine=cos(ours_conv, ref_conv), conv_rel_l2_per_tensor=per_conv,
           frozen_step_rel_l2=rel(ours_rest, ref_rest), frozen_step_cosine=cos(ours_rest, ref_rest),
           rest_vs_frozen_entry_worst_rel_l2=same)
    assert all(torch.isfinite(grads[k]).all() for k in CONV_KEYS)
    assert rel_loss <= 1e-3
    assert same <= 1e-4, same
    assert rel(ours_conv, ref_conv) <= rel(ours_rest, ref_rest) and cos(ours_conv, ref_conv) >= cos(ours_rest, ref_rest)
    assert max(per_conv.values()) <= 1.5 * rel(ours_rest, ref_rest), per_conv


def test_groupnorm_gamma_zero(sd, record):
    """GroupNorm channels with gamma exactly 0 still get a finite, correct d gamma (the gradient is taken without the
    gamma * rstd factor, never by dividing by gamma).  Per-tensor bounds on the 9 conv tensors, aggregate bounds on all:
    on this input the top layer's q projection gradients (1e-5 of the median norm, computed by the unchanged frozen
    step) reach cosine 0.9948, just under the per-tensor 0.995."""
    sd0 = dict(sd)
    gam = sd["ssl_model.feature_extractor.conv_layers.0.2.weight"].clone()
    zero = torch.tensor([0, 5, 77, 300, 511])
    gam[zero] = 0.0
    sd0["ssl_model.feature_extractor.conv_layers.0.2.weight"] = gam
    grads, ref = _check_step(sd0, 4, 6000, 34, 1.0, record, "triplet_conv_step_gamma0",
                             per_tensor=lambda k: "feature_extractor" in k)
    key = "ssl_model.feature_extractor.conv_layers.0.2.weight"
    ours, want = grads[key].cpu().double()[zero], ref[key].double()[zero]
    assert torch.isfinite(ours).all()
    assert float(want.abs().min()) > 0.0
    err = float((ours - want).abs().max() / want.abs().max())
    record("triplet_conv_gamma0_dgamma", max_err_over_max=err)
    assert err <= 3e-2, (ours, want)


def test_frozen_outputs_unchanged_by_conv_mode(sd, record):
    """The conv-training entry returns the frozen step's loss, scale and non-conv gradients (float atomics in the column
    sums: not bit-comparable), and the frozen entry keeps its launch count."""
    from nomad_b200.engine import Engine
    from nomad_b200.triplet import triplet_loss_and_grads
    eng = Engine(sd, 0)
    A, P, Nn = _triplets(4, 6000, 31)
    l0, g0 = triplet_loss_and_grads(eng, sd, A, P, Nn, margin=MARGIN)
    torch.cuda.synchronize()
    n0 = eng.launch_count()
    l0b, _ = triplet_loss_and_grads(eng, sd, A, P, Nn, margin=MARGIN)
    torch.cuda.synchronize()
    frozen_launches = eng.launch_count() - n0
    n1 = eng.launch_count()
    l1, g1 = triplet_loss_and_grads(eng, sd, A, P, Nn, margin=MARGIN, freeze_convnet=False, feature_grad_mult=0.1)
    torch.cuda.synchronize()
    conv_launches = eng.launch_count() - n1
    assert abs(float(l0) - float(l1)) <= 1e-6 * abs(float(l0)) and abs(float(l0) - float(l0b)) <= 1e-6 * abs(float(l0))
    assert set(g1) - set(g0) == set(CONV_KEYS)
    worst = 0.0
    for k, a in g0.items():
        b = g1[k]
        d = float((a - b).norm() / a.norm().clamp_min(1e-30))
        if k.endswith("k_proj.bias"):
            continue
        worst = max(worst, d)
    record("triplet_conv_frozen_outputs", worst_rel_l2_vs_frozen_entry=worst, frozen_launches=frozen_launches,
           conv_launches=conv_launches)
    assert worst <= 1e-4, worst
    assert conv_launches > frozen_launches


def _read(e, name, n, dt):
    from nomad_b200 import _lib
    buf = np.empty(n, dt)
    _lib.check(e.lib.nomad_b200_debug_read_weight(e.handle, name.encode(), buf.ctypes.data_as(C.c_void_p), buf.nbytes), name)
    return buf


def test_conv_weight_refresh_equals_a_fresh_handle(sd):
    """``refresh_conv_weights`` on handle A after perturbing only the conv tensors: every conv buffer has the bits of a
    fresh handle B built from those tensors, embeddings are bit-identical, and A's captured loss-step graph replays the
    new weights."""
    from nomad_b200.engine import Engine
    g = torch.Generator().manual_seed(78)
    sd2 = {k: (v + 0.05 * v.abs().mean() * torch.randn(v.shape, generator=g) if "feature_extractor" in k else v.clone())
           for k, v in sd.items()}
    a = Engine(sd, 0)
    hw, hb = 0.03 * torch.randn(256, 768, generator=g), torch.zeros(256)
    est, cln = (0.1 * torch.randn(2, 8000, generator=g)).cuda(), (0.1 * torch.randn(2, 8000, generator=g)).cuda()
    a.set_loss_head(hw, hb)
    for _ in range(3):   # eager, capture, replay: A's loss step is a CUDA graph from here on
        a.loss_fwd_bwd(est, cln, 0.1)
    waves = [0.1 * torch.randn(n, generator=g) for n in (16000, 20481, 4000)]
    before = a.embed(waves).clone()
    a.refresh_conv_weights({k: v.cuda().contiguous() for k, v in sd2.items()})
    b = Engine(sd2, 0)
    b.set_loss_head(hw, hb)
    bufs = [("conv0_w", 5120, np.float32), ("gn_g", 512, np.float32), ("gn_b", 512, np.float32),
            ("conv0_wh", 16 * 512, np.uint16)]
    for l in range(1, 7):
        k = 3 if l <= 4 else 2
        bufs += [(f"c{l}.w", 512 * 512 * k, np.uint16), (f"c{l}.wt", 512 * 512 * k, np.uint16)]
        if k == 3:
            bufs.append((f"c{l}.wte", 512 * 1024, np.uint16))
    for name, n, dt in bufs:
        x, y = _read(a, name, n, dt), _read(b, name, n, dt)
        assert np.array_equal(x, y), (name, int((x != y).sum()))
    ea, eb = a.embed(waves), b.embed(waves)
    assert float((before - eb).abs().max()) > 1e-4          # the weights really changed
    assert torch.equal(ea, eb)
    out = []
    for e in (a, b):
        for _ in range(3 if e is b else 1):
            l, gr = e.loss_fwd_bwd(est, cln, 0.1)
        out.append((float(l), gr.clone()))
    assert abs(out[0][0] - out[1][0]) <= 1e-6 * abs(out[1][0])
    assert float((out[0][1] - out[1][1]).abs().max()) <= 1e-6 * float(out[1][1].abs().max())


def test_conv_refresh_refuses_bad_tensors(sd):
    from nomad_b200 import _lib
    from nomad_b200.engine import Engine
    a = Engine(sd, 0)
    dev = {k: v.cuda().contiguous() for k, v in sd.items() if k != "ssl_model.feature_extractor.conv_layers.3.0.weight"}
    with pytest.raises(_lib.NomadB200Error, match="conv_layers.3.0.weight"):
        a.refresh_conv_weights(dev)


def test_trainer_with_conv_encoder_trained(sd):
    """``TripletTrainer(freeze_convnet=False)``: four steps on one batch lower its loss, the conv master tensors move, and
    scoring afterwards equals a fresh model built from the trainer's master tensors."""
    from nomad_b200.nomad import Nomad
    from nomad_b200.triplet import TripletTrainer, triplet_loss_and_grads
    nomad = Nomad(state_dict=sd, keep_state_dict=True)
    tr = TripletTrainer(nomad, lr=1e-3, margin=MARGIN, lr_pretrained=1e-4, freeze_convnet=False)
    conv0 = {k: tr.master[k].detach().clone() for k in CONV_KEYS}
    A, P, Nn = _triplets(4, 6000, 5)
    losses = [tr.step(A, P, Nn) for _ in range(4)]
    final, _ = triplet_loss_and_grads(nomad.engine, tr.master, A, P, Nn, margin=MARGIN, freeze_convnet=False,
                                      feature_grad_mult=nomad.feature_grad_mult)
    assert final.item() < losses[0] - 1e-3, (losses, final.item())
    for k in CONV_KEYS:
        assert float((tr.master[k].detach() - conv0[k]).abs().max()) > 0.0, k
    fresh = Nomad(state_dict={k: v.detach().cpu() for k, v in tr.master.items()})
    assert float((nomad.model(A) - fresh.model(A)).abs().max()) <= 2e-6
