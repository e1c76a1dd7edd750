"""Autograd through ``lossnet_layers``, ``model`` and ``forward`` (with ``clean.requires_grad``): the waveform gradient
of any use of the 12 layer outputs and the embedding, against the oracle's CPU autograd (``feature_grad_mult`` as
fairseq's GradMultiply).  Every comparison records the error it achieved (conftest ``record``).  Tolerances, in line
with the loss tests (fp16 operands in the backward): gradient max error <= 0.6 % of max|grad| and cosine >= 0.99998
(achieved on a B200: at most 0.39 % and at least 0.999993, profiles/r04_autograd_achieved.jsonl)."""
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

MAX_ERR = 6e-3
MIN_COS = 0.99998


@pytest.fixture(scope="module")
def nomad(state_dict):
    from nomad_b200.nomad import Nomad
    torch.set_num_threads(os.cpu_count() or 1)
    return Nomad(state_dict=state_dict)


def _head(nomad):
    lin = nomad.lossnet_layers.embedding_layer[1]
    return lin.weight.detach().cpu(), lin.bias.detach().cpu()


def _errors(got, ref):
    got, ref = np.asarray(got, np.float64).ravel(), np.asarray(ref, np.float64).ravel()
    max_rel = float(np.abs(got - ref).max() / np.abs(ref).max())
    cos = float((got * ref).sum() / (np.linalg.norm(got) * np.linalg.norm(ref)))
    return max_rel, cos


def _lossnet_grads(nomad, state_dict, wav, use, fgm):
    """wav.grad of use(lossnet_layers(wav)) on the GPU and with the oracle; ``use(outs, device)`` -> scalar."""
    from oracle import w2v_oracle as O
    nomad.feature_grad_mult = fgm
    w = wav.cuda().requires_grad_(True)
    use(nomad.lossnet_layers(w), "cuda").backward()
    hw, hb = _head(nomad)
    wc = wav.clone().requires_grad_(True)
    use(O.lossnet_layers(state_dict, hw, hb, wc, feature_grad_mult=fgm), "cpu").backward()
    return w.grad.cpu().numpy(), wc.grad.numpy()


def _cotangents(B, T, seed):
    g = torch.Generator().manual_seed(seed)
    return [torch.randn(B, T, 768, generator=g) for _ in range(12)] + [torch.randn(B, 256, generator=g)]


def _dot(cots):
    return lambda outs, dev: sum((o * c.to(dev)).sum() for o, c in zip(outs, cots) if c is not None)


@pytest.mark.parametrize("fgm", [1.0, 0.1])
@pytest.mark.parametrize("B,N", [(1, 400), (3, 16384), (2, 32000)])
def test_random_cotangents_on_all_outputs(nomad, state_dict, B, N, fgm, record):
    g = torch.Generator().manual_seed(B * 7 + N)
    wav = 0.1 * torch.randn(B, N, generator=g)
    T = nomad.engine.num_frames(N)
    got, ref = _lossnet_grads(nomad, state_dict, wav, _dot(_cotangents(B, T, N)), fgm)
    max_rel, cos = _errors(got, ref)
    record("autograd_all_outputs", B=B, N=N, fgm=fgm, grad_max_err_over_max=max_rel, grad_cosine=cos)
    assert got.shape == (B, N) and np.isfinite(got).all()
    assert max_rel <= MAX_ERR and cos >= MIN_COS


@pytest.mark.parametrize("case", ["layer5", "embedding", "mse_9_11"])
def test_sparse_use_of_the_outputs(nomad, state_dict, case, record):
    B, N = 2, 16000
    g = torch.Generator().manual_seed(11)
    wav = 0.1 * torch.randn(B, N, generator=g)
    T = nomad.engine.num_frames(N)
    cots = _cotangents(B, T, 5)
    if case == "layer5":
        use = _dot([None] * 5 + [cots[5]] + [None] * 7)
    elif case == "embedding":
        use = _dot([None] * 12 + [cots[12]])
    else:
        use = lambda outs, dev: sum(F.mse_loss(outs[i], 0.5 * cots[i].to(dev)) for i in (9, 10, 11))
    got, ref = _lossnet_grads(nomad, state_dict, wav, use, 0.1)
    max_rel, cos = _errors(got, ref)
    record("autograd_sparse", case=case, grad_max_err_over_max=max_rel, grad_cosine=cos)
    assert max_rel <= MAX_ERR and cos >= MIN_COS


@pytest.mark.parametrize("fgm", [1.0, 0.1])
def test_reference_composition_with_estimate_only(nomad, golden_dir, fgm, record):
    """``nomad_loss(lossnet_layers(clean), lossnet_layers(est))`` with only ``est`` requiring grad, against the reference
    run and against the fused ``nomad.forward``."""
    gz = np.load(os.path.join(golden_dir, "ref_loss.npz"))
    lin = nomad.lossnet_layers.embedding_layer[1]
    with torch.no_grad():
        lin.weight.copy_(torch.from_numpy(gz["head_w"]))
        lin.bias.copy_(torch.from_numpy(gz["head_b"]))
    nomad.feature_grad_mult = fgm
    clean = torch.from_numpy(gz["clean"]).cuda()
    est = torch.from_numpy(gz["est"]).cuda().requires_grad_(True)
    loss = nomad.nomad_loss(nomad.lossnet_layers(clean), nomad.lossnet_layers(est))
    loss.backward()
    est2 = est.detach().clone().requires_grad_(True)
    fused = nomad.forward(est2, clean)
    fused.backward()
    ref_l, ref_g = float(gz[f"loss_fgm{fgm}"]), gz[f"grad_fgm{fgm}"]
    got = est.grad.cpu().numpy()
    max_rel, cos = _errors(got, ref_g)
    max_rel_f, cos_f = _errors(got, est2.grad.cpu().numpy())
    rel_loss = abs(loss.item() - ref_l) / ref_l
    record("autograd_composition_est_only", fgm=fgm, loss_rel_err=rel_loss, grad_max_err_over_max=max_rel, grad_cosine=cos,
           vs_fused_loss_rel=abs(loss.item() - fused.item()) / ref_l, vs_fused_grad_max_err_over_max=max_rel_f,
           vs_fused_grad_cosine=cos_f)
    assert rel_loss <= 1e-3 and abs(loss.item() - fused.item()) <= 1e-3 * ref_l
    assert max_rel <= MAX_ERR and cos >= MIN_COS
    assert max_rel_f <= MAX_ERR and cos_f >= MIN_COS


def test_gradient_to_clean(nomad, state_dict, record):
    from oracle import w2v_oracle as O
    nomad.feature_grad_mult = 0.1
    B, N = 2, 16000
    g = torch.Generator().manual_seed(23)
    clean = 0.1 * torch.randn(B, 1, N, generator=g)
    est = clean + 0.05 * torch.randn(B, 1, N, generator=g)
    e, c = est.cuda().requires_grad_(True), clean.cuda().requires_grad_(True)
    loss = nomad.forward(e, c)
    loss.backward()
    hw, hb = _head(nomad)
    ec, cc = est.clone().requires_grad_(True), clean.clone().requires_grad_(True)
    lo = O.nomad_forward(state_dict, hw, hb, ec, cc, feature_grad_mult=0.1)
    lo.backward()
    rel_loss = abs(loss.item() - lo.item()) / lo.item()
    me, ce = _errors(e.grad.cpu().numpy(), ec.grad.numpy())
    mc, cc_ = _errors(c.grad.cpu().numpy(), cc.grad.numpy())
    record("autograd_grad_to_clean", loss_rel_err=rel_loss, est_grad_max_err_over_max=me, est_grad_cosine=ce,
           clean_grad_max_err_over_max=mc, clean_grad_cosine=cc_)
    assert rel_loss <= 1e-3
    assert me <= MAX_ERR and ce >= MIN_COS and mc <= MAX_ERR and cc_ >= MIN_COS
    # clean without grad: the fused CUDA-graph step, as many launches as a direct loss step, no gradient to clean
    c2 = clean.cuda()
    e2 = est.cuda().requires_grad_(True)
    for _ in range(3):  # eager, capture, replay
        nomad.forward(e2, c2).backward()
    n0 = nomad.engine.launch_count()
    nomad.forward(e2, c2).backward()
    n_fwd = nomad.engine.launch_count() - n0
    n0 = nomad.engine.launch_count()
    nomad.engine.loss_fwd_bwd(e2, c2, nomad.feature_grad_mult)
    assert n_fwd == nomad.engine.launch_count() - n0
    assert c2.grad is None and e2.grad is not None


@pytest.mark.parametrize("fgm", [1.0, 0.1])
def test_model_embedding_gradient(nomad, state_dict, fgm, record):
    from oracle import w2v_oracle as O
    nomad.feature_grad_mult = fgm
    B, N = 3, 24000
    g = torch.Generator().manual_seed(31)
    wav = 0.1 * torch.randn(B, 1, N, generator=g)
    c = torch.randn(B, 256, generator=g)
    w = wav.cuda().requires_grad_(True)
    emb = nomad.model(w)
    (emb * c.cuda()).sum().backward()
    wc = wav.clone().requires_grad_(True)
    layers = O.ssl_layers(state_dict, wc, feature_grad_mult=fgm)
    ref_emb = O.head(layers[-1], state_dict["embedding_layer.1.weight"], state_dict["embedding_layer.1.bias"])
    (ref_emb * c).sum().backward()
    emb_err = float((emb.detach().cpu() - ref_emb.detach()).abs().max())
    max_rel, cos = _errors(w.grad.cpu().numpy(), wc.grad.numpy())
    record("autograd_model", fgm=fgm, emb_max_abs_err=emb_err, grad_max_err_over_max=max_rel, grad_cosine=cos)
    assert w.grad.shape == wav.shape
    assert emb_err <= 1e-3 and max_rel <= MAX_ERR and cos >= MIN_COS


def test_gradient_scale_invariance(nomad):
    """The scale S is a power of two picked on the device from max|g|: scaling every cotangent by 2^k scales the
    gradient by exactly 2^k."""
    nomad.feature_grad_mult = 0.1
    B, N = 2, 16000
    wav = (0.1 * torch.randn(B, N, generator=torch.Generator().manual_seed(3))).cuda()
    cots = _cotangents(B, nomad.engine.num_frames(N), 9)

    def grad(scale):
        w = wav.clone().requires_grad_(True)
        _dot([c * scale for c in cots])(nomad.lossnet_layers(w), "cuda").backward()
        return w.grad

    g0 = grad(1.0)
    assert float(g0.abs().max()) > 0
    for k in (-20, 12):
        assert torch.equal(grad(2.0 ** k), g0 * 2.0 ** k), k
    gz = grad(0.0)
    assert torch.isfinite(gz).all() and float(gz.abs().max()) == 0.0


def test_saved_state_lifetime(nomad):
    nomad.feature_grad_mult = 0.1
    B, N = 2, 16000
    g = torch.Generator().manual_seed(41)
    wa, wb = (0.1 * torch.randn(B, N, generator=g)).cuda(), (0.1 * torch.randn(B, N, generator=g)).cuda()
    cots = _cotangents(B, nomad.engine.num_frames(N), 13)
    use = _dot(cots)

    def alone(wav):
        w = wav.clone().requires_grad_(True)
        use(nomad.lossnet_layers(w), "cuda").backward()
        return w.grad

    ref_a, ref_b = alone(wa), alone(wb)
    # two forwards, backwards in reverse order, an unrelated embed in between
    a, b = wa.clone().requires_grad_(True), wb.clone().requires_grad_(True)
    la, lb = use(nomad.lossnet_layers(a), "cuda"), use(nomad.lossnet_layers(b), "cuda")
    nomad.engine.embed([torch.randn(48000), torch.randn(20000)])
    lb.backward()
    la.backward()
    assert torch.equal(a.grad, ref_a) and torch.equal(b.grad, ref_b)
    # the head is snapshotted at the forward: a new head synced before the backward does not change the gradient
    lin = nomad.lossnet_layers.embedding_layer[1]
    a = wa.clone().requires_grad_(True)
    la = use(nomad.lossnet_layers(a), "cuda")
    old = (lin.weight.detach().clone(), lin.bias.detach().clone())
    with torch.no_grad():
        lin.weight.mul_(-2.0)
        lin.bias.add_(0.5)
    nomad.lossnet_layers(wb)  # syncs the new head into the engine
    la.backward()
    with torch.no_grad():
        lin.weight.copy_(old[0])
        lin.bias.copy_(old[1])
    assert torch.equal(a.grad, ref_a)


def test_no_grad_paths_are_unchanged(nomad):
    B, N = 3, 16000
    wav = (0.1 * torch.randn(B, N, generator=torch.Generator().manual_seed(4))).cuda()
    nomad.lossnet_layers.sync_head()
    layers, emb = nomad.engine.layers(wav)
    ref = [layers[i] for i in range(12)] + [emb]
    ref_emb = nomad.engine.embed_packed(wav.reshape(-1), np.arange(B + 1, dtype=np.int64) * N)
    w = wav.clone().requires_grad_(True)
    with torch.no_grad():
        for got in (nomad.lossnet_layers(w), nomad.lossnet_layers(wav)):
            assert all(torch.equal(x, y) and not x.requires_grad for x, y in zip(got, ref))
        assert torch.equal(nomad.model(w), ref_emb)
    got = nomad.lossnet_layers(wav)
    assert all(torch.equal(x, y) and not x.requires_grad for x, y in zip(got, ref))
    assert torch.equal(nomad.model(wav), ref_emb) and not nomad.model(wav).requires_grad


def test_differentiable_outputs_match_the_forward(nomad):
    """The save-mode forward returns the same layer outputs and embedding as the scoring forward (within fp16-operand
    rounding), and head 1 without a loss head is refused."""
    B, N = 2, 20000
    wav = (0.1 * torch.randn(B, N, generator=torch.Generator().manual_seed(6))).cuda()
    ref = nomad.lossnet_layers(wav)
    got = nomad.lossnet_layers(wav.clone().requires_grad_(True))
    assert len(got) == 13 and all(x.requires_grad and x.shape == y.shape for x, y in zip(got, ref))
    assert max(float((x - y).abs().max()) for x, y in zip(got, ref)) <= 2e-2
    emb = nomad.model(wav.clone().requires_grad_(True))
    assert emb.requires_grad and float((emb - nomad.model(wav)).abs().max()) <= 1e-3
    from nomad_b200 import _lib
    from nomad_b200.engine import Engine
    from nomad_b200.weights import random_state_dict
    with pytest.raises(_lib.NomadB200Error, match="set_loss_head"):
        Engine(random_state_dict(2), 0).layers_fwd_save(wav, 1)
