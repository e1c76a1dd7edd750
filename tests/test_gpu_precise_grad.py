"""fp32-class waveform gradients (``precision='fp32'``): ``nomad.forward``, ``lossnet_layers`` and ``model`` with grad on,
against the oracle's autograd in fp64.  Each gradient comparison also measures, on the same input, the fp16-operand path
(the same handle switched to ``'fp16'``) and the reference's own fp32 CPU autograd, both against fp64: the fp32-class
error must be at most a tenth of the fp16 path's, and under a fixed bound set from the achieved errors on a B200 (see
DESIGN.md section 5e).  The loss value must be within 1e-5 relative of fp64 (BASELINE section 4).  Every figure goes to
the ``record`` log."""
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

LOSS_REL = 1e-5      # BASELINE section 4, fp32 mode
GRAD_REL = 2e-5      # max error / max|grad| of the fp32-class gradient against fp64 (achieved <= 8.3e-6)
FP16_RATIO = 0.1     # fp32-class error <= FP16_RATIO x the fp16 path's on the same input


@pytest.fixture(scope="module")
def nomad(state_dict):
    from nomad_b200.nomad import Nomad
    torch.set_num_threads(os.cpu_count() or 1)
    return Nomad(state_dict=state_dict, precision="fp32")


def _head(nomad):
    lin = nomad.lossnet_layers.embedding_layer[1]
    return lin.weight.detach().cpu(), lin.bias.detach().cpu()


def _err(got, ref):
    got, ref = np.asarray(got, np.float64).ravel(), np.asarray(ref, np.float64).ravel()
    return float(np.abs(got - ref).max() / np.abs(ref).max())


def _cotangents(B, T, seed):
    g = torch.Generator().manual_seed(seed)
    return [torch.randn(B, T, 768, generator=g) for _ in range(12)] + [torch.randn(B, 256, generator=g)]


def _dot(cots):
    return lambda outs, dev: sum((o * c.to(device=dev, dtype=o.dtype)).sum() for o, c in zip(outs, cots) if c is not None)


def _both_modes(nomad, fn):
    """fn() on the GPU in fp32 mode, then in fp16 mode on the same handle; the handle is left in fp32 mode."""
    got32 = fn()
    nomad.engine.set_precision("fp16")
    try:
        got16 = fn()
    finally:
        nomad.engine.set_precision("fp32")
    return got32, got16


def _check(name, record, got32, got16, ref32, ref64, **kw):
    e32, e16, floor = _err(got32, ref64), _err(got16, ref64), _err(ref32, ref64)
    record(name, fp32_class_err=e32, fp16_err=e16, reference_fp32_err=floor, **kw)
    assert np.isfinite(got32).all()
    assert e32 <= FP16_RATIO * e16, (e32, e16)
    assert e32 <= GRAD_REL, e32


def _lossnet_grad_gpu(nomad, wav, use):
    w = wav.cuda().requires_grad_(True)
    use(nomad.lossnet_layers(w), "cuda").backward()
    return w.grad.cpu().numpy()


def _lossnet_grad_ref(nomad, state_dict, wav, use, fgm, dtype):
    from oracle import w2v_oracle as O
    hw, hb = _head(nomad)
    wc = wav.to(dtype).clone().requires_grad_(True)
    use(O.lossnet_layers(state_dict, hw, hb, wc, dtype=dtype, feature_grad_mult=fgm), "cpu").backward()
    return wc.grad.numpy()


# ------------------------------------------------------------------------------------------------------------ loss value
@pytest.mark.parametrize("fgm", [1.0, 0.1])
def test_loss_value_and_gradient_on_the_reference_fixture(nomad, state_dict, golden_dir, fgm, record):
    from oracle import w2v_oracle as O
    gz = np.load(os.path.join(golden_dir, "ref_loss.npz"))
    lin = nomad.lossnet_layers.embedding_layer[1]
    with torch.no_grad():
        lin.weight.copy_(torch.from_numpy(gz["head_w"]))
        lin.bias.copy_(torch.from_numpy(gz["head_b"]))
    nomad.feature_grad_mult = fgm
    est, clean = torch.from_numpy(gz["est"]), torch.from_numpy(gz["clean"])

    def run():
        e = est.cuda().requires_grad_(True)
        loss = nomad.forward(e, clean.cuda())
        loss.backward()
        return loss.item(), e.grad.cpu().numpy()

    (l32, g32), (l16, g16) = _both_modes(nomad, run)
    hw, hb = _head(nomad)
    e64 = est.double().requires_grad_(True)
    ref = O.nomad_forward(state_dict, hw, hb, e64, clean.double(), dtype=torch.float64, feature_grad_mult=fgm)
    ref.backward()
    l64 = ref.item()
    ref32, g_ref32 = float(gz[f"loss_fgm{fgm}"]), gz[f"grad_fgm{fgm}"]
    rel = abs(l32 - l64) / l64
    record("precise_loss_fixture", fgm=fgm, loss_rel_err=rel, fp16_loss_rel_err=abs(l16 - l64) / l64,
           reference_fp32_loss_rel_err=abs(ref32 - l64) / l64)
    assert rel <= LOSS_REL
    _check("precise_loss_fixture_grad", record, g32, g16, g_ref32, e64.grad.numpy(), fgm=fgm)


_BIG_REF = {}


@pytest.mark.parametrize("fgm", [1.0, 0.1])
def test_loss_value_32x2s(nomad, state_dict, fgm, record):
    """BASELINE C4's loss batch; the value does not depend on feature_grad_mult, the gradient path does."""
    from oracle import w2v_oracle as O
    nomad.feature_grad_mult = fgm
    g = torch.Generator().manual_seed(77)
    clean = 0.1 * torch.randn(32, 1, 32000, generator=g)
    est = clean + 0.05 * torch.randn(32, 1, 32000, generator=g)
    e = est.cuda().requires_grad_(True)
    loss = nomad.forward(e, clean.cuda())
    loss.backward()
    if "l64" not in _BIG_REF:
        hw, hb = _head(nomad)
        with torch.no_grad():
            _BIG_REF["l64"] = O.nomad_forward(state_dict, hw, hb, est.double(), clean.double(), dtype=torch.float64).item()
    rel = abs(loss.item() - _BIG_REF["l64"]) / _BIG_REF["l64"]
    record("precise_loss_32x2s", fgm=fgm, loss_rel_err=rel)
    assert rel <= LOSS_REL
    assert torch.isfinite(e.grad).all() and float(e.grad.abs().max()) > 0


# ------------------------------------------------------------------------------------------------------------ gradients
@pytest.mark.parametrize("fgm", [1.0, 0.1])
@pytest.mark.parametrize("B,N", [(1, 400), (3, 16384), (2, 32000)])
def test_random_cotangents_on_all_outputs(nomad, state_dict, B, N, fgm, record):
    g = torch.Generator().manual_seed(B * 7 + N)
    wav = 0.1 * torch.randn(B, N, generator=g)
    use = _dot(_cotangents(B, nomad.engine.num_frames(N), N))
    nomad.feature_grad_mult = fgm
    g32, g16 = _both_modes(nomad, lambda: _lossnet_grad_gpu(nomad, wav, use))
    r32 = _lossnet_grad_ref(nomad, state_dict, wav, use, fgm, torch.float32)
    r64 = _lossnet_grad_ref(nomad, state_dict, wav, use, fgm, torch.float64)
    assert g32.shape == (B, N)
    _check("precise_all_outputs", record, g32, g16, r32, r64, B=B, N=N, fgm=fgm)


def test_model_embedding_gradient(nomad, state_dict, record):
    from oracle import w2v_oracle as O
    nomad.feature_grad_mult = 0.1
    B, N = 3, 24000
    g = torch.Generator().manual_seed(31)
    wav = 0.1 * torch.randn(B, 1, N, generator=g)
    c = torch.randn(B, 256, generator=g)

    def run():
        w = wav.cuda().requires_grad_(True)
        (nomad.model(w) * c.cuda()).sum().backward()
        return w.grad.cpu().numpy()

    g32, g16 = _both_modes(nomad, run)
    refs = []
    for dt in (torch.float32, torch.float64):
        wc = wav.to(dt).clone().requires_grad_(True)
        layers = O.ssl_layers(state_dict, wc, dtype=dt, feature_grad_mult=0.1)
        emb = O.head(layers[-1], state_dict["embedding_layer.1.weight"], state_dict["embedding_layer.1.bias"])
        (emb * c.to(dt)).sum().backward()
        refs.append(wc.grad.numpy())
    _check("precise_model", record, g32, g16, refs[0], refs[1])


def test_gradient_to_clean(nomad, state_dict, record):
    from oracle import w2v_oracle as O
    nomad.feature_grad_mult = 0.1
    B, N = 2, 16000
    g = torch.Generator().manual_seed(23)
    clean = 0.1 * torch.randn(B, 1, N, generator=g)
    est = clean + 0.05 * torch.randn(B, 1, N, generator=g)

    def run():
        e, c = est.cuda().requires_grad_(True), clean.cuda().requires_grad_(True)
        loss = nomad.forward(e, c)
        loss.backward()
        return loss.item(), e.grad.cpu().numpy(), c.grad.cpu().numpy()

    (l32, e32, c32), (_, e16, c16) = _both_modes(nomad, run)
    hw, hb = _head(nomad)
    refs = []
    for dt in (torch.float32, torch.float64):
        ec, cc = est.to(dt).clone().requires_grad_(True), clean.to(dt).clone().requires_grad_(True)
        lo = O.nomad_forward(state_dict, hw, hb, ec, cc, dtype=dt, feature_grad_mult=0.1)
        lo.backward()
        refs.append((lo.item(), ec.grad.numpy(), cc.grad.numpy()))
    rel = abs(l32 - refs[1][0]) / refs[1][0]
    record("precise_composition_loss", loss_rel_err=rel)
    assert rel <= LOSS_REL
    _check("precise_composition_est", record, e32, e16, refs[0][1], refs[1][1])
    _check("precise_composition_clean", record, c32, c16, refs[0][2], refs[1][2])


# tile edges: T0 (conv0 frames) = 64 k +- 1, frame counts T = 64 k +- 1 (attention tiles), and one 10 s utterance
_EDGE_N = [5 * (127 - 1) + 10, 5 * (129 - 1) + 10, 5 * (255 - 1) + 10, 20240, 20880, 40720, 41360, 160000]


@pytest.mark.parametrize("N", _EDGE_N)
def test_tile_edges(nomad, state_dict, N, record):
    nomad.feature_grad_mult = 0.1
    B = 1 if N >= 160000 else 2
    g = torch.Generator().manual_seed(N)
    wav = 0.1 * torch.randn(B, N, generator=g)
    T = nomad.engine.num_frames(N)
    use = _dot(_cotangents(B, T, N + 1))
    g32, g16 = _both_modes(nomad, lambda: _lossnet_grad_gpu(nomad, wav, use))
    r32 = _lossnet_grad_ref(nomad, state_dict, wav, use, 0.1, torch.float32)
    r64 = _lossnet_grad_ref(nomad, state_dict, wav, use, 0.1, torch.float64)
    _check("precise_tile_edges", record, g32, g16, r32, r64, N=N, T0=(N - 10) // 5 + 1, T=T)


# ------------------------------------------------------------------------------------------------------------ exactness
def test_scale_invariance_zeros_and_retain_graph(nomad):
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
    # one saved forward, differentiated twice
    w = wav.clone().requires_grad_(True)
    y = _dot(cots)(nomad.lossnet_layers(w), "cuda")
    first = torch.autograd.grad(y, w, retain_graph=True)[0]
    second = torch.autograd.grad(y, w)[0]
    assert torch.equal(first, second) and torch.equal(first, g0)


# ------------------------------------------------------------------------------------------------------------ mode safety
def test_backward_after_a_precision_switch_is_refused(nomad):
    from nomad_b200 import _lib
    B, N = 1, 8000
    w = (0.1 * torch.randn(B, N, generator=torch.Generator().manual_seed(5))).cuda().requires_grad_(True)
    y = nomad.model(w).sum()
    nomad.engine.set_precision("fp16")
    try:
        with pytest.raises(_lib.NomadB200Error, match="precision_mode 1"):
            y.backward()
    finally:
        nomad.engine.set_precision("fp32")


def test_alternating_fused_loss_modes(nomad):
    """fp16 steps go through the CUDA-graph cache (eager, capture, replay), fp32 steps run eagerly on the same handle:
    every step reproduces its mode's first result bit for bit, and the fp16 step keeps its launch count."""
    nomad.feature_grad_mult = 0.1
    g = torch.Generator().manual_seed(19)
    clean = (0.1 * torch.randn(4, 16000, generator=g)).cuda()
    est = clean + 0.05 * torch.randn(4, 16000, generator=g).cuda()
    eng = nomad.engine

    def step(mode):
        eng.set_precision(mode)
        n0 = eng.launch_count()
        loss, grad = eng.loss_fwd_bwd(est, clean, 0.1)
        torch.cuda.synchronize()
        return loss.clone(), grad.clone(), eng.launch_count() - n0

    try:
        first = {"fp16": step("fp16"), "fp32": step("fp32")}
        launches16 = []
        for i in range(4):
            for mode in ("fp16", "fp32"):
                loss, grad, n = step(mode)
                assert torch.equal(loss, first[mode][0]) and torch.equal(grad, first[mode][1]), (i, mode)
                if mode == "fp16":
                    launches16.append(n)
        assert len(set(launches16)) == 1 and launches16[0] == first["fp16"][2]
        assert not torch.equal(first["fp16"][1], first["fp32"][1])
    finally:
        eng.set_precision("fp32")
