"""CPU checks of oracle/tc16.py, the fp16-faithful restatement of the tensor-core decoders.

With the fp16 rounding turned off the module must compute the exact decoders and their gradients: its outputs and gradients
are compared with FieldOracle's decoders differentiated by torch autograd, in float64, to ~1e-12.  With the rounding on, the
rounding helpers, the loss-scale reference and the operand-image layout are checked on hand-made values.
"""
import math

import pytest
import torch
from torch import nn

from oracle import tc16
from oracle.field import FieldOracle

TOL = 1e-11


class _Fixed(nn.Module):
    """A 'grid' that returns a fixed feature tensor (the decoders' input), whatever the coordinates."""

    def __init__(self, x):
        super().__init__()
        self.x = x

    def forward(self, coords):
        return self.x


def _rand_linear(out_f, in_f, gen, scale=1.0):
    w = (torch.rand(out_f, in_f, generator=gen, dtype=torch.float64) * 2 - 1) * (scale / in_f ** 0.5)
    b = (torch.rand(out_f, generator=gen, dtype=torch.float64) * 2 - 1) * 0.1
    return [w, b]


def _load(lin, w, b):
    with torch.no_grad():
        lin.weight.copy_(w)
        lin.bias.copy_(b)


def _field(IN, Cs, Ci, f, df, lodw, weights_dc, weights_pan, sem_softmax=True, inst_softmax=True, temperature=0.0):
    fo = FieldOracle(_Fixed(f), _Fixed(df) if df is not None else None, feat_dim=IN, num_classes=max(Cs, 1),
                     num_instances=max(Ci, 1), sem_softmax=sem_softmax, inst_softmax=inst_softmax,
                     inst_soft_temperature=temperature).double()
    fo.lod_weights = lodw
    if weights_dc is not None:
        w = weights_dc
        _load(fo.decoder_density.layers[0], w[0], w[1]); _load(fo.decoder_density.lout, w[2], w[3])
        _load(fo.decoder_color.layers[0], w[4], w[5]); _load(fo.decoder_color.layers[1], w[6], w[7])
        _load(fo.decoder_color.lout, w[8], w[9])
    if weights_pan is not None:
        w = weights_pan
        _load(fo.decoder_semantics.layers[0], w[0], w[1]); _load(fo.decoder_semantics.lout, w[2], w[3])
        _load(fo.decoder_inst.layers[0], w[4], w[5]); _load(fo.decoder_inst.layers[1], w[6], w[7])
        _load(fo.decoder_inst.lout, w[8], w[9])
    return fo


def _close(a, b, msg):
    a, b = a.double(), b.double()
    assert a.shape == b.shape, msg
    err = float((a - b).abs().max()) if a.numel() else 0.0
    assert err <= TOL * max(1.0, float(b.abs().max()) if b.numel() else 0.0), f"{msg}: max err {err:.3e}"


def _dc_weights(IN, gen):
    return _rand_linear(64, IN, gen) + _rand_linear(16, 64, gen) + _rand_linear(64, 43, gen) + _rand_linear(64, 64, gen) + \
        _rand_linear(3, 64, gen)


def _pan_weights(IN, Cs, Ci, gen):
    return _rand_linear(64, IN, gen) + _rand_linear(max(Cs, 1), 64, gen, 4.0) + _rand_linear(64, IN, gen) + \
        _rand_linear(64, 64, gen) + _rand_linear(max(Ci, 1), 64, gen, 4.0)


@pytest.mark.parametrize("IN,S,lod,g_sigma,g_rgb", [(12, 1, True, True, True), (48, 4, False, True, True),
                                                     (4, 2, True, False, True), (64, 1, True, True, False)])
def test_dc_exact_equals_autograd(IN, S, lod, g_sigma, g_rgb):
    gen = torch.Generator().manual_seed(IN * 10 + S)
    R = 37
    M = R * S
    w = _dc_weights(IN, gen)
    f = torch.randn(M, IN, generator=gen, dtype=torch.float64)
    lodw = torch.rand(IN, generator=gen, dtype=torch.float64) + 0.5 if lod else torch.ones(IN, dtype=torch.float64)
    d = nn.functional.normalize(torch.randn(R, 3, generator=gen, dtype=torch.float64), dim=-1)
    gs = torch.randn(M, generator=gen, dtype=torch.float64) if g_sigma else None
    gr = torch.randn(M, 3, generator=gen, dtype=torch.float64) if g_rgb else None

    fl = f.clone().requires_grad_(True)
    dl = d.clone().requires_grad_(True)
    fo = _field(IN, 1, 1, fl, None, lodw, w, None)
    out = fo(torch.zeros(R, S, 3, dtype=torch.float64), dl, {'density', 'rgb'})
    loss = 0
    if gs is not None:
        loss = loss + (out['density'].reshape(-1) * gs).sum()
    if gr is not None:
        loss = loss + (out['rgb'].reshape(-1, 3) * gr).sum()
    loss.backward()

    ray_rows = d.repeat_interleave(S, 0)
    fw = tc16.dc_forward(f, lodw if lod else None, ray_rows, w, want_rgb=True, fp16=False)
    _close(fw['sigma'], out['density'].reshape(-1).detach(), "sigma")
    _close(fw['rgb'], out['rgb'].reshape(-1, 3).detach(), "rgb")
    assert not fw['amb'].any()
    bw = tc16.dc_backward(fw, gs, gr, scale=8.0)
    params = [fo.decoder_density.layers[0], fo.decoder_density.lout, fo.decoder_color.layers[0], fo.decoder_color.layers[1],
              fo.decoder_color.lout]
    for i, lin in enumerate(params):
        for j, p in enumerate((lin.weight, lin.bias)):
            got = bw['grads'][2 * i + j]
            if i >= 2 and gr is None:
                assert got is None
                continue
            _close(got, p.grad if p.grad is not None else torch.zeros_like(p), f"grad {2 * i + j}")
    _close(bw['g_feats'], fl.grad, "g_feats")
    _close(bw['g_dir'].view(R, S, 3).sum(1), dl.grad if dl.grad is not None else torch.zeros_like(d), "g_dir")


@pytest.mark.parametrize("IN,Cs,Ci,softmax,temp,delta", [(12, 6, 20, True, 0.0, True), (48, 1, 129, False, 2.0, True),
                                                         (28, 32, 1, True, 0.5, False), (4, 16, 51, False, 0.0, True)])
def test_pan_exact_equals_autograd(IN, Cs, Ci, softmax, temp, delta):
    gen = torch.Generator().manual_seed(IN + Cs + Ci)
    M = 300
    w = _pan_weights(IN, Cs, Ci, gen)
    f = torch.randn(M, IN, generator=gen, dtype=torch.float64)
    df = torch.randn(M, IN, generator=gen, dtype=torch.float64) * 0.3 if delta else torch.zeros(M, IN, dtype=torch.float64)
    lodw = torch.rand(IN, generator=gen, dtype=torch.float64) + 0.5
    gs = torch.randn(M, Cs, generator=gen, dtype=torch.float64)
    gi = torch.randn(M, Ci, generator=gen, dtype=torch.float64)

    dfl = df.clone().requires_grad_(True)
    fo = _field(IN, Cs, Ci, f, dfl, lodw, None, w, softmax, softmax, temp)
    out = fo(torch.zeros(M, 1, 3, dtype=torch.float64), torch.zeros(M, 3, dtype=torch.float64), {'semantics', 'inst_embedding'})
    ((out['semantics'] * gs).sum() + (out['inst_embedding'] * gi).sum()).backward()

    fw = tc16.pan_forward(f, df if delta else None, lodw, w, Cs, Ci, softmax, softmax, temp, fp16=False)
    _close(fw['sem'], out['semantics'].detach(), "sem")
    _close(fw['inst'], out['inst_embedding'].detach(), "inst")
    bw = tc16.pan_backward(fw, gs, gi, scale=0.25)
    lins = [fo.decoder_semantics.layers[0], fo.decoder_semantics.lout, fo.decoder_inst.layers[0], fo.decoder_inst.layers[1],
            fo.decoder_inst.lout]
    for i, lin in enumerate(lins):
        _close(bw['grads'][2 * i], lin.weight.grad, f"grad W{i}")
        _close(bw['grads'][2 * i + 1], lin.bias.grad, f"grad b{i}")
    _close(bw['g_panop'], dfl.grad, "g_panop")


@pytest.mark.parametrize("IN,Cs,Ci,softmax,temp", [(12, 6, 20, True, 0.0), (48, 16, 208, True, 0.5), (4, 1, 51, False, 2.0)])
def test_comp_exact_equals_autograd(IN, Cs, Ci, softmax, temp):
    gen = torch.Generator().manual_seed(IN * 3 + Ci)
    M, N = 400, 60
    w = _pan_weights(IN, Cs, Ci, gen)
    f = torch.randn(M, IN, generator=gen, dtype=torch.float64)
    df = torch.randn(M, IN, generator=gen, dtype=torch.float64) * 0.3
    lodw = torch.rand(IN, generator=gen, dtype=torch.float64) + 0.5
    ridx = torch.sort(torch.randint(0, N, (M,), generator=gen)).values
    wgt = torch.rand(M, generator=gen, dtype=torch.float64)
    alpha = torch.rand(N, generator=gen, dtype=torch.float64)
    gs = torch.randn(N, Cs, generator=gen, dtype=torch.float64)
    gi = torch.randn(N, Ci, generator=gen, dtype=torch.float64)

    dfl = df.clone().requires_grad_(True)
    fo = _field(IN, Cs, Ci, f, dfl, lodw, None, w, softmax, softmax, temp)
    out = fo(torch.zeros(M, 1, 3, dtype=torch.float64), torch.zeros(M, 3, dtype=torch.float64), {'semantics', 'inst_embedding'})
    coef = (alpha[ridx] * wgt).requires_grad_(True)
    ref_s = torch.zeros(N, Cs, dtype=torch.float64).index_add(0, ridx, out['semantics'] * coef[:, None])
    ref_i = torch.zeros(N, Ci, dtype=torch.float64).index_add(0, ridx, out['inst_embedding'] * coef[:, None])
    # d out / d coef split per head: two backward passes
    gw_s, = torch.autograd.grad((ref_s * gs).sum(), coef, retain_graph=True)
    gw_i, = torch.autograd.grad((ref_i * gi).sum(), coef, retain_graph=True)
    ((ref_s * gs).sum() + (ref_i * gi).sum()).backward()

    fw = tc16.comp_forward(f, df, lodw, w, wgt, alpha, ridx, N, Cs, Ci, softmax, softmax, temp, fp16=False)
    _close(fw['sem'], ref_s.detach(), "sem")
    _close(fw['inst'], ref_i.detach(), "inst")
    if softmax:
        it = 1.0 / temp if temp > 0 else 1.0
        lse = torch.logsumexp(fo.decoder_inst(((f + df) * lodw)) * it, 1) / math.log(2.0)
        _close(fw['inst_lse'], lse.detach(), "inst_lse")
    bw = tc16.comp_backward(fw, gs, gi, scale=4.0)
    lins = [fo.decoder_semantics.layers[0], fo.decoder_semantics.lout, fo.decoder_inst.layers[0], fo.decoder_inst.layers[1],
            fo.decoder_inst.lout]
    for i, lin in enumerate(lins):
        _close(bw['grads'][2 * i], lin.weight.grad, f"grad W{i}")
        _close(bw['grads'][2 * i + 1], lin.bias.grad, f"grad b{i}")
    _close(bw['g_panop'], dfl.grad, "g_panop")
    _close(bw['gw_sem'], gw_s, "gw_sem")
    _close(bw['gw_inst'], gw_i, "gw_inst")


def test_rounding_points_are_fp16_and_flag_midpoints():
    num = tc16._Num(True, 4)
    x = torch.tensor([[1.0 + 2.0 ** -11], [1.0 + 3 * 2.0 ** -12], [0.1], [1e-9]], dtype=torch.float64)
    y = num.r(x)
    assert torch.equal(y, x.to(torch.float16).double())
    assert num.amb.tolist() == [True, False, False, False]     # row 0 is exactly the midpoint between 1 and 1 + 2^-10
    off = tc16._Num(False, 4)
    assert torch.equal(off.r(x), x) and not off.amb.any()


def test_relu_flag_is_relative_to_the_terms():
    num = tc16._Num(True, 2)
    X = torch.tensor([[1.0, 1.0], [1.0, 0.5]], dtype=torch.float64)
    W = torch.tensor([[1.0, -1.0]], dtype=torch.float64)
    pre, sa = num.lin(X, W, None)
    m = num.relu_mask(pre, sa)
    assert m[:, 0].tolist() == [False, True]
    assert num.amb.tolist() == [True, False]


def test_grad_scale_reference():
    t = lambda *v: torch.tensor(v, dtype=torch.float64)
    assert tc16.grad_scale(1024.0, t(1.0, -3.0)) == 256.0             # 1024 / 3 = 341.3 -> 2^8
    assert tc16.grad_scale(1024.0, t(4.0)) == 256.0                   # exactly a power of two
    assert tc16.grad_scale(1024.0, t(4.0 * (1 + 2.0 ** -40))) == 128.0   # just above: the next power down
    assert tc16.grad_scale(1024.0, t(0.0, 0.0)) == 2.0 ** 60          # all zero: clamped
    assert tc16.grad_scale(1024.0, t(float('nan'), 2.0)) == 512.0      # NaN ignored
    assert tc16.grad_scale(1024.0, t(float('inf'), 2.0)) == 2.0 ** -24
    assert tc16.grad_scale(1024.0, t(1.0), t(8.0)) == 128.0


def test_image16_layout_round_trip():
    M, IN = 300, 12
    x = torch.randn(M, IN).half()
    img = tc16.image16(x, IN)
    assert img.shape == (3, 2, 128, 8)
    assert torch.equal(img[1, 1, 5, 3], x[128 + 5, 8 + 3])
    assert torch.equal(img[2, 1, 50:, :], torch.zeros_like(img[2, 1, 50:, :]))
    assert torch.equal(img[0, 1, :, 4:], torch.zeros_like(img[0, 1, :, 4:]))    # features 12..15 are padding
    assert torch.equal(tc16.from_image16(img, M, IN), x)
