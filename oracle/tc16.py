"""Oracle: the tensor-core decoders' fp16 numerics restated in float64.  TEST INFRASTRUCTURE ONLY.

The three kernel families of csrc/decoder_tc.cu and csrc/decoder_tc_fused.cu, forward and backward: the density / colour
decoders (`dc_*`), the modular semantic / instance heads (`pan_*`) and the heads fused with their compositing (`comp_*`).
Every value is rounded to fp16 exactly where the kernel rounds it; everything else (tensor-core products of fp16 operands,
their fp32 accumulation, softmax, unscaling) is computed in float64.  The kernel and this module then differ only by fp32
rounding and summation order, so tests can hold the kernels to a tight bar.  `fp16=False` turns every rounding into the
identity: the functions then compute the exact gradients of the decoders (tests/test_host_tc16.py checks them against
FieldOracle and torch autograd).

Rounding points (r16 = round to fp16, nearest even; s = the power-of-two loss scale the backward receives):
  * operand tiles
    - density / colour and fused heads: X = r16(f) or r16(f + df) from f32 rows (stage_x_coalesced / xpfc_consume); the LOD
      weights are folded into the first-layer weight image, r16(W1 * lodw) (stage_w16's colscale);
    - modular heads: X = r16((f + df) * lodw) (stage_x) with unweighted first-layer weights;
    - fp16 operand-image input: X = f16 (+ df16 added in fp16, tile_add16).
  * weights r16(W); biases fp32.  Hidden activations r16(relu(acc + b)) (epi_relu16 / epi_relu64).  Colour input
    [r16(y[0:16]) | r16(PE(-d)) | 0] (stage_cin_pe: view_embed in fp32 then r16; pag_view_pe16 stores the same fp16 values).
  * outputs: sigma = relu(y0), rgb = sigmoid(c) in fp32.  Modular heads: fp32 softmax of z / T (temperature as 1 / T, T = 0
    means 1), z / T without softmax.  Fused forward: every probability (or z / T, or the semantic logit without softmax) is
    rounded to fp16 before the weighted segment sum out[ray] += alpha[ray] w[m] p (comp_block); inst_lse = log2(sum 2^(z/T
    log2 e)), i.e. the natural log-sum-exp of z / T divided by ln 2.
  * backward: the upstream gradient is multiplied by s and every gradient tile is r16 of its scaled value:
    - dc: G3 = r16(g_rgb sg (1 - sg) s); G2, G1 = r16(mask * (G W)); Gy = r16(d cin[0:16] + [y0 > 0] g_sigma s);
      Gd = r16(mask * (Gy Wd2)).  Every bias gradient comes from a ones tile: the column sum of the fp16 tile.
    - modular heads: head dz = r16((p (g - <p, g>) or g) / T * s); Gs1, G2, G1 = r16(mask * (G W)).  Every bias gradient is
      the fp32 sum of the UNROUNDED values (warp reductions, head_grad_tile / epi_grad64).
    - fused: g_inst rows are cached (first 16 rays of a tile) or loaded (the others) as r16(g * s); p = 2^(z/T log2 e - lse)
      from the forward's lse; Gi = r16(c p (gc - <p, gc>) / T) with c = alpha[ray] w[m]; the semantic gradient is not cached
      in f32-row mode: Gs = r16(c s p (g - <p, g>)) with fp32 g and p.  Bias gradients: semantic L1/L2 and instance L1 are
      fp32 sums of unrounded values (grad16_store / epi_grad16), instance L2/L3 come from ones tiles (sums of the fp16 tiles).
    - weight and bias gradients are fp32 sums divided by s; first-layer weight gradients of dc / fused are G^T X with the
      unweighted X, multiplied by lodw afterwards (the kernels' flush).
    - dX = G W1 / s (dc and fused: with W1 = r16(W1 lodw); modular: (G W1) lodw / s).  In image mode dX is r16(G W1), an
      fp16 image that still carries s.
    - g_dir: d cin[16:43] through the derivative of PE(-d) in fp32, divided by s, per sample (the op sums it per ray).
    - DD outputs: gw_sem = <p_s, g_ray> (fp32 g, fp32 p), gw_inst = <p_s, r16(g_ray s)> / s, where p_s is the probability
      vector, or z (semantic) and z / T (instance) without softmax.

Ambiguity: a row whose reference pre-activation lies within AMB_RELU of 0 (relative to the sum of |terms| that produced it),
or one of whose fp16 roundings lies within AMB_MID of a rounding midpoint (relative to the value), can legitimately differ in
the kernel: fp32 accumulation order moves such a value across the boundary.  Every function returns `amb`, a bool [M] flag
of those rows.  Tests compare unflagged rows elementwise at a tight bar and bound the number of flagged rows.
"""
import math

import torch

from .decoders import PositionalEmbedderOracle

AMB_RELU = 2.0 ** -16
AMB_MID = 2.0 ** -26

_PE = PositionalEmbedderOracle(4).double()


def view_pe(ray_d):
    """PE(-d) [R, 27] in float64: [v, sin(2^f v), cos(2^f v)], v = -d (the layout of view_embed / FieldOracle's embedder)."""
    return _PE(-ray_d.double())


class _Num:
    """The fp16 rounding and the per-row ambiguity flags of one call."""

    def __init__(self, fp16, M):
        self.fp16 = fp16
        self.amb = torch.zeros(M, dtype=torch.bool)

    def r(self, x, rows=True):
        """r16(x); rows: x is [M, ...] and rows near a midpoint are flagged."""
        if not self.fp16:
            return x
        y = x.to(torch.float16).double()
        if rows and x.numel():
            ax = x.abs()
            ulp = torch.exp2(torch.floor(torch.log2(ax.clamp_min(2.0 ** -14))) - 10)
            near = (ulp / 2 - (x - y).abs()) <= AMB_MID * ax
            near &= ax > 0
            self.amb |= near.reshape(x.shape[0], -1).any(1)
        return y

    def relu_mask(self, pre, sumabs):
        """pre > 0, flagging rows with a pre-activation within AMB_RELU * sum|terms| of 0."""
        if self.fp16:
            self.amb |= (pre.abs() <= AMB_RELU * sumabs).any(1)
        return pre > 0

    def lin(self, x, W, b):
        """x W^T + b and the sum of |terms| (for the ReLU flag)."""
        y = x @ W.t()
        sa = x.abs() @ W.abs().t()
        if b is not None:
            y = y + b
            sa = sa + b.abs()
        return y, sa


def _d(t):
    return None if t is None else t.detach().double().cpu()


def _tc_weights(num, weights, lodw, fold=()):
    """r16 weight images and f64 biases; the weights at the indices `fold` (first layers) are multiplied by lodw first."""
    w = [_d(x) for x in weights]
    out = []
    for i in range(0, len(w), 2):
        W, b = w[i], w[i + 1]
        if i in fold and lodw is not None:
            W = W * lodw[None]
        out += [num.r(W, rows=False), b]
    return out


def _inv_temp(temperature):
    return 1.0 / temperature if temperature > 0 else 1.0


# ------------------------------------------------------------------------------------------------------------------------
# density + colour (dc_tc_fwd_kernel / dc_tc_bwd_kernel)
# ------------------------------------------------------------------------------------------------------------------------
def dc_forward(feats, lodw, ray_d, weights, want_rgb=True, fp16=True, img=False):
    """feats [M, IN] (f32 rows, or the fp16 values of an operand image with img=True), ray_d [M, 3] per SAMPLE,
    weights [Wd1, bd1, Wd2, bd2, Wc1, bc1, Wc2, bc2, Wc3, bc3] -> dict(sigma [M], y0 [M] (pre-activation), rgb [M, 3] or
    None, amb [M], ctx)."""
    f, lw, d = _d(feats), _d(lodw), _d(ray_d)
    M = f.shape[0]
    num = _Num(fp16, M)
    Wd1, bd1, Wd2, bd2, Wc1, bc1, Wc2, bc2, Wc3, bc3 = _tc_weights(num, weights, lw, (0,))
    X = f if img else num.r(f)
    pre_d, sa = num.lin(X, Wd1, bd1)
    mask_d = num.relu_mask(pre_d, sa)
    Hd = num.r(torch.relu(pre_d))
    y, sa = num.lin(Hd, Wd2, bd2)
    y0pos = num.relu_mask(y[:, :1], sa[:, :1])[:, 0]
    out = dict(sigma=torch.relu(y[:, 0]), y0=y[:, 0], rgb=None)
    ctx = dict(num=num, X=X, lw=lw, W=(Wd1, Wd2, Wc1, Wc2, Wc3), mask_d=mask_d, Hd=Hd, y0pos=y0pos, d=d)
    if want_rgb:
        pe = view_pe(d)
        cin = torch.cat([num.r(y), num.r(pe)], 1)
        pre1, sa = num.lin(cin, Wc1, bc1)
        mask_1 = num.relu_mask(pre1, sa)
        H1 = num.r(torch.relu(pre1))
        pre2, sa = num.lin(H1, Wc2, bc2)
        mask_2 = num.relu_mask(pre2, sa)
        H2 = num.r(torch.relu(pre2))
        c, _ = num.lin(H2, Wc3, bc3)
        out['rgb'] = torch.sigmoid(c)
        ctx.update(cin=cin, mask_1=mask_1, H1=H1, mask_2=mask_2, H2=H2, sg=out['rgb'])
    out['amb'] = num.amb
    out['ctx'] = ctx
    return out


def dc_backward(fwd, g_sigma, g_rgb, scale=1.0, need_feats=True, need_dir=True, img=False):
    """Backward of dc_forward(..., want_rgb=g_rgb is not None).  -> dict(grads [10] (colour entries None without g_rgb),
    g_feats [M, IN] (img: the fp16 image values, still times scale), g_dir [M, 3] per sample, amb [M])."""
    c = fwd['ctx']
    num = c['num']
    s = float(scale)
    Wd1, Wd2, Wc1, Wc2, Wc3 = c['W']
    M = c['X'].shape[0]
    gs = _d(g_sigma) if g_sigma is not None else torch.zeros(M, dtype=torch.float64)
    dy = torch.zeros(M, 16, dtype=torch.float64)
    grads = [None] * 10
    g_dir = None
    if g_rgb is not None:
        sg = c['sg']
        G3 = num.r(_d(g_rgb) * sg * (1 - sg) * s)
        grads[8], grads[9] = G3.t() @ c['H2'] / s, G3.sum(0) / s
        G2 = num.r((G3 @ Wc3) * c['mask_2'])
        grads[6], grads[7] = G2.t() @ c['H1'] / s, G2.sum(0) / s
        G1 = num.r((G2 @ Wc2) * c['mask_1'])
        grads[4], grads[5] = G1.t() @ c['cin'] / s, G1.sum(0) / s
        dcin = G1 @ Wc1
        dy = dcin[:, :16].clone()
        if need_dir:
            dd = c['d'].clone().requires_grad_(True)
            with torch.enable_grad():
                g_dir, = torch.autograd.grad(view_pe(dd), dd, dcin[:, 16:])
            g_dir = g_dir / s
    elif need_dir:
        g_dir = torch.zeros(M, 3, dtype=torch.float64)
    dy[:, 0] += torch.where(c['y0pos'], gs * s, torch.zeros_like(gs))
    Gy = num.r(dy)
    grads[2], grads[3] = Gy.t() @ c['Hd'] / s, Gy.sum(0) / s
    Gd = num.r((Gy @ Wd2) * c['mask_d'])
    lw = c['lw'] if c['lw'] is not None else 1.0
    grads[0], grads[1] = (Gd.t() @ c['X']) / s * lw, Gd.sum(0) / s
    g_feats = None
    if need_feats:
        g_feats = num.r(Gd @ Wd1) if img else (Gd @ Wd1) / s
    return dict(grads=grads, g_feats=g_feats, g_dir=g_dir, amb=num.amb)


# ------------------------------------------------------------------------------------------------------------------------
# modular semantic + instance heads (pan_tc_fwd_kernel / pan_tc_bwd_kernel)
# ------------------------------------------------------------------------------------------------------------------------
def _heads_forward(num, X, Ws1, bs1, Ws2, bs2, Wi1, bi1, Wi2, bi2, Wi3, bi3, Cs, Ci, inv_temp):
    ctx = {}
    if Cs:
        pre, sa = num.lin(X, Ws1, bs1)
        ctx['mask_s'] = num.relu_mask(pre, sa)
        ctx['Hs'] = num.r(torch.relu(pre))
        ctx['zs'] = num.lin(ctx['Hs'], Ws2, bs2)[0]
    if Ci:
        pre, sa = num.lin(X, Wi1, bi1)
        ctx['mask_1'] = num.relu_mask(pre, sa)
        ctx['H1'] = num.r(torch.relu(pre))
        pre, sa = num.lin(ctx['H1'], Wi2, bi2)
        ctx['mask_2'] = num.relu_mask(pre, sa)
        ctx['H2'] = num.r(torch.relu(pre))
        ctx['zi'] = num.lin(ctx['H2'], Wi3, bi3)[0] * inv_temp
    return ctx


def pan_forward(feats, dfeats, lodw, weights, Cs, Ci, sem_softmax, inst_softmax, temperature, fp16=True):
    """panop = (feats + dfeats) * lodw -> dict(sem [M, Cs] or None, inst [M, Ci] or None, amb [M], ctx).
    weights [Ws1, bs1, Ws2, bs2, Wi1, bi1, Wi2, bi2, Wi3, bi3] (torch Linear layout)."""
    f, df, lw = _d(feats), _d(dfeats), _d(lodw)
    num = _Num(fp16, f.shape[0])
    W = _tc_weights(num, weights, lw)
    p = f if df is None else f + df
    X = num.r(p * lw[None] if lw is not None else p)
    it = _inv_temp(temperature)
    ctx = _heads_forward(num, X, *W, Cs, Ci, it)
    ctx.update(num=num, X=X, lw=lw, W=W, it=it, ss=sem_softmax, si=inst_softmax)
    sem = (torch.softmax(ctx['zs'], 1) if sem_softmax else ctx['zs']) if Cs else None
    inst = (torch.softmax(ctx['zi'], 1) if inst_softmax else ctx['zi']) if Ci else None
    ctx.update(sem=sem, inst=inst)
    return dict(sem=sem, inst=inst, amb=num.amb, ctx=ctx)


def pan_backward(fwd, g_sem, g_inst, scale=1.0, need_panop=True):
    """-> dict(grads [10] (None for a head without gradient), g_panop [M, IN] (d/d feats = d/d dfeats), amb [M])."""
    c = fwd['ctx']
    num = c['num']
    s = float(scale)
    Ws1, _, Ws2, _, Wi1, _, Wi2, _, Wi3, _ = c['W']
    grads = [None] * 10
    dX = None
    if g_sem is not None and 'zs' in c:
        g, p = _d(g_sem), c['sem']
        dz = (p * (g - (p * g).sum(1, keepdim=True)) if c['ss'] else g) * s
        Gs = num.r(dz)
        grads[2], grads[3] = Gs.t() @ c['Hs'] / s, dz.sum(0) / s
        a = (Gs @ Ws2) * c['mask_s']
        Gs1 = num.r(a)
        grads[0], grads[1] = Gs1.t() @ c['X'] / s, a.sum(0) / s
        dX = Gs1 @ Ws1
    if g_inst is not None and 'zi' in c:
        g, p = _d(g_inst), c['inst']
        dz = (p * (g - (p * g).sum(1, keepdim=True)) if c['si'] else g) * c['it'] * s
        Gi = num.r(dz)
        grads[8], grads[9] = Gi.t() @ c['H2'] / s, dz.sum(0) / s
        a = (Gi @ Wi3) * c['mask_2']
        G2 = num.r(a)
        grads[6], grads[7] = G2.t() @ c['H1'] / s, a.sum(0) / s
        a = (G2 @ Wi2) * c['mask_1']
        G1 = num.r(a)
        grads[4], grads[5] = G1.t() @ c['X'] / s, a.sum(0) / s
        dX = G1 @ Wi1 if dX is None else dX + G1 @ Wi1
    g_panop = None
    if need_panop and dX is not None:
        g_panop = dX / s * (c['lw'][None] if c['lw'] is not None else 1.0)
    return dict(grads=grads, g_panop=g_panop, amb=num.amb)


# ------------------------------------------------------------------------------------------------------------------------
# heads fused with their compositing (pan_comp_fwd_kernel / pan_comp_bwd_kernel)
# ------------------------------------------------------------------------------------------------------------------------
def comp_forward(feats, dfeats, lodw, weights, w, alpha, ridx, N, Cs, Ci, sem_softmax, inst_softmax, temperature,
                 fp16=True, img=False):
    """out[ray] = alpha[ray] * sum_s w[s] * r16(p_s) -> dict(sem [N, Cs], inst [N, Ci], inst_lse [M] (log2 domain, softmax
    only), amb [M], ctx).  img: feats / dfeats hold the fp16 values of operand images (their sum is rounded to fp16)."""
    f, df, lw = _d(feats), _d(dfeats), _d(lodw)
    M = f.shape[0]
    num = _Num(fp16, M)
    W = _tc_weights(num, weights, lw, (0, 4))
    X = num.r(f if df is None else f + df, rows=not img)     # image mode: an fp16 add of fp16 values, rounded alike
    it = _inv_temp(temperature)
    ctx = _heads_forward(num, X, *W, Cs, Ci, it)
    ridx = ridx.detach().long().cpu()
    coef = _d(alpha).reshape(-1)[ridx] * _d(w).reshape(-1)
    out = dict(sem=None, inst=None, inst_lse=None)
    if Cs:
        ps = torch.softmax(ctx['zs'], 1) if sem_softmax else ctx['zs']
        out['sem'] = torch.zeros(N, Cs, dtype=torch.float64).index_add_(0, ridx, num.r(ps) * coef[:, None])
    if Ci:
        pi = torch.softmax(ctx['zi'], 1) if inst_softmax else ctx['zi']
        out['inst'] = torch.zeros(N, Ci, dtype=torch.float64).index_add_(0, ridx, num.r(pi) * coef[:, None])
        if inst_softmax:
            out['inst_lse'] = torch.logsumexp(ctx['zi'], 1) / math.log(2.0)
    ctx.update(num=num, X=X, lw=lw, W=W, it=it, ss=sem_softmax, si=inst_softmax, ridx=ridx, coef=coef)
    out['amb'] = num.amb
    out['ctx'] = ctx
    return out


def comp_backward(fwd, g_sem, g_inst, scale=1.0, need_panop=True, img=False, inst_lse=None):
    """g_sem [N, Cs], g_inst [N, Ci] per RAY -> dict(grads [10], g_panop [M, IN] (img: fp16 image values times scale),
    gw_sem [M], gw_inst [M], amb [M]).  inst_lse: the lse the kernel is given (default: the exact one)."""
    c = fwd['ctx']
    num = c['num']
    s = float(scale)
    Ws1, _, Ws2, _, Wi1, _, Wi2, _, Wi3, _ = c['W']
    ridx, coef = c['ridx'], c['coef'][:, None]
    grads = [None] * 10
    dX = None
    out = dict(gw_sem=None, gw_inst=None)
    if g_sem is not None and 'zs' in c:
        g = _d(g_sem)[ridx]
        if c['ss']:
            p = torch.softmax(c['zs'], 1)
            dot = (p * g).sum(1, keepdim=True)
            dz = coef * s * p * (g - dot)
            out['gw_sem'] = dot[:, 0]
        else:
            dz = coef * s * g
            out['gw_sem'] = (c['zs'] * g).sum(1)
        Gs = num.r(dz)
        grads[2], grads[3] = Gs.t() @ c['Hs'] / s, dz.sum(0) / s
        a = (Gs @ Ws2) * c['mask_s']
        Gs1 = num.r(a)
        grads[0], grads[1] = Gs1.t() @ c['X'] / s, a.sum(0) / s
        dX = Gs1 @ Ws1
    if g_inst is not None and 'zi' in c:
        gc = num.r(_d(g_inst) * s, rows=False)[ridx]
        if c['si']:
            lse = _d(inst_lse) if inst_lse is not None else torch.logsumexp(c['zi'], 1) / math.log(2.0)
            p = torch.exp2(c['zi'] / math.log(2.0) - lse[:, None])
            dot = (p * gc).sum(1, keepdim=True)
            Gi = num.r(coef * c['it'] * p * (gc - dot))
            out['gw_inst'] = dot[:, 0] / s
        else:
            Gi = num.r(coef * c['it'] * gc)
            out['gw_inst'] = (c['zi'] * gc).sum(1) / s
        grads[8], grads[9] = Gi.t() @ c['H2'] / s, Gi.sum(0) / s
        G2 = num.r((Gi @ Wi3) * c['mask_2'])
        grads[6], grads[7] = G2.t() @ c['H1'] / s, G2.sum(0) / s
        a = (G2 @ Wi2) * c['mask_1']
        G1 = num.r(a)
        grads[4], grads[5] = G1.t() @ c['X'] / s, a.sum(0) / s
        dX = G1 @ Wi1 if dX is None else dX + G1 @ Wi1
    lw = c['lw'] if c['lw'] is not None else 1.0
    for i in (0, 4):
        if grads[i] is not None:
            grads[i] = grads[i] * lw
    g_panop = None
    if need_panop and dX is not None:
        g_panop = num.r(dX) if img else dX / s
    out.update(grads=grads, g_panop=g_panop, amb=num.amb)
    return out


# ------------------------------------------------------------------------------------------------------------------------
# helpers shared by the tests
# ------------------------------------------------------------------------------------------------------------------------
def grad_scale(target, *grads):
    """2^floor(log2(target / max|g|)) over the finite entries, clamped to [2^-24, 2^60] (the exponent taken from the exact
    quotient); max|g| = 0 (or no finite entry) counts as 1e-30."""
    m = 0.0
    for g in grads:
        if g is not None and g.numel():
            a = _d(g).abs()
            a = a[~torch.isnan(a)]
            if a.numel():
                m = max(m, float(a.max()))
    m = max(m, 1e-30)
    if math.isinf(m):
        return 2.0 ** -24
    q = target / m
    e = math.frexp(q)[1] - 1          # q = mant * 2^(e+1), mant in [0.5, 1): floor(log2 q) exactly
    return float(min(max(2.0 ** e, 2.0 ** -24), 2.0 ** 60))


def image16(x16, IN):
    """fp16 rows [M, IN] -> the operand-image layout of pag_permuto_fwd_img16_dyn: per 128-row tile, INP / 8 chunks of
    [128 rows][8 halfs] (INP = IN rounded up to 16, zero padded; the last tile zero padded)."""
    M = x16.shape[0]
    INP = (IN + 15) // 16 * 16
    T = (M + 127) // 128
    pad = torch.zeros(T * 128, INP, dtype=x16.dtype, device=x16.device)
    pad[:M, :IN] = x16
    return pad.view(T, 128, INP // 8, 8).permute(0, 2, 1, 3).contiguous()


def from_image16(img, M, IN):
    """inverse of image16 -> [M, IN]."""
    T, nXc = img.shape[0], img.shape[1]
    return img.permute(0, 2, 1, 3).reshape(T * 128, nXc * 8)[:M, :IN]
