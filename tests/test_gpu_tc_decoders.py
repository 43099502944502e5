"""Op-level tests of the tensor-core training decoders against their fp16-faithful float64 restatement (oracle/tc16.py).

Every output, input gradient and parameter gradient of csrc/decoder_tc.cu (density / colour, modular semantic / instance heads)
and csrc/decoder_tc_fused.cu (heads fused with their compositing) is compared with oracle/tc16.py, which rounds to fp16 where
the kernels do.  The two sides then differ by fp32 accumulation order only, except on the few sample rows the oracle flags as
ambiguous (a ReLU pre-activation next to 0 or an fp16 rounding next to a midpoint): those rows are counted and compared loosely.

Bars (TOL), per tensor kind, come from the worst error measured over this file on an NVIDIA B200 (1000 W power limit):
  kind    metric                                                     measured (worst case)                      bar
  out     max |a - b| / (|b| + 0.05 max|b|), unflagged rows         4.2e-3 (modular heads, wide gradients)     1.7e-2
  dx      the same for g_feats / g_panop / g_dir / gw_*             4.1e-3 (fused, M = 20000)                 1.7e-2
  dW      ||a - b|| / ||b|| per weight gradient (all rows)          1.3e-3 (dc, M = 20000); others <= 1.4e-4  2.5e-3
  db      ||a - b|| / ||b|| per bias gradient (all rows)            9.8e-4 (dc, M = 20000); others <= 1.6e-4  2.5e-3
  dxl2    ||a - b|| / ||b|| of g_feats / g_panop (all rows)         1.0e-4 (modular heads, wide gradients)    4e-4
  amb     share of flagged sample rows                              0.31 (modular heads, Cs = 2, Ci = 51)     0.35
  flag    max |a - b| / max|b| on flagged rows                      3.0e-2 (dc g_dir, M = 20000)              0.12
Most bars are 4x the measured worst.  The weight and bias gradient bars are 1.9x and 2.6x: their worst case comes from the few
of 20000 rows whose ReLU pre-activation the kernel's fp32 accumulation puts on the other side of 0 (with gradient on the rows
of one tile only, the same weights and inputs give 3e-5), and 2.5e-3 keeps those bars 10x tighter than test_gpu_parity.py's
test_tc_decoders_vs_fp32 (tensor cores against exact FP32), which allows 2.5e-2 .. 4e-2 relative l2 on weight gradients and
0.1 relative l2 with 30 % max error on the coordinate gradient.  The output bar is elementwise and relative: single fp16
roundings of hidden activations that land on the other side of a rounding midpoint move a softmax output by up to ~4e-3
with weights at 3x their init scale.

The multi-tile cases reserve 120 SMs (pag_set_reserved_sms, a process-global library setting, restored afterwards): the
persistent grids shrink to 28 backward / 56 forward CTAs, so at M = 28 * 128 * 3 + 37 every backward CTA sweeps three or four
tiles (weight-gradient accumulation across tiles, next-tile prefetch, deferred dX copy-out).
"""
import ctypes
import math

import pytest
import torch

from oracle import tc16

pytestmark = pytest.mark.gpu
DEV = "cuda"
FLOOR = 0.05

TOL = dict(out=1.7e-2, dx=1.7e-2, dW=2.5e-3, db=2.5e-3, dxl2=4e-4, amb=0.35, flag=0.12)
ERR = {}      # kind -> (worst error seen in this process, where): the numbers behind TOL

M_MULTI = 28 * 128 * 3 + 37


def _rec(kind, v, msg):
    if v > ERR.get(kind, (0.0, ""))[0]:
        ERR[kind] = (v, msg)
    assert v <= TOL[kind], f"{msg}: {kind} error {v:.3e} > {TOL[kind]:.1e}"


def _rows(x, M):
    return x.reshape(M, -1) if M else x.reshape(0, 1)


def check_elem(got, ref, amb, kind, msg):
    """elementwise on unflagged rows (tight), loosely on flagged rows; amb: bool [rows] or None."""
    assert got is not None, msg
    a, b = got.detach().double().cpu(), ref.double()
    assert a.shape == b.shape, f"{msg}: shape {tuple(a.shape)} vs {tuple(b.shape)}"
    assert torch.isfinite(a).all(), f"{msg}: non-finite values"
    if not b.numel():
        return
    mx = float(b.abs().max())
    n = b.shape[0]
    e = _rows((a - b).abs() / (b.abs() + FLOOR * mx + 1e-30), n)
    ok = ~amb if amb is not None else torch.ones(n, dtype=torch.bool)
    _rec(kind, float(e[ok].max()) if ok.any() else 0.0, msg)
    if (~ok).any() and mx > 0:
        _rec("flag", float(_rows((a - b).abs(), n)[~ok].max()) / mx, msg + " (flagged rows)")


def check_l2(got, ref, kind, msg):
    if ref is None:
        assert got is None or not got.any(), f"{msg}: expected no gradient"
        return
    assert got is not None, msg
    a, b = got.detach().double().cpu(), ref.double()
    assert a.shape == b.shape, f"{msg}: shape {tuple(a.shape)} vs {tuple(b.shape)}"
    assert torch.isfinite(a).all(), f"{msg}: non-finite values"
    nb = float(b.norm())
    _rec(kind, float((a - b).norm()) / nb if nb > 0 else float(a.norm()), msg)


def check_grads(got, ref, msg):
    for i, (g, r) in enumerate(zip(got, ref)):
        check_l2(g, r, "db" if i % 2 else "dW", f"{msg} grad[{i}]")


def check_amb(amb, msg):
    frac = float(amb.float().mean()) if amb.numel() else 0.0
    _rec("amb", frac, msg)


def ray_flags(amb, ridx, N):
    f = torch.zeros(N, dtype=torch.bool)
    f[ridx.cpu()[amb]] = True
    return f


@pytest.fixture
def few_ctas(cuda_lib):
    """Persistent grids of 28 backward / 56 forward CTAs (148 SMs, 120 reserved); the previous value is restored."""
    prev = ctypes.c_int(0)
    assert cuda_lib.pag_set_reserved_sms(120, ctypes.addressof(prev)) == 0
    try:
        yield
    finally:
        cuda_lib.pag_set_reserved_sms(prev.value, None)


def _rand_linear(out_f, in_f, gen, scale=1.0):
    w = (torch.rand(out_f, in_f, generator=gen) * 2 - 1) * (scale / in_f ** 0.5)
    b = (torch.rand(out_f, generator=gen) * 2 - 1) * 0.1
    return [w.to(DEV), b.to(DEV)]


def _dc_weights(IN, gen, scale=1.0):
    return (_rand_linear(64, IN, gen, scale) + _rand_linear(16, 64, gen, scale) + _rand_linear(64, 43, gen, scale)
            + _rand_linear(64, 64, gen, scale) + _rand_linear(3, 64, gen, scale))


def _pan_weights(IN, Cs, Ci, gen, scale=1.0):
    return (_rand_linear(64, IN, gen, scale) + _rand_linear(max(Cs, 1), 64, gen, 4.0 * scale)
            + _rand_linear(64, IN, gen, scale) + _rand_linear(64, 64, gen, scale) + _rand_linear(max(Ci, 1), 64, gen, 4.0 * scale))


def _grad(shape, gen, wide):
    """upstream gradient: N(0, 1) / 64, or (wide) random signs times 2^U(-20, 10) within one tensor."""
    if wide:
        e = torch.rand(shape, generator=gen) * 30 - 20
        g = torch.sign(torch.randn(shape, generator=gen)) * torch.exp2(e)
        g.view(-1)[0] = 1024.0
        return g.to(DEV)
    return (torch.randn(shape, generator=gen) / 64).to(DEV)


def _img(x, IN):
    return tc16.image16(x.half(), IN)


def _scale(a, b=None, m_dev=None, wa=1, wb=1):
    from pagnerf_b200 import ops
    return ops.grad_scale_dyn(a if a is not None else b, b if a is not None else None, m_dev, wa, wb)


# ------------------------------------------------------------------------------------------------------------------------
# density + colour
# ------------------------------------------------------------------------------------------------------------------------
# id: (M, IN, S, lodw, want_rgb, g_sigma, g_rgb, g_feats, g_dir, path, few_ctas, workspace, m_dev, wide)
DC_CASES = {
    "M1": (1, 12, 1, True, True, True, True, True, True, "op", False, False, None, False),
    "M127": (127, 48, 1, True, True, True, True, True, True, "op", False, False, None, False),
    "M128_IN4": (128, 4, 1, True, True, True, True, True, True, "op", False, False, None, False),
    "M136_IN28_S8": (136, 28, 8, False, True, True, True, True, True, "op", False, False, None, False),
    "M3000_IN64_S8": (3000, 64, 8, True, True, True, True, True, True, "op", False, False, None, False),
    "M20000_more_tiles_than_ctas": (20000, 48, 1, True, True, True, True, True, True, "op", False, False, None, False),
    "no_rgb": (1000, 12, 1, True, False, True, False, True, False, "op", False, False, None, False),
    "no_feats_no_dir": (1000, 48, 4, True, True, True, True, False, False, "op", False, False, None, False),
    "dyn_no_g_sigma": (2000, 48, 1, True, True, False, True, True, True, "dyn", False, True, None, False),
    "dyn_no_g_rgb_dir": (2000, 28, 1, True, True, True, False, True, True, "dyn", False, False, None, False),
    "dyn_multi_ws": (M_MULTI, 48, 1, True, True, True, True, True, True, "dyn", True, True, None, False),
    "dyn_multi_atomic": (M_MULTI, 28, 1, False, True, True, True, True, False, "dyn", True, False, None, False),
    "dyn_mdev": (5000, 48, 1, True, True, True, True, True, True, "dyn", False, True, 4321, False),
    "img_multi_ws": (M_MULTI, 48, 1, True, True, True, True, True, True, "img", True, True, None, False),
    "img_IN12_mdev": (3000, 12, 1, True, True, True, True, True, False, "img", False, False, 2900, False),
    "wide_grads": (4000, 48, 1, True, True, True, True, True, True, "dyn", False, True, None, True),
}


@pytest.mark.parametrize("case", list(DC_CASES))
def test_dc_tc_vs_oracle(cuda_lib, request, case):
    from pagnerf_b200 import ops
    from pagnerf_b200._lib import call, ptr, ptr_array, query_i64
    M, IN, S, lod, want_rgb, gsig, grgb, gfe, gdir, path, few, use_ws, mdev, wide = DC_CASES[case]
    tag = "dc " + case
    if few:
        request.getfixturevalue("few_ctas")
    gen = torch.Generator().manual_seed(sum(map(ord, case)))
    w = _dc_weights(IN, gen, 3.0 if wide else 1.0)
    feats = torch.randn(M, IN, generator=gen).to(DEV)
    lodw = (torch.rand(IN, generator=gen) + 0.5).to(DEV) if lod else None
    gs = _grad((M,), gen, wide) if gsig else None
    gr = _grad((M, 3), gen, wide) if grgb else None
    img = path == "img"
    if path == "op":
        R = M // S
        ray_d = torch.nn.functional.normalize(torch.randn(R, 3, generator=gen), dim=-1).to(DEV)
        rows_d = ray_d.repeat_interleave(S, 0)
        m = M
        f = feats.clone().requires_grad_(gfe)
        d = ray_d.clone().requires_grad_(gdir)
        wl = [x.clone().requires_grad_(True) for x in w]
        sigma, rgb = ops.DecodeDCFn.apply(f, lodw, d, S, want_rgb, True, *wl)
        outs, gouts = [sigma], [gs]
        if grgb:
            outs.append(rgb); gouts.append(gr)
        sc = float(ops.grad_scale(gs, gr if grgb else None))
        inputs = wl + ([f] if gfe else []) + ([d] if gdir else [])
        res = torch.autograd.grad(outs, inputs, gouts, allow_unused=True)
        grads, rest = list(res[:10]), list(res[10:])
        g_feats = rest.pop(0) if gfe else None
        g_dir = rest.pop(0) if gdir else None
        y0 = None
    else:
        R = max(1, M // 3)
        ray_d = torch.nn.functional.normalize(torch.randn(R, 3, generator=gen), dim=-1).to(DEV)
        ridx = torch.sort(torch.randint(0, R, (M,), generator=gen)).values.to(DEV)
        rows_d = ray_d[ridx]
        m = mdev if mdev is not None else M
        m_dev = torch.tensor([m], dtype=torch.int64, device=DEV) if mdev is not None else None
        pe16 = torch.empty(R, 32, dtype=torch.float16, device=DEV)
        call("pag_view_pe16", ptr(ray_d), R, ptr(pe16))
        x = _img(feats, IN) if img else feats
        nan = float("nan")
        sigma = torch.full((M,), nan, device=DEV)
        y0 = torch.full((M,), nan, device=DEV)
        rgb = torch.full((M, 3), nan, device=DEV) if want_rgb else None
        call("pag_decode_dc_fwd_tc_dyn", ptr(x), ptr(lodw), ptr(ray_d), ptr(ridx), M, ptr(m_dev), IN, ptr_array(w), 64, 27,
             int(want_rgb), ptr(sigma), ptr(rgb), ptr(y0), ptr(pe16), int(img))
        grads = [torch.zeros_like(t) for t in w]
        g_feats = (torch.full_like(x, nan) if img else torch.full((M, IN), nan, device=DEV)) if gfe else None
        g_dir = torch.full((M, 3), nan, device=DEV) if gdir else None
        scale_t = _scale(gs, gr, m_dev, 1, 3)
        sc = float(scale_t)
        wsb = query_i64("pag_decode_dc_bwd_workspace", M, IN) if use_ws else 0
        ws = torch.empty(wsb // 4, device=DEV) if wsb else None
        call("pag_decode_dc_bwd_tc_dyn", ptr(x), ptr(lodw), ptr(ray_d), ptr(ridx), M, ptr(m_dev), IN, ptr_array(w), ptr_array(grads),
             64, 27, ptr(gs), ptr(gr), ptr(scale_t), ptr(g_feats), ptr(g_dir), ptr(pe16), ptr(ws), wsb, int(img))
        torch.cuda.synchronize()
        if not grgb:
            grads[4:10] = [None] * 6
        if m < M:      # rows past m_dev are not written
            for name, t in (("sigma", sigma), ("y0", y0), ("rgb", rgb), ("g_dir", g_dir)) + ((("g_feats", g_feats),) if not img else ()):
                if t is not None:
                    assert torch.isnan(t[m:]).all(), f"{case}: {name} written past m_dev"
        if img and g_feats is not None:
            g_feats = tc16.from_image16(g_feats, M, IN).float()
    fin = feats[:m].half() if img else feats[:m]
    fw = tc16.dc_forward(fin, lodw, rows_d[:m], w, want_rgb=want_rgb or grgb, img=img)
    bw = tc16.dc_backward(fw, gs[:m] if gs is not None else None, gr[:m] if gr is not None else None, sc,
                          need_feats=gfe, need_dir=gdir, img=img)
    amb = fw["amb"] | bw["amb"]
    check_amb(amb, tag)
    check_elem(sigma[:m], fw["sigma"], amb, "out", f"{tag} sigma")
    if y0 is not None:
        check_elem(y0[:m], fw["y0"], amb, "out", f"{tag} y0")
    if want_rgb:
        check_elem(rgb[:m], fw["rgb"], amb, "out", f"{tag} rgb")
    check_grads(grads, bw["grads"], tag)
    if gfe:
        check_elem(g_feats[:m], bw["g_feats"], amb, "dx", f"{tag} g_feats")
        check_l2(g_feats[:m], bw["g_feats"], "dxl2", f"{tag} g_feats")
    if gdir:
        ref = bw["g_dir"]
        if path == "op" and S > 1:
            ref, ramb = ref.view(-1, S, 3).sum(1), amb.view(-1, S).any(1)
        else:
            ramb = amb
        check_elem(g_dir[:ref.shape[0]], ref, ramb, "dx", f"{tag} g_dir")


# ------------------------------------------------------------------------------------------------------------------------
# modular semantic + instance heads
# ------------------------------------------------------------------------------------------------------------------------
# id: (M, IN, Cs, Ci, softmax, temperature, delta, few_ctas, wide)
PAN_CASES = {
    "M1": (1, 12, 6, 20, True, 0.0, True, False, False),
    "M127_Cs0_Ci200": (127, 48, 0, 200, True, 0.5, True, False, False),
    "M128_Cs32_Ci1_nosoftmax": (128, 28, 32, 1, False, 2.0, False, False, False),
    "M129_Ci0": (129, 64, 6, 0, True, 0.0, True, False, False),
    "M3000_Cs2_Ci51": (3000, 64, 2, 51, True, 2.0, True, False, False),
    "M3000_IN4_Ci129_nosoftmax": (3000, 4, 6, 129, False, 0.5, True, False, False),
    "M2500_Ci224": (2500, 48, 6, 224, True, 0.0, False, False, False),
    "multi_Ci200": (M_MULTI, 48, 6, 200, True, 0.5, True, True, False),
    "M20000_more_tiles_than_ctas": (20000, 48, 6, 200, True, 0.0, True, False, False),
    "wide_grads": (4000, 48, 6, 200, True, 2.0, True, False, True),
}


@pytest.mark.parametrize("case", list(PAN_CASES))
def test_pan_tc_vs_oracle(cuda_lib, request, case):
    from pagnerf_b200 import ops
    M, IN, Cs, Ci, sm, temp, delta, few, wide = PAN_CASES[case]
    tag = "pan " + case
    if few:
        request.getfixturevalue("few_ctas")
    gen = torch.Generator().manual_seed(sum(map(ord, case)))
    w = _pan_weights(IN, Cs, Ci, gen, 3.0 if wide else 1.0)
    feats = torch.randn(M, IN, generator=gen).to(DEV)
    dfeats = (torch.randn(M, IN, generator=gen) * 0.3).to(DEV) if delta else None
    lodw = (torch.rand(IN, generator=gen) + 0.5).to(DEV)
    gs = _grad((M, Cs), gen, wide) if Cs else None
    gi = _grad((M, Ci), gen, wide) if Ci else None
    f = feats.clone().requires_grad_(True)
    df = dfeats.clone().requires_grad_(True) if delta else None
    wl = [x.clone().requires_grad_(True) for x in w]
    sem, inst = ops.DecodePanFn.apply(f, df, lodw, Cs, Ci, sm, sm, temp, True, *wl)
    outs = [o for o in (sem, inst) if o is not None]
    gouts = [g for g in (gs, gi) if g is not None]
    sc = float(ops.grad_scale(gs, gi))
    res = torch.autograd.grad(outs, wl + [f] + ([df] if delta else []), gouts, allow_unused=True)
    fw = tc16.pan_forward(feats, dfeats, lodw, w, Cs, Ci, sm, sm, temp)
    bw = tc16.pan_backward(fw, gs, gi, sc)
    amb = fw["amb"] | bw["amb"]
    check_amb(amb, tag)
    if Cs:
        check_elem(sem, fw["sem"], amb, "out", f"{tag} sem")
    if Ci:
        check_elem(inst, fw["inst"], amb, "out", f"{tag} inst")
    check_grads(list(res[:10]), bw["grads"], tag)
    check_elem(res[10], bw["g_panop"], amb, "dx", f"{tag} g_feats")
    check_l2(res[10], bw["g_panop"], "dxl2", f"{tag} g_feats")
    if delta:
        assert torch.equal(res[10], res[11])


@pytest.mark.parametrize("M,Cs,sm,temp", [(1000, 6, True, 0.5), (300, 0, False, 2.0)])
def test_pan_tc_backward_ci256_vs_oracle(cuda_lib, M, Cs, sm, temp):
    """Ci = 256 is a backward-only shape (the forward stops at 224): probabilities from the oracle, both dWi3 row blocks."""
    from pagnerf_b200 import ops
    from pagnerf_b200._lib import call, ptr, ptr_array
    IN, Ci = 48, 256
    gen = torch.Generator().manual_seed(M + Cs)
    w = _pan_weights(IN, Cs, Ci, gen)
    feats = torch.randn(M, IN, generator=gen).to(DEV)
    dfeats = (torch.randn(M, IN, generator=gen) * 0.3).to(DEV)
    lodw = (torch.rand(IN, generator=gen) + 0.5).to(DEV)
    gs = _grad((M, Cs), gen, False) if Cs else None
    gi = _grad((M, Ci), gen, False)
    fw = tc16.pan_forward(feats, dfeats, lodw, w, Cs, Ci, sm, sm, temp)
    sem = fw["sem"].float().to(DEV) if Cs else None
    inst = fw["inst"].float().to(DEV)
    grads = [torch.zeros_like(t) for t in w]
    gp = torch.empty(M, IN, device=DEV)
    sc = ops.grad_scale(gs, gi)
    call("pag_decode_pan_bwd_tc", ptr(feats), ptr(dfeats), ptr(lodw), M, IN, ptr_array(w), ptr_array(grads), 64, Cs, Ci, int(sm),
         int(sm), float(temp), ptr(sem), ptr(inst), ptr(gs), ptr(gi), ptr(sc), ptr(gp))
    bw = tc16.pan_backward(fw, gs, gi, float(sc))
    amb = fw["amb"] | bw["amb"]
    check_amb(amb, "ci256")
    if not Cs:
        grads[0:4] = [None] * 4
    check_grads(grads, bw["grads"], f"ci256 Cs={Cs}")
    check_elem(gp, bw["g_panop"], amb, "dx", "ci256 g_panop")


# ------------------------------------------------------------------------------------------------------------------------
# heads fused with their compositing
# ------------------------------------------------------------------------------------------------------------------------
def _ray_layout(kind, M, gen):
    """sorted per-sample ray index [M] and the ray count N."""
    if kind == "one":          # one sample per ray: 128 rays per tile, the 16-ray gradient cache misses most of them
        return torch.arange(M), M
    if kind == "random":       # sorted random rays, some empty
        N = max(2, M // 9)
        return torch.sort(torch.randint(0, N, (M,), generator=gen)).values, N
    # mixed: a ray over several tiles (and CTAs), empty rays, rays starting at a tile / 32-row quadrant boundary, short rays
    # at the end of the batch (ray0 + 16 > R)
    sizes = [0, 300, 0, 0, 84, 128, 32, 32, 64, 1, 31, 96, 2 * 128 * 3 + 5, 0, 7]
    while sum(sizes) < M - 40:
        sizes.append(int(torch.randint(0, 40, (1,), generator=gen)))
    sizes += [1] * 40
    out, n = [], 0
    for r, s in enumerate(sizes):
        take = min(s, M - n)
        out += [r] * take
        n += take
    return torch.tensor(out[:M]), len(sizes)


# id: (M, IN, Cs, Ci, softmax, temperature, layout, img, workspace, dd, few_ctas, wide)
COMP_CASES = {
    "M1": (1, 12, 6, 20, True, 0.0, "random", False, True, False, False, False),
    "M127_Cs0": (127, 4, 0, 51, True, 0.5, "random", False, True, False, False, False),
    "M129_Cs16_Ci208_nosoftmax": (129, 48, 16, 208, False, 2.0, "random", False, False, True, False, False),
    "one_per_ray": (3000, 12, 6, 200, True, 0.5, "one", False, True, False, False, False),
    "mixed_Ci1_nosoftmax": (3000, 48, 6, 1, False, 2.0, "mixed", False, True, True, False, False),
    "mixed_Ci0": (3000, 48, 16, 0, True, 0.0, "mixed", False, False, False, False, False),
    "multi_ws": (M_MULTI, 48, 6, 200, True, 0.5, "mixed", False, True, False, True, False),
    "multi_atomic_dd": (M_MULTI, 48, 6, 51, True, 2.0, "mixed", False, False, True, True, False),
    "multi_img": (M_MULTI, 48, 6, 200, True, 0.5, "mixed", True, True, True, True, False),
    "img_IN12_nosoftmax_dd": (3000, 12, 6, 51, False, 0.5, "random", True, False, True, False, False),
    "M20000_more_tiles_than_ctas": (20000, 48, 6, 208, True, 0.0, "random", False, True, False, False, False),
    "wide_grads": (4000, 48, 6, 200, True, 2.0, "mixed", False, True, True, False, True),
}


@pytest.mark.parametrize("case", list(COMP_CASES))
def test_pan_composite_tc_vs_oracle(cuda_lib, request, case):
    from pagnerf_b200._lib import call, ptr, ptr_array, query_i64
    M, IN, Cs, Ci, sm, temp, layout, img, use_ws, dd, few, wide = COMP_CASES[case]
    tag = "comp " + case
    if few:
        request.getfixturevalue("few_ctas")
    gen = torch.Generator().manual_seed(sum(map(ord, case)))
    w = _pan_weights(IN, Cs, Ci, gen, 3.0 if wide else 1.0)
    feats = torch.randn(M, IN, generator=gen).to(DEV)
    dfeats = (torch.randn(M, IN, generator=gen) * 0.3).to(DEV)
    lodw = (torch.rand(IN, generator=gen) + 0.5).to(DEV)
    ridx, N = _ray_layout(layout, M, gen)
    ridx = ridx.to(DEV)
    wgt = torch.rand(M, generator=gen).to(DEV)
    alpha = torch.rand(N, generator=gen).to(DEV)
    gs = _grad((N, Cs), gen, wide) if Cs else None
    gi = _grad((N, Ci), gen, wide) if Ci else None
    x, dx = (_img(feats, IN), _img(dfeats, IN)) if img else (feats, dfeats)
    sem = torch.zeros(N, Cs, device=DEV) if Cs else None
    inst = torch.zeros(N, Ci, device=DEV) if Ci else None
    lse = torch.empty(M, device=DEV) if (Ci and sm) else None
    call("pag_pan_composite_fwd_tc", ptr(x), ptr(dx), ptr(lodw), M, IN, ptr_array(w), 64, Cs, Ci, int(sm), int(sm), float(temp),
         ptr(wgt), ptr(alpha), ptr(ridx), ptr(sem), ptr(inst), ptr(lse), None, int(img))
    grads = [torch.zeros_like(t) for t in w]
    gp = torch.empty_like(x)
    gw_sem = torch.empty(M, device=DEV) if (dd and Cs) else None
    gw_inst = torch.empty(M, device=DEV) if (dd and Ci) else None
    sc = _scale(gs, gi)
    wsb = query_i64("pag_pan_composite_bwd_workspace", M, IN, Cs, Ci) if use_ws else 0
    ws = torch.empty(wsb // 4, device=DEV) if wsb else None
    call("pag_pan_composite_bwd_tc", ptr(x), ptr(dx), ptr(lodw), M, IN, ptr_array(w), ptr_array(grads), 64, Cs, Ci, int(sm), int(sm),
         float(temp), ptr(wgt), ptr(alpha), ptr(ridx), N, ptr(gs), ptr(gi), ptr(lse), ptr(sc), ptr(gp), None, ptr(ws), wsb, int(img),
         ptr(gw_sem), ptr(gw_inst))
    torch.cuda.synchronize()
    if img:
        gp = tc16.from_image16(gp, M, IN).float()
    fi, dfi = (feats.half(), dfeats.half()) if img else (feats, dfeats)
    fw = tc16.comp_forward(fi, dfi, lodw, w, wgt, alpha, ridx, N, Cs, Ci, sm, sm, temp, img=img)
    bw = tc16.comp_backward(fw, gs, gi, float(sc), img=img, inst_lse=lse.cpu() if lse is not None else None)
    amb = fw["amb"] | bw["amb"]
    check_amb(amb, tag)
    ramb = ray_flags(amb, ridx, N)
    if Cs:
        check_elem(sem, fw["sem"], ramb, "out", f"{tag} sem")
    if Ci:
        check_elem(inst, fw["inst"], ramb, "out", f"{tag} inst")
    if lse is not None:
        check_elem(lse, fw["inst_lse"], amb, "out", f"{tag} inst_lse")
    if not Cs:
        grads[0:4] = [None] * 4
    if not Ci:
        grads[4:10] = [None] * 6
    check_grads(grads, bw["grads"], tag)
    check_elem(gp, bw["g_panop"], amb, "dx", f"{tag} g_panop")
    check_l2(gp, bw["g_panop"], "dxl2", f"{tag} g_panop")
    if gw_sem is not None:
        check_elem(gw_sem, bw["gw_sem"], amb, "dx", f"{tag} gw_sem")
    if gw_inst is not None:
        check_elem(gw_inst, bw["gw_inst"], amb, "dx", f"{tag} gw_inst")


def test_pan_composite_op_vs_oracle(cuda_lib):
    """PanCompositeFn (workspace, loss scale from grad_scale) end to end through autograd."""
    from pagnerf_b200 import ops
    M, IN, Cs, Ci, temp = 5000, 48, 6, 200, 0.5
    gen = torch.Generator().manual_seed(7)
    w = _pan_weights(IN, Cs, Ci, gen)
    feats = torch.randn(M, IN, generator=gen).to(DEV)
    dfeats = (torch.randn(M, IN, generator=gen) * 0.3).to(DEV)
    lodw = (torch.rand(IN, generator=gen) + 0.5).to(DEV)
    ridx, N = _ray_layout("mixed", M, gen)
    ridx = ridx.to(DEV)
    wgt, alpha = torch.rand(M, generator=gen).to(DEV), torch.rand(N, 1, generator=gen).to(DEV)
    gs, gi = _grad((N, Cs), gen, False), _grad((N, Ci), gen, False)
    df = dfeats.clone().requires_grad_(True)
    wl = [t.clone().requires_grad_(True) for t in w]
    sem, inst = ops.PanCompositeFn.apply(feats, df, lodw, wgt, alpha, ridx, N, Cs, Ci, True, True, temp, *wl)
    res = torch.autograd.grad([sem, inst], wl + [df], [gs, gi])
    fw = tc16.comp_forward(feats, dfeats, lodw, w, wgt, alpha, ridx, N, Cs, Ci, True, True, temp)
    bw = tc16.comp_backward(fw, gs, gi, float(ops.grad_scale(gs, gi)))
    amb = fw["amb"] | bw["amb"]
    ramb = ray_flags(amb, ridx, N)
    check_elem(sem, fw["sem"], ramb, "out", "op sem")
    check_elem(inst, fw["inst"], ramb, "out", "op inst")
    check_grads(list(res[:10]), bw["grads"], "op")
    check_elem(res[10], bw["g_panop"], amb, "dx", "op g_panop")


# ------------------------------------------------------------------------------------------------------------------------
# loss scale
# ------------------------------------------------------------------------------------------------------------------------
def _kernel_scale(a, b=None, m_dev=None, wa=1, wb=1):
    return float(_scale(a, b, m_dev, wa, wb))


def test_grad_scale_exact(cuda_lib):
    """pag_grad_scale = 2^floor(log2(1024 / max|g|)) over the finite entries, clamped to [2^-24, 2^60].
    The kernel takes the exponent from floorf(log2f(1024 / amax)) in fp32.  When the quotient lies just below a power of two,
    log2f may round up to the integer and the kernel then picks the next power: the scale is a soft target (fp16 holds up to
    65504 = 2^16 (1 - 2^-11), and the scaled maximum stays below 2048), so that neighbour is accepted there and only there --
    within 2^-20 relative of a power of two.  Everywhere else the exponent must be exact."""
    T = 1024.0
    dev = DEV

    def ref(*gs):
        return tc16.grad_scale(T, *gs)

    def expect(got, want, amax, msg):
        q = T / amax if amax > 0 else math.inf
        near = math.isfinite(q) and q > 0 and abs(q / 2.0 ** round(math.log2(q)) - 1) < 2.0 ** -20
        assert got == want or (near and got == 2 * want), f"{msg}: {got} vs {want}"

    g = torch.tensor([1.0, -4.0, 0.5], device=dev)
    assert _kernel_scale(g) == 256.0                                    # 1024 / 4 = 2^8 exactly
    g = torch.tensor([4.0 * (1 - 2.0 ** -24)], device=dev)             # quotient just above 2^8: exactly 2^8
    assert _kernel_scale(g) == 256.0
    g = torch.tensor([4.0 * (1 + 2.0 ** -23)], device=dev)             # quotient just below 2^8: 2^7, or 2^8 from log2f
    assert _kernel_scale(g) in (128.0, 256.0)
    assert _kernel_scale(torch.zeros(1000, device=dev)) == 2.0 ** 60      # all zero: clamped
    g = torch.randn(5000, device=dev)
    g[17] = float("nan"); g[4000] = float("nan")
    amax = float(g[~torch.isnan(g)].abs().max())
    expect(_kernel_scale(g), ref(g), amax, "NaN entries ignored")
    g[99] = float("inf")
    assert _kernel_scale(g) == 2.0 ** -24                                # an inf entry: the smallest scale
    # m_dev with widths: only the first m * wa / m * wb entries count
    a = torch.rand(1000, device=dev)
    b = torch.rand(1000, 3, device=dev) * 3
    a[500:] = 1e6
    b[500:] = 1e6
    m_dev = torch.tensor([500], dtype=torch.int64, device=dev)
    expect(_kernel_scale(a, b, m_dev, 1, 3), ref(a[:500], b[:500]), max(float(a[:500].max()), float(b[:500].max())), "m_dev")
    # a second tensor whose pointer is not 16-byte aligned (scalar path), its maximum in the unaligned tail
    buf = torch.rand(1001, device=dev)
    buf[1000] = 77.0
    bu = buf[1:]
    assert bu.data_ptr() % 16 != 0
    expect(_kernel_scale(a[:500], bu), ref(a[:500], bu), 77.0, "unaligned b")
    # random maxima: exact exponent except within 2^-20 of a power of two
    gen = torch.Generator().manual_seed(3)
    for k in range(40):
        x = (torch.randn(int(torch.randint(1, 70000, (1,), generator=gen)), generator=gen)
             * float(torch.exp2(torch.rand(1, generator=gen) * 60 - 30))).to(dev)
        expect(_kernel_scale(x), ref(x), float(x.abs().max()), f"random {k}")


def test_grad_scale_scratch_returns_to_zero_on_two_streams(cuda_lib):
    from pagnerf_b200 import ops
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
    xs = [torch.randn(4096, device=DEV) * 2.0 ** k for k in range(-8, 8)]
    torch.cuda.synchronize()
    outs = []
    for i, x in enumerate(xs):
        with torch.cuda.stream(s1 if i % 2 else s2):
            outs.append(ops.grad_scale(x))
    torch.cuda.synchronize()
    for x, o in zip(xs, outs):
        want = tc16.grad_scale(1024.0, x)
        assert float(o) in (want, 2 * want)
    for st in (s1, s2):
        scratch = ops._SCALE_SCRATCH[(str(xs[0].device), st.cuda_stream)]
        assert not scratch.any(), "scratch words not reset"


# ------------------------------------------------------------------------------------------------------------------------
# limits of the C entry points
# ------------------------------------------------------------------------------------------------------------------------
def _refused(name, *args):
    from pagnerf_b200._lib import call
    with pytest.raises(RuntimeError, match="unsupported"):
        call(name, *args)


def test_tc_entry_point_limits(cuda_lib):
    """Past each shape limit an entry point refuses (PAG_ERR_UNSUPPORTED) and writes nothing; the limits themselves are
    computed right by the tests above (dc IN 64, fused IN 48 / Cs 16 / Ci 208, modular Cs 32 / Ci 224 forward / 256 backward)."""
    from pagnerf_b200._lib import ptr, ptr_array
    M = 256
    gen = torch.Generator().manual_seed(0)

    def bufs(IN, Cs, Ci, N=16):
        feats = torch.randn(M, IN, generator=gen).to(DEV)
        lodw = torch.ones(IN, device=DEV)
        dc = _dc_weights(IN, gen)
        pan = _pan_weights(IN, Cs, Ci, gen)
        return feats, lodw, dc, pan

    sentinel = -7.0
    d = torch.nn.functional.normalize(torch.randn(M, 3, device=DEV), dim=-1)
    one = torch.ones(1, device=DEV)
    # density / colour: IN 64 is the limit, 68 and IN % 4 != 0 are refused
    for IN in (68, 10):
        feats, lodw, dc, _ = bufs(IN, 1, 1)
        sigma, rgb = torch.full((M,), sentinel, device=DEV), torch.full((M, 3), sentinel, device=DEV)
        _refused("pag_decode_dc_fwd_tc", ptr(feats), ptr(lodw), ptr(d), 1, M, IN, ptr_array(dc), 64, 27, 1, ptr(sigma), ptr(rgb))
        ridx = torch.arange(M, device=DEV)
        _refused("pag_decode_dc_fwd_tc_dyn", ptr(feats), ptr(lodw), ptr(d), ptr(ridx), M, None, IN, ptr_array(dc), 64, 27, 1,
                 ptr(sigma), ptr(rgb), None, None, 0)
        grads = [torch.zeros_like(t) for t in dc]
        gf = torch.full((M, IN), sentinel, device=DEV)
        gs = torch.randn(M, device=DEV)
        _refused("pag_decode_dc_bwd_tc", ptr(feats), ptr(lodw), ptr(d), 1, M, IN, ptr_array(dc), ptr_array(grads), 64, 27, ptr(gs),
                 None, ptr(one), ptr(gf), None)
        _refused("pag_decode_dc_bwd_tc_dyn", ptr(feats), ptr(lodw), ptr(d), ptr(ridx), M, None, IN, ptr_array(dc), ptr_array(grads),
                 64, 27, ptr(gs), None, ptr(one), ptr(gf), None, None, None, 0, 0)
        torch.cuda.synchronize()
        assert (sigma == sentinel).all() and (rgb == sentinel).all() and (gf == sentinel).all()
        assert not any(g.any() for g in grads)
    # modular heads: Cs 32 / Ci 224 (forward) / Ci 256 (backward) are the limits; IN % 4 != 0 is refused by both
    for IN, Cs, Ci, fwd, bwd in ((48, 33, 20, True, True), (48, 6, 225, True, False), (48, 6, 257, True, True),
                                 (10, 6, 20, True, True), (68, 6, 20, True, True)):
        feats, lodw, _, pan = bufs(IN, Cs, Ci)
        sem, inst = torch.full((M, Cs), sentinel, device=DEV), torch.full((M, Ci), sentinel, device=DEV)
        if fwd:
            _refused("pag_decode_pan_fwd_tc", ptr(feats), None, ptr(lodw), M, IN, ptr_array(pan), 64, Cs, Ci, 1, 1, 0.0,
                     ptr(sem), ptr(inst))
        if bwd:
            grads = [torch.zeros_like(t) for t in pan]
            gp = torch.full((M, IN), sentinel, device=DEV)
            p_s, p_i = torch.softmax(torch.randn(M, Cs, device=DEV), 1), torch.softmax(torch.randn(M, Ci, device=DEV), 1)
            g_s, g_i = torch.randn(M, Cs, device=DEV), torch.randn(M, Ci, device=DEV)
            _refused("pag_decode_pan_bwd_tc", ptr(feats), None, ptr(lodw), M, IN, ptr_array(pan), ptr_array(grads), 64, Cs, Ci, 1, 1,
                     0.0, ptr(p_s), ptr(p_i), ptr(g_s), ptr(g_i), ptr(one), ptr(gp))
            torch.cuda.synchronize()
            assert (gp == sentinel).all() and not any(g.any() for g in grads)
        torch.cuda.synchronize()
        assert (sem == sentinel).all() and (inst == sentinel).all()
    # fused: IN 48 / Cs 16 / Ci 208 are the limits
    N = 16
    for IN, Cs, Ci in ((52, 6, 20), (10, 6, 20), (48, 17, 20), (48, 6, 209)):
        feats, lodw, _, pan = bufs(IN, Cs, Ci)
        ridx = torch.sort(torch.randint(0, N, (M,), device=DEV)).values
        wgt, alpha = torch.rand(M, device=DEV), torch.rand(N, device=DEV)
        sem, inst = torch.full((N, Cs), sentinel, device=DEV), torch.full((N, Ci), sentinel, device=DEV)
        lse = torch.full((M,), sentinel, device=DEV)
        for img in (0, 1):
            _refused("pag_pan_composite_fwd_tc", ptr(feats), None, ptr(lodw), M, IN, ptr_array(pan), 64, Cs, Ci, 1, 1, 0.0, ptr(wgt),
                     ptr(alpha), ptr(ridx), ptr(sem), ptr(inst), ptr(lse), None, img)
            grads = [torch.zeros_like(t) for t in pan]
            gp = torch.full((M, IN), sentinel, device=DEV)
            g_s, g_i = torch.randn(N, Cs, device=DEV), torch.randn(N, Ci, device=DEV)
            _refused("pag_pan_composite_bwd_tc", ptr(feats), None, ptr(lodw), M, IN, ptr_array(pan), ptr_array(grads), 64, Cs, Ci,
                     1, 1, 0.0, ptr(wgt), ptr(alpha), ptr(ridx), N, ptr(g_s), ptr(g_i), ptr(lse), ptr(one), ptr(gp), None, None, 0, img,
                     None, None)
            torch.cuda.synchronize()
            assert (gp == sentinel).all() and not any(g.any() for g in grads)
        assert (sem == sentinel).all() and (inst == sentinel).all() and (lse == sentinel).all()
