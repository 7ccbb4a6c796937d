"""GPU parity at the BASELINE shapes (round 2; VERDICT r1 "next" #1): the code paths the benchmark runs — CTA-pair / 256-row GEMM
tiles, hyper-connection kernels at D = 512 / 1024, tcgen05 attention at N' = 1056 with 8 heads, the whole d512 / depth-8 model and
a d1024 / 16-head model — against the fp32 oracle (oracle/e2tts_oracle.py) computed on the box's CPU inside the test, never against
a sibling kernel. All calls go through the C ABI. Tolerances as in test_gpu_parity.py (bf16 tensor-core path vs fp32 oracle).
"""
import math
import random

import pytest
import torch
import torch.nn.functional as F

from conftest import rel_l2
from oracle import e2tts_oracle as O

pytestmark = pytest.mark.gpu


@pytest.fixture(scope='module')
def pkg():
    import e2_tts_pytorch_b200 as pkg
    assert torch.cuda.is_available()
    pkg.lib.load()
    return pkg


def dev():
    return torch.device('cuda:0')


def bf(t):
    return t.to(torch.bfloat16).contiguous()


def cos(a, b):
    a, b = a.double().flatten(), b.double().flatten()
    return float((a @ b) / (a.norm() * b.norm() + 1e-30))


def check(name, got, want, tol):
    e = rel_l2(got.float().cpu(), want.float().cpu())
    assert e < tol, f'{name}: rel-L2 {e:.4g} >= {tol}'


# ----------------------------------------------------------------------------------------------------------------------
# (c) every GEMM tile configuration, at sizes where the auto-selection of the benchmark picks it, incl. all epilogues
@pytest.mark.parametrize('force_tile', [0, 1, 2, 3])
def test_gemm_tiles_and_epilogues(pkg, force_tile):
    torch.manual_seed(10 + force_tile)
    ops = pkg.ops
    M, N, K = 1096, 520, 320        # ragged in M and N: partial tiles in both directions for every tile shape
    A, B = bf(torch.randn(M, K, device=dev())), bf(torch.randn(N, K, device=dev()) * 0.1)
    ref = A.float() @ B.float().t()
    kw = dict(force_tile=force_tile)
    check('plain', ops.gemm(A, B, M, N, K, **kw)[:, :N], ref, 1e-2)
    At, Bt = A.t().contiguous(), B.t().contiguous()
    check('b mn-major', ops.gemm(A, Bt, M, N, K, b_mn=True, **kw)[:, :N], ref, 1e-2)
    check('a mn-major', ops.gemm(At, B, M, N, K, lda=M, a_mn=True, **kw)[:, :N], ref, 1e-2)
    got = ops.gemm(At, Bt, M, N, K, lda=M, ldb=N, a_mn=True, b_mn=True, out_fp32=True, split_k=3, **kw)
    check('dW split-k', got, ref, 1e-3)
    got = ops.gemm(At, Bt, M, N, K, lda=M, ldb=N, a_mn=True, b_mn=True, out_fp32=True, **kw)
    check('fp32 out', got, ref, 1e-3)
    A1, A2 = A[:, :192].contiguous(), A[:, 192:].contiguous()
    check('two-source', ops.gemm(A1, B, M, N, K, lda=192, A2=A2, lda2=128, K1=192, **kw)[:, :N], ref, 1e-2)
    # fused epilogue: bias, per-batch column gate (rows_per_batch not a multiple of 32: warps straddle batch elements), row mask, residual
    rpb = 274
    bias = torch.randn(N, device=dev())
    cs = torch.rand(M // rpb, N, device=dev()) + 0.5
    mask = (torch.rand(M, device=dev()) > 0.2).to(torch.uint8)
    resid = bf(torch.randn(M, N + 0, device=dev()))
    ldr = (N + 7) // 8 * 8
    resid_p = torch.zeros(M, ldr, device=dev(), dtype=torch.bfloat16)
    resid_p[:, :N] = resid
    want = (ref + bias) * cs.repeat_interleave(rpb, 0) * mask[:, None].float() + resid.float()
    got = ops.gemm(A, B, M, N, K, bias=bias, colscale=cs, rows_per_batch=rpb, rowmask=mask, resid=resid_p, ldr=ldr, **kw)[:, :N]
    check('epilogue', got, want, 1e-2)
    # GEGLU (N multiple of 128, packed [u(64) | gate(64)] rows) with the saved pre-activations
    N2 = 512
    W = bf(torch.randn(N2, K, device=dev()) * 0.1)
    b2 = torch.randn(N2, device=dev()) * 0.1
    ug = torch.empty(M, N2, device=dev(), dtype=torch.bfloat16)
    h = ops.gemm(A, W, M, N2, K, D2=ug, ldd2=N2, bias=b2, geglu=True, **kw)
    z = A.float() @ W.float().t() + b2
    zz = z.view(M, N2 // 128, 2, 64)
    want_h = (zz[:, :, 0] * F.gelu(zz[:, :, 1])).reshape(M, N2 // 2)
    check('geglu pre-activations', ug, z, 1e-2)
    check('geglu', h[:, :N2 // 2], want_h, 1.5e-2)


# ----------------------------------------------------------------------------------------------------------------------
# (b) hyper-connection width/depth at every template instantiation: D = 128/256 (<1,*>), 512 (<2,*>, the benchmark), 1024 (<4,false>),
#     with enough tokens that every warp of the persistent forward grid walks several tokens (prefetch double buffer wraps)
@pytest.mark.parametrize('D', [128, 256, 512, 1024])
def test_hyper_width_depth_all_widths(pkg, D):
    torch.manual_seed(20 + D)
    ops = pkg.ops
    B, n, S = 2, 1300, 4
    T = B * n
    x = (torch.randn(T, S, D, device=dev()) * 1.5).to(torch.bfloat16).requires_grad_()
    P = dict(gamma=torch.randn(D) * 0.1, afn=torch.randn(D, S + 1) * 0.05, ascale=torch.tensor(0.5), salpha=torch.randn(S, S + 1) * 0.5 + 0.3,
             bfn=torch.randn(D) * 0.05, bscale=torch.tensor(0.7), sbeta=torch.randn(S) * 0.3 + 1)
    P = {k: v.to(dev()).requires_grad_() for k, v in P.items()}
    gain = (1 + 0.2 * torch.randn(B, D, device=dev())).requires_grad_()
    y = bf(torch.randn(T, D, device=dev())).requires_grad_()
    for mode, ng in ((2, gain), (1, gain[0].detach().clone().requires_grad_()), (0, None)):
        br, res, beta = ops.HcWidth.apply(x, P['gamma'], P['afn'], P['ascale'], P['salpha'], P['bfn'], P['bscale'], P['sbeta'], ng, mode, n)
        out = ops.HcDepth.apply(res, y, beta)
        wb, wo = torch.randn_like(br, dtype=torch.float32), torch.randn_like(out, dtype=torch.float32)
        loss = (br.float() * wb).sum() + (out.float() * wo).sum()
        leaves = [x, y] + list(P.values()) + ([ng] if ng is not None else [])
        grads = torch.autograd.grad(loss, leaves)
        xr = x.detach().float().cpu().view(B, n, S, D).requires_grad_()
        yr = y.detach().float().cpu().view(B, n, D).requires_grad_()
        sd = {'p.norm.gamma': P['gamma'], 'p.dynamic_alpha_fn': P['afn'], 'p.dynamic_alpha_scale': P['ascale'], 'p.static_alpha': P['salpha'],
              'p.dynamic_beta_fn': P['bfn'], 'p.dynamic_beta_scale': P['bscale'], 'p.static_beta': P['sbeta']}
        sd = {k: v.detach().cpu().clone().requires_grad_() for k, v in sd.items()}
        ngr = ng.detach().cpu().clone().requires_grad_() if ng is not None else None
        b0, rest, be = O.hyper_width(sd, 'p', xr, S)
        if mode == 2:
            b0 = F.normalize(b0, dim=-1) * D ** 0.5 * ngr[:, None, :]
        elif mode == 1:
            b0 = F.normalize(b0, dim=-1) * D ** 0.5 * ngr
        o = O.hyper_depth(rest, be, yr)
        lr = (b0 * wb.cpu().view(B, n, D)).sum() + (o * wo.cpu().view(B, n, S, D)).sum()
        rleaves = [xr, yr] + list(sd.values()) + ([ngr] if ng is not None else [])
        rgrads = torch.autograd.grad(lr, rleaves)
        check(f'branch m{mode}', br, b0.reshape(T, D), 2e-2)
        check(f'out m{mode}', out, o.reshape(T, S, D), 2e-2)
        check(f'beta m{mode}', beta, be.reshape(T, S), 1e-3)
        names = ['d_xres', 'd_y', 'gamma', 'afn', 'ascale', 'salpha', 'bfn', 'bscale', 'sbeta', 'gain']
        for nm, a, b in zip(names, grads, rgrads):
            check(f'{nm} m{mode} D{D}', a.reshape(-1), b.reshape(-1), 3e-2)


# (b') the depth connection of sub-block k fused into the width connection of sub-block k+1 (ops.HcDepthWidth): forward outputs and every
#      gradient — d residual', d branch_out, d beta of the folded depth connection and all parameter gradients (the parameter GEMM runs on
#      two K sources, residual' rows then branch rows) — against the oracle's hyper_depth followed by hyper_width
@pytest.mark.parametrize('D', [128, 256, 512, 1024])
def test_hyper_depth_width_fused(pkg, D):
    torch.manual_seed(40 + D)
    ops = pkg.ops
    B, n, S = 2, 1312, 4          # T * S = 10496 = 64 * 164
    T = B * n
    assert ops.hc_can_fuse(T, S)
    rest = (torch.randn(T, S, D, device=dev()) * 1.5).to(torch.bfloat16).requires_grad_()
    yp = bf(torch.randn(T, D, device=dev())).requires_grad_()
    bp = (1 + 0.3 * torch.randn(T, S, device=dev())).requires_grad_()
    P = dict(gamma=torch.randn(D) * 0.1, afn=torch.randn(D, S + 1) * 0.05, ascale=torch.tensor(0.5), salpha=torch.randn(S, S + 1) * 0.5 + 0.3,
             bfn=torch.randn(D) * 0.05, bscale=torch.tensor(0.7), sbeta=torch.randn(S) * 0.3 + 1)
    P = {k: v.to(dev()).requires_grad_() for k, v in P.items()}
    gain = (1 + 0.2 * torch.randn(B, D, device=dev())).requires_grad_()
    for mode, ng in ((2, gain), (0, None)):
        br, res, beta = ops.HcDepthWidth.apply(rest, yp, bp, P['gamma'], P['afn'], P['ascale'], P['salpha'], P['bfn'], P['bscale'], P['sbeta'], ng, mode, n)
        wb, wr, wbe = torch.randn_like(br, dtype=torch.float32), torch.randn_like(res, dtype=torch.float32), torch.randn_like(beta)
        loss = (br.float() * wb).sum() + (res.float() * wr).sum() + (beta * wbe).sum()
        leaves = [rest, yp, bp] + list(P.values()) + ([ng] if ng is not None else [])
        grads = torch.autograd.grad(loss, leaves)
        rr = rest.detach().float().cpu().view(B, n, S, D).requires_grad_()
        yr = yp.detach().float().cpu().view(B, n, D).requires_grad_()
        br_ = bp.detach().cpu().view(B, n, S).requires_grad_()
        sd = {'p.norm.gamma': P['gamma'], 'p.dynamic_alpha_fn': P['afn'], 'p.dynamic_alpha_scale': P['ascale'], 'p.static_alpha': P['salpha'],
              'p.dynamic_beta_fn': P['bfn'], 'p.dynamic_beta_scale': P['bscale'], 'p.static_beta': P['sbeta']}
        sd = {k: v.detach().cpu().clone().requires_grad_() for k, v in sd.items()}
        ngr = ng.detach().cpu().clone().requires_grad_() if ng is not None else None
        x_in = O.hyper_depth(rr, br_, yr)                     # the streams the fused kernel never writes out
        b0, rst, be = O.hyper_width(sd, 'p', x_in, S)
        if mode == 2:
            b0 = F.normalize(b0, dim=-1) * D ** 0.5 * ngr[:, None, :]
        lr = (b0 * wb.cpu().view(B, n, D)).sum() + (rst * wr.cpu().view(B, n, S, D)).sum() + (be * wbe.cpu().view(B, n, S)).sum()
        rleaves = [rr, yr, br_] + list(sd.values()) + ([ngr] if ng is not None else [])
        rgrads = torch.autograd.grad(lr, rleaves)
        check(f'branch m{mode}', br, b0.reshape(T, D), 2e-2)
        check(f'res m{mode}', res, rst.reshape(T, S, D), 2e-2)
        check(f'beta m{mode}', beta, be.reshape(T, S), 1e-3)
        names = ['d_rest', 'd_y_prev', 'd_beta_prev', 'gamma', 'afn', 'ascale', 'salpha', 'bfn', 'bscale', 'sbeta', 'gain']
        for nm, a, b in zip(names, grads, rgrads):
            check(f'{nm} m{mode} D{D}', a.reshape(-1), b.reshape(-1), 3e-2)


# ----------------------------------------------------------------------------------------------------------------------
# (d) tcgen05 attention core at the benchmark's sequence length against an fp32 softmax written here (x-transformers Attend as the
#     reference configures it, SURVEY A.4 steps 4-5: scale, tanh soft clamp 50, key-padding mask, fp32 softmax, per-head gate)
def _attn_core_ref(q, k, v, gate, mask, clamp=50.0):
    B, H, Np, dh = q.shape
    sim = torch.einsum('bhid,bhjd->bhij', q, k) * dh ** -0.5
    sim = torch.tanh(sim / clamp) * clamp
    if mask is not None:
        sim = sim.masked_fill(~mask[:, None, None, :], -torch.finfo(sim.dtype).max)
    out = torch.einsum('bhij,bhjd->bhid', torch.softmax(sim, dim=-1), v)
    out = out * gate.view(B, Np, H).permute(0, 2, 1)[..., None]
    return out.permute(0, 2, 1, 3).reshape(B * Np, H * dh)


@pytest.mark.parametrize('Np,H,big_logits', [(1056, 8, False), (1056, 8, True), (2080, 16, False), (331, 3, True)])
def test_attention_core_vs_fp32_softmax(pkg, Np, H, big_logits):
    torch.manual_seed(30 + Np + H)
    ops = pkg.ops
    B = 2 if Np < 2000 else 1
    s = 3.0 if big_logits else 1.0      # big_logits: |q.k|/8/50 beyond the polynomial-tanh range -> the MUFU.TANH path
    q, k, v = (bf(torch.randn(B, H, Np, 64, device=dev()) * (s if i < 2 else 1.0)) for i in range(3))
    gate = torch.rand(B * Np, H, device=dev())
    m = torch.ones(B, Np, dtype=torch.bool, device=dev())
    m[0, Np // 3: Np // 3 + 40] = False
    m[B - 1, Np - 29:] = False
    leaves = [t.clone().requires_grad_() for t in (q, k, v)] + [gate.clone().requires_grad_()]
    og = ops.AttnCore.apply(*leaves, m.to(torch.uint8).contiguous(), 0.0, 0, 50.0, None)
    w = bf(torch.randn(B * Np, H * 64, device=dev()))
    grads = torch.autograd.grad(og, leaves, w)
    rl = [t.detach().float().cpu().requires_grad_() for t in leaves]
    ref = _attn_core_ref(*rl, m.cpu())
    rgrads = torch.autograd.grad(ref, rl, w.float().cpu())
    check('attention out', og, ref, 1e-2)
    for nm, a, b in zip(['dq', 'dk', 'dv', 'dgate'], grads, rgrads):
        check(f'attention {nm}', a, b, 2e-2)


# ----------------------------------------------------------------------------------------------------------------------
# (a), (e) whole model at the BASELINE widths against the oracle run on the host CPU
def _whole_model(pkg, tkw, B, N, lens, seed, tol_pred=3e-2, model_kw=None, e2tts_kw=None):
    torch.manual_seed(seed)
    random.seed(seed)   # the hyper-connections pick their initial stream with python's randrange (SURVEY A.5): same model on every run
    model = pkg.E2TTS(transformer=dict(dropout=0., max_seq_len=N, **tkw, **(model_kw or {})), use_vocos=False, **(e2tts_kw or {}))
    # dyn_scale 0.05 (5x the reference's init of the hyper-connections' dynamic scales): with the 0.5 of the 2-layer fixtures a depth-8
    # stack amplifies bf16 rounding of the residual streams ~10x — the fp32 oracle with its OWN stage outputs rounded to bf16
    # (O.STAGE_ROUND) then moves its prediction by 12.6 %, exactly what the kernels showed (gpurun_out/r2b_pytest.log). The probe below
    # keeps this test honest: the case must be well conditioned for a bf16 path before the kernels are held to 3e-2.
    sd = O.randomize_zero_init({k: v.clone() for k, v in model.state_dict().items()}, seed=seed + 1, dyn_scale=0.05)
    model.load_state_dict(sd)
    model.to(dev()).train()
    mel = torch.randn(B, N, 100)
    text = ['Hello', 'Goodbye'][:B]
    x0, times = torch.randn(B, N, 100), torch.rand(B)
    lens_t = torch.tensor(lens)
    span = torch.zeros(B, N, dtype=torch.bool)
    for b in range(B):
        span[b, lens[b] // 8: lens[b] - lens[b] // 10] = True
    with pkg.inject_randomness(x0=x0.to(dev()), times=times.to(dev()), span_mask=span.to(dev()), drop_text_cond=False):
        out = model(mel.to(dev()), text=text, lens=lens_t.to(dev()))
    out.loss.backward()
    torch.cuda.synchronize()
    # oracle on the host (fp32, all cores)
    osd = {k: v.clone().requires_grad_(v.is_floating_point()) for k, v in sd.items()}
    ref = O.e2tts_forward(osd, O.TransformerCfg(**tkw), mel, O.list_str_to_tensor(text), x0=x0, times=times, span_mask=span, lens=lens_t)
    ref['loss'].backward()
    O.STAGE_ROUND = O.bf16_ste
    try:
        with torch.no_grad():
            probe = O.e2tts_forward(sd, O.TransformerCfg(**tkw), mel, O.list_str_to_tensor(text), x0=x0, times=times, span_mask=span, lens=lens_t)
    finally:
        O.STAGE_ROUND = None
    e_probe = rel_l2(probe['pred'], ref['pred'].detach())
    assert e_probe < 1.5e-2, f'test case is ill-conditioned for bf16 activations (oracle vs bf16-stage oracle: {e_probe:.3g})'
    loss, rloss = float(out.loss), float(ref['loss'])
    assert abs(loss - rloss) <= 1e-2 * abs(rloss), (loss, rloss)
    check('pred', out.pred_flow, ref['pred'].detach(), tol_pred)
    print(f'pred rel-L2 {rel_l2(out.pred_flow.float().cpu(), ref["pred"].detach()):.4g} (bf16-stage oracle probe {e_probe:.4g})')
    total = float(torch.cat([v.grad.flatten() for v in osd.values() if v.grad is not None]).norm())
    worst = (1.0, None)
    for k, p in model.named_parameters():
        gr = osd[k].grad
        if gr is None:
            assert p.grad is None or float(p.grad.abs().max()) == 0.0, f'{k} should be unused'
            continue
        assert p.grad is not None, k
        if float(gr.norm()) < 1e-4 * total:     # negligible next to the whole gradient: direction is rounding noise in any bf16 path
            continue
        cs_ = cos(p.grad.cpu(), gr)
        worst = min(worst, (cs_, k))
        assert cs_ >= 0.99, (k, cs_)
    print(f'whole model {tkw}: loss {loss:.5f} (oracle {rloss:.5f}), worst grad cosine {worst}')


def test_e2tts_cfg2_shape_vs_oracle(pkg):
    """BASELINE cfg2's model (d512, depth 8, 8 heads) at its sequence length (N = 1024, N' = 1056), B = 2 with a ragged batch:
    T = 2112 rows -> the CTA-pair GEMM tile, hc_width_*<2,true>, 9-tile tcgen05 attention — what bench.py times."""
    _whole_model(pkg, dict(dim=512, depth=8, heads=8), B=2, N=1024, lens=[1024, 800], seed=40)


def test_e2tts_cfg3_kernels_vs_oracle(pkg):
    """cfg3 / cfg5's width (d1024, 16 heads, dim_text 512) at N = 2048 (N' = 2080): hc_width_*<4,false>, 16-head qkv packing,
    17-tile attention; depth 2 keeps the host oracle within seconds."""
    _whole_model(pkg, dict(dim=1024, depth=2, heads=16), B=1, N=2048, lens=[1900], seed=50)


def test_e2tts_attn_fourier_embed_input_vs_oracle(pkg):
    """SURVEY §8f row 4, first variant: Transformer(attn_fourier_embed_input=True) (e2_tts.py:545-546; LinearFourierEmbed :368-386 on the
    attention input, :909) — tcgen05 GEMM + b200_fourier_feat_* against the oracle, which tests/test_oracle_vs_reference.py pins to the
    reference's own code with the switch on. Loss, prediction and every parameter gradient incl. `layers.{i}.0.4.linear.weight`."""
    _whole_model(pkg, dict(dim=256, depth=2, heads=4), B=2, N=224, lens=[224, 170], seed=60, model_kw=dict(attn_fourier_embed_input=True))


def test_e2tts_concat_cond_vs_oracle(pkg):
    """SURVEY §8f row 4, third variant: E2TTS(concat_cond=True) (e2_tts.py:1134, :1200-1201, :1263-1267): the stem GEMM reads
    cat(cond, x) (b200_stem_prepare concat layout) against ONE packed Linear(2C -> dim); oracle pinned to the reference's own code."""
    _whole_model(pkg, dict(dim=256, depth=2, heads=4), B=2, N=224, lens=[224, 190], seed=80, e2tts_kw=dict(concat_cond=True))


def test_e2tts_interpolated_text_vs_oracle(pkg):
    """SURVEY §8f row 4, second variant: E2TTS(interpolated_text=True) (e2_tts.py:1135, :1233; InterpolatedCharacterEmbed :414-482) —
    b200_interp_text_* + the abs-pos Linear as a tcgen05 GEMM with bias / residual / row-mask epilogue, against the oracle (pinned to
    the reference's own code in tests/test_oracle_vs_reference.py): ragged text and audio lengths, gradients of the embedding table
    and both abs_pos_mlp linears included."""
    _whole_model(pkg, dict(dim=256, depth=2, heads=4), B=2, N=224, lens=[224, 150], seed=70, e2tts_kw=dict(interpolated_text=True))


# ----------------------------------------------------------------------------------------------------------------------
# (f) sampling: euler, 32 steps, autoguidance null model — against the oracle's fixed-grid ODE on the host
def _small_model(pkg, seed, depth=2):
    torch.manual_seed(seed)
    random.seed(seed)   # the hyper-connections pick their initial stream with python's randrange (SURVEY A.5): same model on every run
    tkw = dict(dim=128, depth=depth, heads=2)
    model = pkg.E2TTS(transformer=dict(dropout=0., max_seq_len=256, **tkw), use_vocos=False)
    sd = O.randomize_zero_init({k: v.clone() for k, v in model.state_dict().items()}, seed=seed + 1)
    model.load_state_dict(sd)
    return model.to(dev()), sd, O.TransformerCfg(**tkw)


def test_sample_32_steps_vs_oracle(pkg):
    model, sd, cfg = _small_model(pkg, 60)
    torch.manual_seed(61)
    cond = torch.randn(2, 24, 100)
    text = ['Hello', 'Goodbye']
    y0 = torch.randn(2, 64, 100)
    with pkg.inject_randomness(y0=y0.to(dev())):
        out = model.sample(cond.to(dev()), text=text, duration=64, steps=32, cfg_strength=1.0, return_raw_output=True)
    want = O.e2tts_sample(sd, cfg, cond, O.list_str_to_tensor(text), duration=64, y0=y0, steps=32, cfg_strength=1.0)
    assert out.shape == want.shape
    assert rel_l2(out.cpu(), want) < 5e-2


def test_sample_euler_and_null_model(pkg):
    """odeint method 'euler' (e2_tts.py:1122-1126 odeint_kwargs) and `cfg_null_model` autoguidance (:1318-1321: the null prediction
    comes from a second, weaker model WITH text instead of this model without text)."""
    model, sd, cfg = _small_model(pkg, 70)
    weak, wsd, _ = _small_model(pkg, 80)
    model.odeint_kwargs = dict(method='euler')
    torch.manual_seed(71)
    cond = torch.randn(2, 20, 100)
    text = ['Hello', 'Goodbye']
    tid = O.list_str_to_tensor(text)
    y0 = torch.randn(2, 48, 100)
    steps, strength = 6, 1.5
    with pkg.inject_randomness(y0=y0.to(dev())):
        out = model.sample(cond.to(dev()), text=text, duration=48, steps=steps, cfg_strength=strength, cfg_null_model=weak, return_raw_output=True)
    # host restatement of the same loop with the oracle's pieces (euler on linspace(0, 1, steps), SURVEY A.7)
    with torch.no_grad():
        lens = torch.maximum((tid != -1).sum(-1), torch.full((2,), 20))
        cond_mask = F.pad(O.lens_to_mask(lens, int(lens.amax())), (0, 48 - int(lens.amax())), value=False)[..., None]
        condp = F.pad(cond, (0, 0, 0, 48 - 20))
        step_cond = torch.where(cond_mask, condp, torch.zeros_like(condp))
        mask = O.lens_to_mask(torch.full((2,), 48), 48)
        ts = torch.linspace(0, 1, steps)
        y = y0
        for i in range(steps - 1):
            pred = O.transformer_with_pred_head(sd, cfg, y, step_cond, ts[i], mask, tid, False)
            null = O.transformer_with_pred_head(wsd, cfg, y, step_cond, ts[i], mask, tid, False)
            _, orth = O.project(pred - null, pred)
            y = y + (ts[i + 1] - ts[i]) * (pred + orth * strength)
        want = torch.where(cond_mask, condp, y)
    assert rel_l2(out.cpu(), want) < 5e-2


# ----------------------------------------------------------------------------------------------------------------------
# SURVEY §8f row 2: velocity-consistency loss (e2_tts.py:1556-1576; trainer hook trainer.py:259-268) — a second, no-grad forward of the
# EMA model at t + delta through the same kernels, fused into the loss head
def test_velocity_consistency_loss_vs_oracle(pkg):
    model, sd, cfg = _small_model(pkg, 90)
    ema, esd, _ = _small_model(pkg, 91)
    ema.eval()
    model.train()
    model.velocity_consistency_weight = 0.7
    torch.manual_seed(92)
    B, N = 2, 96
    mel = torch.randn(B, N, 100)
    text = ['Hello', 'Goodbye']
    lens = torch.tensor([96, 70])
    x0, times = torch.randn(B, N, 100), torch.rand(B) * 0.9
    span = torch.zeros(B, N, dtype=torch.bool)
    span[:, 10:60] = True
    with pkg.inject_randomness(x0=x0.to(dev()), times=times.to(dev()), span_mask=span.to(dev()), drop_text_cond=False):
        out = model(mel.to(dev()), text=text, lens=lens.to(dev()), velocity_consistency_model=ema, velocity_consistency_delta=1e-3)
    out.loss.backward()
    osd = {k: v.clone().requires_grad_(v.is_floating_point()) for k, v in sd.items()}
    ref = O.e2tts_forward(osd, cfg, mel, O.list_str_to_tensor(text), x0=x0, times=times, span_mask=span, lens=lens, velocity_sd=esd,
                          velocity_consistency_weight=0.7, velocity_consistency_delta=1e-3)
    ref['loss'].backward()
    assert abs(float(out.loss) - float(ref['loss'])) <= 1e-2 * abs(float(ref['loss']))
    assert abs(float(out.loss_breakdown.flow) - float(ref['flow_loss'])) <= 1e-2 * abs(float(ref['flow_loss']))
    assert abs(float(out.loss_breakdown.velocity_consistency) - float(ref['velocity_loss'])) <= 2e-2 * abs(float(ref['velocity_loss']))
    assert float(ref['velocity_loss']) > 0.1 * float(ref['flow_loss'])      # the term matters in this case
    total = float(torch.cat([v.grad.flatten() for v in osd.values() if v.grad is not None]).norm())
    for k, p in model.named_parameters():
        gr = osd[k].grad
        if gr is None or float(gr.norm()) < 1e-4 * total:
            continue
        assert cos(p.grad.cpu(), gr) >= 0.99, k
    assert all(p.grad is None for p in ema.parameters())
    # without a velocity model the breakdown's second entry is the zero buffer, as in the reference (:1554)
    with pkg.inject_randomness(x0=x0.to(dev()), times=times.to(dev()), span_mask=span.to(dev()), drop_text_cond=False):
        out2 = model(mel.to(dev()), text=text, lens=lens.to(dev()))
    assert float(out2.loss_breakdown.velocity_consistency) == 0.0
    assert abs(float(out2.loss) - float(ref['flow_loss'])) <= 1e-2 * abs(float(ref['flow_loss']))


# ----------------------------------------------------------------------------------------------------------------------
# SURVEY §8f row 3: on-device data path — MelSpec per item (trainer.py:101-131) + collate_fn (:61-82) + 'b d n -> b n d' (:253) as one launch
def test_melspec_collate_ragged_batch_vs_per_item_reference(pkg):
    torch.manual_seed(100)
    ms = pkg.MelSpec().to(dev())
    lens = [256 * 24, 256 * 17 + 100, 5000, 256 * 24 - 1]
    waves = [torch.randn(n) * 0.3 for n in lens]
    batch = ms.collate(waves)
    per_item = [O.melspec(w[None])[0] for w in waves]                 # [n_mels, frames_i] each (torchaudio semantics, pinned by test_oracle_*)
    n_max = max(m.shape[-1] for m in per_item)
    want = torch.stack([F.pad(m, (0, n_max - m.shape[-1])) for m in per_item]).transpose(1, 2)   # collate_fn zero-pads, trainer transposes
    assert batch['mel'].shape == want.shape, (batch['mel'].shape, want.shape)
    assert batch['mel_lengths'].tolist() == [m.shape[-1] for m in per_item]
    assert float((batch['mel'].cpu() - want).abs().max()) < 1e-3
    # the batched output feeds the model directly
    model = pkg.E2TTS(transformer=dict(dim=128, depth=2, heads=2), use_vocos=False).to(dev())
    out = model(batch['mel'], text=['a', 'b', 'c', 'd'], lens=batch['mel_lengths'])
    assert torch.isfinite(out.loss)
    # a long wave at the benchmark's frame count (1024 frames) against the oracle
    wave = torch.randn(2, 256 * 1023) * 0.2
    got = ms(wave.to(dev()))
    assert got.shape == (2, 100, 1024)
    assert float((got.cpu() - O.melspec(wave)).abs().max()) < 1e-3
