"""-m gpu: the fused generator + GEMM kernel of the linear activation sweeps (lin_fused_gemm_err.cu) against the
generator -> workspace -> GEMM path it replaces, on the shapes of the BASELINE models (both schedules: RESIDENT for the
int8 sweeps with K <= 1024, STREAMED for the post-GELU AdaLog sweeps with K = 4 x dim, one and two passes), ragged K
and N, fewer units than SMs, and against an independent FP64 evaluation."""
import pytest
import torch

import adalog_oracle as O      # candidate seeding only (test infrastructure)

pytestmark = pytest.mark.gpu
DEV = 'cuda'


def _uq(bits, scale, zp):
    from adalog_b200.quantizers import UniformQuantizer
    q = UniformQuantizer(bits)
    q.scale, q.zero_point, q.inited = scale, zp, True
    return q


def _setup(tokens, in_f, out_f, gelu=False, seed=3):
    torch.manual_seed(seed)
    x = torch.randn(tokens, in_f, device=DEV) * (torch.rand(in_f, device=DEV) * 2) + 0.3 * torch.randn(in_f, device=DEV)
    if gelu:
        x = torch.nn.functional.gelu(x)
    W = torch.nn.init.trunc_normal_(torch.empty(out_f, in_f, device=DEV), std=.02)
    b = torch.randn(out_f, device=DEV) * 0.02
    return x.view(1, tokens, in_f), W, b, torch.nn.functional.linear(x, W, b).view(1, tokens, out_f)


def _both(fn):
    from adalog_b200 import sweep
    with pytest.MonkeyPatch.context() as mp:
        mp.setattr(sweep, '_lin_fused_passes', lambda: 1 << 30)   # every shape that fits, not only the ones the policy picks
        fused = fn()
        mp.setattr(sweep, '_lin_fused_passes', lambda: None)
        plain = fn()
    return fused, plain


@pytest.mark.parametrize('tokens,in_f,out_f,bits', [
    (6304, 384, 1152, 3),      # DeiT-S qkv: RESIDENT, 3 K blocks, 5 N tiles
    (6304, 384, 384, 3),       # proj
    (3152, 768, 3072, 4),      # DeiT-B fc1: 6 K blocks, 12 N tiles
    (128, 384, 1000, 4),       # head: fewer units than SMs, ragged last N tile
    (777, 100, 52, 4),         # ragged K (one partial int8 block), tiny N
    (1500, 1024, 512, 6),      # Swin-B stage-4 width, W6A6: 8 K blocks resident
    (2000, 192, 192, 8),       # 8-bit activations: bf16 uniform operands
    (900, 768, 768, 8),        # bf16 uniform, 12 K blocks: STREAMED, 2 passes
])
def test_fused_uniform_sweep_matches_two_kernel_path(tokens, in_f, out_f, bits):
    from adalog_b200 import ops, sweep
    nl = 2 ** (bits - 1)
    x, W, b, y = _setup(tokens, in_f, out_f)
    W3 = W.view(1, out_f, in_f)
    wcs, wcz = O.weight_candidates(W, 1, nl, 128)
    wq = _uq(bits, wcs[64].clone(), wcz[64].clone().float())
    acs, acz = O.activation_candidates(x, nl, 128, False)
    ctx = sweep.LinearCtx(x, y, out_f)
    n0 = len(ops.PROFILE['lin'])
    ops.PROFILE['on'] = True
    try:
        fused, plain = _both(lambda: sweep.linear_err_a(ctx, W3, b, wq, acs, acz, nl))
    finally:
        ops.PROFILE['on'] = False
    assert len(ops.PROFILE['lin']) == n0 + 1, 'the fused kernel must have taken this shape'
    ops.profile_reset(False)
    assert torch.allclose(fused.double(), plain.double(), rtol=2e-6, atol=0), \
        ((fused.double() - plain.double()).abs() / plain.double().abs()).max().item()
    # independent evaluation of a few candidates: fake-quant forward kernels + FP64 matmul
    w_hat = wq(W3).view(out_f, in_f).double()
    for p in (0, 77, 127):
        aq = _uq(bits, acs[:, p].clone(), acz[:, p].clone().float())
        y_hat = aq(x).reshape(-1, in_f).double() @ w_hat.t() + b.double()
        ref = -((y.reshape(-1, out_f).double() - y_hat) ** 2).mean()
        assert abs(fused[0, p].item() - ref.item()) <= 1e-5 * abs(ref.item()), (p, fused[0, p].item(), ref.item())
    # equal candidates give bit-equal scores (exact ties), wherever they sit
    perm = torch.randperm(128, device=DEV)
    again, _ = _both(lambda: sweep.linear_err_a(ctx, W3, b, wq, acs[:, perm].contiguous(), acz[:, perm].contiguous(), nl))
    assert torch.equal(again, fused[:, perm])


@pytest.mark.parametrize('tokens,in_f,out_f,bits', [
    (6304, 1536, 384, 3),      # DeiT-S fc2: STREAMED, one pass of 2 x 192 columns
    (3152, 3072, 768, 4),      # DeiT-B fc2: two passes
    (1000, 768, 192, 4),       # DeiT-T fc2: one N tile
    (700, 200, 52, 6),         # ragged K, 6-bit LUT
    (100, 512, 128, 4),        # fewer units than SMs
])
def test_fused_log_sweep_matches_two_kernel_path(tokens, in_f, out_f, bits):
    from adalog_b200 import ops, sweep
    from adalog_b200.quantizers import ShiftAdaLogQuantizer
    nl = 2 ** (bits - 1)
    x, W, b, y = _setup(tokens, in_f, out_f, gelu=True)
    W3 = W.view(1, out_f, in_f)
    lq = ShiftAdaLogQuantizer(bits).to(DEV)
    lq.scale = torch.nn.Parameter(torch.tensor([float(x.max()) * 0.9 + O.SHIFT_GELU], device=DEV))
    lq.shift.data.fill_(O.SHIFT_GELU)
    lq.q.fill_(27)
    lq.update_table()
    lq.inited = True
    wcs, wcz = O.weight_candidates(W, 1, nl, 128)
    wq = _uq(bits, wcs[64].clone(), wcz[64].clone().float())
    s0 = float(lq.scale.detach())
    sc = torch.linspace(s0 * 0.7, s0 * 1.1, 128, device=DEV).view(1, -1)
    qc = (torch.arange(128, device=DEV) % 24 + 18).view(1, -1)
    ctx = sweep.LinearCtx(x, y, out_f)
    n0 = len(ops.PROFILE['lin'])
    ops.PROFILE['on'] = True
    try:
        fused, plain = _both(lambda: sweep.linear_err_log(ctx, W3, b, wq, lq, sc, qc))
        base_f, base_p = _both(lambda: sweep.linear_err_log(ctx, W3, b, wq, lq, None, qc))
    finally:
        ops.PROFILE['on'] = False
    assert len(ops.PROFILE['lin']) == n0 + 2
    ops.profile_reset(False)
    for f, p in ((fused, plain), (base_f, base_p)):
        assert torch.allclose(f.double(), p.double(), rtol=5e-6, atol=0), \
            ((f.double() - p.double()).abs() / p.double().abs()).max().item()
    perm = torch.randperm(128, device=DEV)
    again, _ = _both(lambda: sweep.linear_err_log(ctx, W3, b, wq, lq, sc[:, perm].contiguous(), qc[:, perm].contiguous()))
    assert torch.equal(again, fused[:, perm])


def test_fixed_operand_cache_follows_quantizer_updates():
    """The fixed (weight / activation) operand of a sweep is cached on the calibration context and keyed on the fixed
    side's quantizer parameters: scoring, updating a parameter through quantizers/_ste.assign and scoring again must
    give exactly what a cache-free evaluation gives (a stale operand would be off by far more than rounding)."""
    from adalog_b200 import sweep
    from adalog_b200.quantizers._ste import assign
    bits, nl = 4, 8
    x, W, b, y = _setup(1576, 192, 384)
    W3 = W.view(1, 384, 192)
    wcs, wcz = O.weight_candidates(W, 1, nl, 128)
    acs, acz = O.activation_candidates(x, nl, 128, False)
    wq = _uq(bits, torch.nn.Parameter(wcs[64].clone()), torch.nn.Parameter(wcz[64].clone().float()))
    aq = _uq(bits, torch.nn.Parameter(acs[:, 64].clone()), torch.nn.Parameter(acz[:, 64].clone().float()))
    ctx = sweep.LinearCtx(x, y, 384)

    def fresh(fn):
        old = sweep.FIXED_CACHE
        sweep.FIXED_CACHE = False
        try:
            return fn()
        finally:
            sweep.FIXED_CACHE = old

    score_a = lambda: sweep.linear_err_a(ctx, W3, b, wq, acs, acz, nl)
    score_w = lambda: sweep.linear_err_w(ctx, W3, b, aq, wcs, wcz, nl)
    for score, param, new in ((score_a, wq.scale, wcs[90]), (score_a, wq.zero_point, wcz[30].float()),
                              (score_w, aq.scale, acs[:, 20]), (score_w, aq.zero_point, acz[:, 100].float())):
        first = score()
        assert torch.equal(first, score()), 'a cache hit must reproduce the evaluation bit for bit'
        assert torch.equal(first, fresh(score))
        assign(param, new.clone().reshape(param.shape))
        second = score()
        assert torch.equal(second, fresh(score)), 'stale fixed operand after a quantizer update'
        assert not torch.equal(first, second)
