"""Per-evaluation candidate sweeps: the device replacements of the reference's `_search_best_*` bodies.

Each function scores P <= 128 candidates on all calibration samples held by this rank and returns the
reference's *similarity* tensor (= -error, FP32, same shape as the tensor the reference hands to
torch.topk), accumulated in FP64 on a static partition so equal candidates get bit-equal scores.
Under torch.distributed the FP64 sums are all-reduced before normalisation (utils/dist.py).

Factorisation used by every GEMM sweep (DESIGN.md section 3): fake-quantised operands are
(integer) x scale, so the tensor cores multiply the exact integer parts in bf16 with FP32 accumulation
and the scales, biases and shift corrections are applied in the fused epilogue.
"""
import functools
import math

import torch

from . import _const, ops
from .quantizers._ste import flag as _flag
from .utils import dist as adist

# operand workspace of the generator -> GEMM path (two buffers of half this size).  8 GiB of the 180 GB: fewer, larger
# chunks -- the DeiT-B fc2 AdaLog sweep (9.9 GB of candidate operand) measured 16.1 ms with 2 GiB, 14.7 ms with 8 GiB
WS_BYTES = 8 << 30
NUM_SMS = 148
R_BASE = 37.0


def _lin_fused_passes():
    """Policy for the linear activation sweeps: None = generator -> workspace -> GEMM; else the largest number of times
    the fused kernel may generate a unit's operand.  Measured on 128 x 197 tokens after the lean MMA issuer
    (tests/gpu_lin_bench.py, fused vs two-kernel, ms per evaluation): DeiT-S int8 K=384: N=1152 1.78 vs 2.15, N=384 1.10
    vs 1.16, N=1536 2.05 vs 2.36, AdaLog K=1536 N=384 4.08 vs 5.41; DeiT-B int8 K=768: N=2304 4.31 vs 4.93, N=768 2.09
    vs 2.40, N=3072 5.51 vs 6.47.  Only the schedules that regenerate the operand (DeiT-B AdaLog K=3072 N=768: two
    512-column TMEM passes, 17.4 vs 16.9) stay on the two-kernel path."""
    return 1

_workspaces = {}


def _workspace(device, n_bytes):
    key = (device.type, device.index)
    buf = _workspaces.get(key)
    if buf is None or buf.numel() < n_bytes:
        buf = torch.empty(n_bytes, dtype=torch.uint8, device=device)
        _workspaces[key] = buf
    return buf


def release_workspaces():
    _workspaces.clear()


def require_cuda(device):
    """The sweeps exist only as sm_100a kernels: refuse to run anywhere else (no CPU fallback)."""
    if device.type != 'cuda':
        raise EnvironmentError('CUDA is not available for this module: adalog_b200 has no CPU path')


def _pad128(t, dim=-1):
    """repeat the last candidate up to 128 entries along `dim` (pad rows are ignored by the caller)."""
    P = t.shape[dim]
    if P == ops.P_TILE:
        return t
    idx = torch.clamp(torch.arange(ops.P_TILE, device=t.device), max=P - 1)
    return t.index_select(dim, idx)


_side = {}


def _side_streams(device):
    key = (device.type, device.index)
    if key not in _side:
        # the GEMM stream has priority: its one-CTA-per-SM grid must get onto the SMs first, the generator's small CTAs
        # then fill the registers / shared memory it leaves (the other way round the big CTAs never find room)
        _side[key] = (torch.cuda.Stream(device=device, priority=0), torch.cuda.Stream(device=device, priority=-1))
    return _side[key]


L2_SLICE_BYTES = 32 << 20     # fixed-operand slice that concurrently running CTAs should share out of the 126 MB L2
L2_CAND_BYTES = 48 << 20      # candidate-operand bytes that co-resident CTAs may hold before L2 starts to thrash
L2_CAND_TARGET = 16 << 20
CTA_FIXED_COST = 8000        # prologue + pipeline fill + epilogue drain of one CTA, SM clocks (~4 us)


@functools.lru_cache(maxsize=4096)
def _launch_plan(nu, ug, NT, b_bytes_per_group=0, unit_bytes=0, tile_cost=16384, max_tps=1 << 30):
    """static CTA partition of one launch: (groups, units per CTA, CTAs per group, N-tile splits, split_fast).

    L2 residency.  A CTA re-reads its unit's 128 candidate rows (unit_bytes) once per N tile, and all CTAs walk the
    fixed operand.  Which of the two stays in the 126 MB L2 depends on who is co-resident:
    * unit-fast order (default): neighbours hold different units and walk the same fixed-operand tiles at the same
      time, so those are fetched from HBM once -- provided one split's slice fits (enough splits are made that it
      does), and provided 148 units of candidate rows fit beside it;
    * split-fast order: for K >= 1536 they do not (148 x 786 KB at K=3072: ncu showed 2.7x the algorithmic DRAM
      reads), so the S CTAs that share one unit list are made neighbours instead: the unit's rows are fetched once
      and hit L2 for the other S-1 splits, and the ~148/S units that are co-resident still share fixed tiles.

    Wave quantisation.  All CTAs of a launch do equal work, so the launch takes ceil(CTAs / 148) rounds of the
    largest CTA; among the partitions the L2 rules allow, the one minimising rounds x (tiles per CTA x tile_cost +
    fixed CTA cost) is taken (tile_cost in SM clocks: the larger of the tile's MMA time and its 8 x BN TMEM read-out).
    max_tps: most N tiles one CTA may cover (the kernel stages column scales for at most 1024 columns per CTA)."""
    groups = nu // ug
    s_min, split_fast = min(NT, max(1, math.ceil(b_bytes_per_group / L2_SLICE_BYTES), math.ceil(NT / max_tps))), False
    if NT > 1 and unit_bytes * min(NUM_SMS, nu) > L2_CAND_BYTES:
        split_fast = True
        s_min = min(NT, max(s_min, math.ceil(unit_bytes * NUM_SMS / L2_CAND_TARGET)))
    best = None
    for S in range(s_min, min(NT, max(s_min, 16)) + 1):
        tps = math.ceil(NT / S)
        cands = {ug, 1}
        for w in range(1, 9):
            c = (NUM_SMS * w) // (groups * S)
            if c >= 1:
                cands.add(math.ceil(ug / min(c, ug)))
        for upc in cands:
            cpg = math.ceil(ug / upc)
            ctas = groups * cpg * S
            cost = math.ceil(ctas / NUM_SMS) * (math.ceil(ug / cpg) * tps * tile_cost + CTA_FIXED_COST)
            key = (cost, ctas)
            if best is None or key < best[0]:
                best = (key, upc, cpg, S)
    _, upc, cpg, S = best
    return groups, upc, cpg, S, split_fast


def run_cand_gemm(gen_cand, U, ka, UG, Bm, brpg, N, y, ldy, rs, rb=None, rs_div=1, rs_mod=1, cs=None, cb=None,
                  k_true=None, i8=False):
    """Chunk the units through the bf16 workspace: generate candidate rows, launch the fused GEMM.

    gen_cand(u0, nu, out) fills out[nu*128, ka] for units [u0, u0+nu).
    UG == U: one group (linear): returns [n_launch, 128]; else whole groups per launch: returns [U/UG, 128].

    The generator is ALU-bound and the GEMM tensor-core-bound, so with more than one chunk they run on two side
    streams over a double-buffered workspace: chunk i+1 is generated while chunk i is multiplied.  The chunk
    schedule (and therefore every partial sum) is identical in both modes.
    """
    dev = Bm.device
    single = UG == U
    unit_elems = ops.P_TILE * ka * (1 if i8 else 2)      # bytes of one unit's 128 candidate rows
    max_units = max(1, (WS_BYTES // 2) // unit_elems)
    step = min(U, max_units) if single else min(U, max(1, max_units // UG) * UG)
    n_chunks = (U + step - 1) // step
    BN = ops.pick_bn(N, 32 if rb is not None else 16)
    NT = (N + BN - 1) // BN
    overlap = n_chunks > 1 and dev.type == 'cuda'
    ws_all = _workspace(dev, (2 if overlap else 1) * step * unit_elems)
    bufs = [ws_all[:step * unit_elems], ws_all[step * unit_elems:]] if overlap else [ws_all]

    def gemm(u0, nu, buf):
        ug = nu if single else UG
        groups, upc, cpg, S, sf = _launch_plan(nu, ug, NT, N * ka * (1 if i8 else 2), unit_elems,
                                               max((ka // 64) * BN * (1 if i8 else 2), 8 * BN),
                                               (1024 // BN) if cs is not None else 1 << 30)
        part = ops.cand_gemm_err(buf, nu * ops.P_TILE, Bm, ka, N, nu, ug, brpg, 0 if single else u0 // UG, u0, y,
                                 u0 * ldy, ldy, rs, rb, rs_div, rs_mod, cs, cb, upc, S, BN, k_true, i8, sf)
        return part.view(S, groups, cpg, ops.P_TILE).sum(dim=(0, 2))

    outs = []
    if not overlap:
        for u0 in range(0, U, step):
            nu = min(step, U - u0)
            gen_cand(u0, nu, bufs[0])
            outs.append(gemm(u0, nu, bufs[0]))
        return torch.cat(outs, dim=0)

    main = torch.cuda.current_stream(dev)
    s_gen, s_mma = _side_streams(dev)
    start = main.record_event()
    s_gen.wait_event(start)
    s_mma.wait_event(start)
    freed = [None, None]
    for i, u0 in enumerate(range(0, U, step)):
        nu = min(step, U - u0)
        b = i & 1
        with torch.cuda.stream(s_gen):
            if freed[b] is not None:
                s_gen.wait_event(freed[b])
            gen_cand(u0, nu, bufs[b])
            ready = s_gen.record_event()
        with torch.cuda.stream(s_mma):
            s_mma.wait_event(ready)
            o = gemm(u0, nu, bufs[b])
            freed[b] = s_mma.record_event()
        o.record_stream(main)
        outs.append(o)
    main.wait_stream(s_gen)
    main.wait_stream(s_mma)
    return torch.cat(outs, dim=0)


def _f32(t):
    return t.detach().float().contiguous()


def _cand2d(cs, cz):
    """reference candidate tensors (candidate axis first) -> contiguous [P, G] float32 pair."""
    P = cs.shape[0]
    return _f32(cs).reshape(P, -1), _f32(cz).reshape(P, -1)


# ================================================================================================
# Linear family
# ================================================================================================
class LinearCtx:
    """Device-resident calibration tensors of one linear layer (raw_input / raw_out of the reference)."""

    def __init__(self, raw_input, raw_out, out_features):
        self.raw_input, self.raw_out = raw_input, raw_out
        self.x2d = _f32(raw_input).reshape(-1, raw_input.shape[-1])
        self.y2d = _f32(raw_out).reshape(-1, out_features)
        self.n_samples = raw_input.shape[0]
        adist.check_equal_shards(self.n_samples, 'linear raw_input')
        self.tok_per_sample = self.x2d.shape[0] // self.n_samples
        self._yT = None

    @property
    def yT(self):
        if self._yT is None:
            self._yT = self.y2d.t().contiguous()
        return self._yT


def uniform_operand_params(q):
    """(scale, round_ste(zp)) flattened, from a UniformQuantizer-like object."""
    s = _f32(q.scale).reshape(-1)
    z = _f32(q.zero_point).reshape(-1)
    return s, (z.round() - z) + z


def search_table_ints(n_levels, device):
    """integer numerators of the 37 live entries of the search LUT (linear.py:750-752 / matmul.py:313-315)."""
    return _const.search_table_ints(n_levels, device)


def linear_err_w_self(weight3, cs, cz, n_levels):
    """linear.py:296-309 -> similarities [P, n_V, rows]."""
    n_V, rows, in_f = weight3.shape
    c2, z2 = _cand2d(cs, cz)
    esum = ops.sweep_err_w_self(_f32(weight3).reshape(-1, in_f), c2, z2, n_levels)
    # similarity = -(sum / count); written as sum / -(count): bit-identical in IEEE arithmetic, one kernel less
    return (esum / -(in_f)).float().reshape(cs.shape[0], n_V, rows)


def linear_err_a_self(ctx, cs, cz, n_levels, channel_wise):
    """linear.py:320-345 -> similarities [C|1, P]."""
    esum = ops.sweep_err_a_self(ctx.x2d, _f32(cs), _f32(cz), n_levels, channel_wise)
    esum = adist.all_reduce_sum(esum)
    denom = ctx.tok_per_sample * (1 if channel_wise else ctx.x2d.shape[1])
    return (esum / -(denom)).float()


def _i8_ok(*n_levels):
    """uniform x uniform sweeps (every quantizer up to 7 bits: |code - zp| <= 127) run on the INT8 tensor cores
    (tcgen05.mma.kind::i8, S32 accumulation: exact) at twice the bf16 MMA rate and half the operand bytes"""
    return all(nl <= 64 for nl in n_levels)


FIXED_CACHE = True     # False rebuilds the fixed operand on every evaluation: the reference the cache is tested against


def _pkey(*tensors):
    """identity of quantizer parameters for the fixed-operand cache: (storage address, version counter, shape).  The
    quantizers' parameters are long-lived tensors written in place through quantizers/_ste.assign (which bumps the
    version), so equal keys mean equal values."""
    return tuple(None if t is None else (t.data_ptr(), t._version, tuple(t.shape)) for t in tensors)


def _cached_fixed(ctx, name, key, build):
    """The FIXED operand of a sweep -- the fake-quantised weight during an activation search, the fake-quantised
    activation during a weight search, the other matmul operand -- only changes when the fixed side's quantizer
    parameters do, i.e. once per search round, while a round scores it 6-18 times.  One entry per role on the module's
    calibration context (dropped with it in _finish): regenerating it per evaluation was 1.6% of a DeiT-S step in
    kernels plus ~5 launches per evaluation."""
    if not FIXED_CACHE or ctx is None:
        return build()
    cache = ctx.__dict__.setdefault('_fixed_cache', {})
    hit = cache.get(name)
    if hit is not None and hit[0] == key:
        return hit[1]
    val = build()
    cache[name] = (key, val)
    return val


def _is_adalog(q):
    return getattr(q, 'is_log', False) and hasattr(q, 'table2')


def _generic_fixed_operand(q, x2d):
    """A fake-quantised tensor with no (integer x one scale) form -- TwinUniform (two scales), Log2 / LogSqrt2 with
    their FP32 sqrt(2) factor and shift -- enters the tensor cores exactly as THREE bf16 pieces of its FP32 value
    (gen_split3, the patch-embedding trick): fixed operand [x_l | x_m | x_h], candidate operand replicated 3x along K."""
    with torch.no_grad():
        return ops.gen_split3(q(x2d))


def _fixed_act_operand(ctx, aq, i8=False):
    """quant_input(x) as an exact bf16 / int8 operand + the epilogue factors it implies.

    returns (Bm [tokens, krep * ka], a_scale FP64 [1], shift or None, krep)
    uniform:       x_hat = a_scale * I
    shift-adalog:  x_hat = a_scale/(4n-2) * (m 2^-e) - shift        (logarithm.py:127-135, not bias-reparamed)
    anything else: x_hat itself as three bf16 pieces (krep = 3)
    """
    if _is_adalog(aq):
        def build_log():
            nl = aq.n_levels
            m2 = torch.round(_f32(aq.table2) * (4 * nl - 2))
            Bm = ops.gen_log_fixed(ctx.x2d, aq.scale, aq.q, aq.shift, aq.table1, m2, nl)
            return Bm, _f32(aq.scale).double().reshape(1) / (4 * nl - 2), _f32(aq.shift).double().reshape(1), 1
        return _cached_fixed(ctx, 'act', ('log', aq.n_levels) + _pkey(aq.scale, aq.q, aq.shift, aq.table1, aq.table2),
                             build_log)
    if getattr(aq, 'is_log', False) or type(aq).__name__ != 'UniformQuantizer':
        return _generic_fixed_operand(aq, ctx.x2d), torch.ones(1, dtype=torch.float64, device=ctx.x2d.device), None, 3

    def build_uniform():
        s, z = uniform_operand_params(aq)
        Bm, _ = ops.gen_uniform_fixed(ctx.x2d, s, z, 1 << 62, 1, aq.n_levels, i8=i8)
        return Bm, s.double(), None, 1
    return _cached_fixed(ctx, 'act', ('uniform', aq.n_levels, bool(i8)) + _pkey(aq.scale, aq.zero_point), build_uniform)


def linear_err_w(ctx, weight3, bias, aq, cs, cz, n_levels_w):
    """linear.py:355-384 -> similarities [P, n_V, rows]."""
    n_V, rows, in_f = weight3.shape
    out_f = n_V * rows
    P = cs.shape[0]
    dev = weight3.device
    c2, z2 = _cand2d(cs, cz)                         # [P, out]
    i8 = type(aq).__name__ == 'UniformQuantizer' and _i8_ok(aq.n_levels, n_levels_w)
    Bm, a_scale, shift, krep = _fixed_act_operand(ctx, aq, i8)
    ka = krep * ops.kpad(in_f, i8)
    W2d = _f32(weight3).reshape(out_f, in_f)
    c2p = _pad128(c2.t().contiguous())               # [out, 128] candidate scales per row
    rs = (c2p.double() * a_scale).float().contiguous()
    b = _f32(bias) if bias is not None else torch.zeros(out_f, device=dev)
    rb = b.reshape(-1, 1).expand(out_f, ops.P_TILE).contiguous()
    rowsum = torch.empty(out_f, ops.P_TILE, dtype=torch.float32, device=dev) if shift is not None else None

    def gen(u0, nu, out):
        ops.gen_uniform_cand(W2d, u0, nu, c2, z2, P, out_f, 1, 1, out_f, n_levels_w, out, krep,
                             rowsum[u0:] if rowsum is not None else None, i8=i8)
        if shift is not None:
            # sum_k (v s - shift) w = s sum_k v w - shift sum_k w  (linear.py:879): fold the second term into the
            # row bias, using the integer row sums the generator just produced (same stream, ordered)
            rb[u0:u0 + nu] = (b[u0:u0 + nu].double().reshape(-1, 1)
                              - shift * c2p[u0:u0 + nu].double() * rowsum[u0:u0 + nu].double()).float()

    ntok = ctx.x2d.shape[0]
    res = run_cand_gemm(gen, out_f, ka, 1, Bm, 0, ntok, ctx.yT, ntok, rs, rb, 1, out_f, k_true=in_f, i8=i8)
    res = adist.all_reduce_sum(res)                  # [out, 128]
    sims = -(res[:, :P] / ctx.tok_per_sample)
    return sims.t().float().reshape(P, n_V, rows)


def _fixed_weight_operand(weight3, wq, i8=False, ctx=None):
    n_V, rows, in_f = weight3.shape

    def build():
        s, z = uniform_operand_params(wq)
        Bm, colsum = ops.gen_uniform_fixed(_f32(weight3).reshape(-1, in_f), s, z, 1, n_V * rows, wq.n_levels, not i8, i8)
        return Bm, s, colsum
    return _cached_fixed(ctx, 'weight', (wq.n_levels, bool(i8)) + _pkey(weight3, wq.scale, wq.zero_point), build)


def linear_quant_forward(x2d, weight3, bias, wq, aq, cache=None):
    """F.linear(Q_a(x), Q_w(W), b) of the inference forward (linear.py:46-51, :90-92) as ONE exact integer GEMM on the
    tensor cores: integer part of Q_a(x) (int8 when both quantizers have <= 7 bits, else bf16; AdaLog: m 2^-e in
    bf16) x integer part of Q_w(W), dequantised in the epilogue  out = s_a s_w[n] D + b[n]  (the post-GELU shift
    enters the bias: sum_k (v s - shift) w = s sum_k v w - shift sum_k w).  Returns None when the quantizer pair has
    no exact operand form (the caller then takes the generic torch path).  `cache`: dict kept by the module for the
    weight operand, which only changes when the weight or its quantizer parameters do."""
    n_V, rows, in_f = weight3.shape
    out_f = n_V * rows
    is_log = getattr(aq, 'is_log', False)
    if getattr(wq, 'sym', False) or wq.scale.numel() != out_f or wq.n_levels > 128:
        return None
    if is_log:
        if not hasattr(aq, 'table2') or aq.scale.numel() != 1 or 2 * aq.n_levels > 64:
            return None
    elif getattr(aq, 'sym', False) or aq.scale.numel() != 1 or aq.n_levels > 128 or type(aq).__name__ != 'UniformQuantizer':
        return None
    i8 = not is_log and _i8_ok(aq.n_levels, wq.n_levels)
    key = (weight3.data_ptr(), weight3._version, wq.scale.data_ptr(), wq.scale._version, wq.zero_point.data_ptr(),
           wq.zero_point._version, i8)
    if cache is not None and cache.get('key') == key:
        Bm, s_w, colsum = cache['val']
    else:
        Bm, s_w, colsum = _fixed_weight_operand(weight3, wq, i8)
        if colsum is None and is_log:
            colsum = None
        if cache is not None:
            cache['key'], cache['val'] = key, (Bm, s_w, colsum)
    dev = weight3.device
    b = _f32(bias) if bias is not None else torch.zeros(out_f, device=dev)
    M = x2d.shape[0]
    if is_log:
        nl = aq.n_levels
        m2 = torch.round(_f32(aq.table2) * (4 * nl - 2))
        A = ops.gen_log_fixed(x2d, aq.scale, aq.q, aq.shift, aq.table1, m2, nl)
        a_scale = _f32(aq.scale).double().reshape(1) / (4 * nl - 2)
        if not _flag(aq.bias_reparamed):
            b = (b.double() - _f32(aq.shift).double().reshape(1) * s_w.double() * colsum.double()).float()
    else:
        s_a, z_a = uniform_operand_params(aq)
        A, _ = ops.gen_uniform_fixed(x2d, s_a, z_a, 1 << 62, 1, aq.n_levels, i8=i8)
        a_scale = s_a.double()
    ka = ops.kpad(in_f, i8)
    rs = a_scale.float().expand(ops.P_TILE).contiguous()
    BN = ops.pick_bn(out_f)
    NT = (out_f + BN - 1) // BN
    U = (M + ops.P_TILE - 1) // ops.P_TILE
    _, upc, _, S, sf = _launch_plan(U, U, NT, out_f * ka * (1 if i8 else 2), ops.P_TILE * ka * (1 if i8 else 2),
                                    max((ka // 64) * BN * (1 if i8 else 2), 8 * BN), 1024 // BN)
    return ops.gemm_dequant(A, M, Bm, ka, out_f, rs, s_w.contiguous(), b.contiguous(), upc, S, i8, sf)


def linear_err_a(ctx, weight3, bias, wq, cs, cz, n_levels_a, y2d=None):
    """linear.py:394-423 -> similarities [1, P].  y2d: score against this target instead of raw_out (the twin-uniform
    search folds its fixed negative branch into it)."""
    n_V, rows, in_f = weight3.shape
    out_f = n_V * rows
    P = cs.shape[-1]
    dev = weight3.device
    i8 = _i8_ok(wq.n_levels, n_levels_a)
    Bm, s_w, _ = _fixed_weight_operand(weight3, wq, i8, ctx)
    c1, z1 = _f32(cs).reshape(-1), _f32(cz).reshape(-1)
    ka = ops.kpad(in_f, i8)

    def gen(u0, nu, out):
        ops.gen_uniform_cand(ctx.x2d, u0, nu, c1, z1, P, 1, 0, 1 << 62, 1, n_levels_a, out, i8=i8)

    rs = _pad128(c1).contiguous()
    cb = _f32(bias) if bias is not None else torch.zeros(out_f, device=dev)
    ntok = ctx.x2d.shape[0]
    y = ctx.y2d if y2d is None else y2d
    res = None
    passes = _lin_fused_passes()
    if out_f % 4 == 0 and passes is not None:
        # candidates generated inside the GEMM kernel: one launch, nothing expanded in HBM (lin_fused_gemm_err.cu)
        res = ops.lin_fused_cand_gemm_err(ctx.x2d, Bm, out_f, y, rs, s_w.contiguous(), cb.contiguous(), n_levels_a, P,
                                          c1, cz=z1, i8=i8, max_passes=passes)
    if res is None:
        res = run_cand_gemm(gen, ntok, ka, ntok, Bm, 0, out_f, y, out_f, rs, None, 1 << 62, 1, s_w, cb,
                            k_true=in_f, i8=i8)
    res = adist.all_reduce_sum(res.sum(dim=0, keepdim=True))
    return (res[:, :P] / -((ctx.tok_per_sample * out_f))).float()


def linear_err_a_twin(ctx, weight3, bias, wq, s_neg, cands, n_levels):
    """linear.py:664-690 (PTQ4ViT twin-uniform baseline): x_hat_p = clamp(rint(x/s_p), 0, n-1) s_p + x_neg with the
    negative branch x_neg = clamp(rint(x/s_neg), -n, 0) s_neg fixed.  The candidate branch is a uniform quantizer with
    zero point 0 and n levels (the device sweep of linear_err_a with n_levels/2); the fixed branch's contribution
    F.linear(x_neg, W_hat) is computed once and folded into the target.  -> similarities [P]."""
    n_V, rows, in_f = weight3.shape
    out_f = n_V * rows
    with torch.no_grad():
        w_hat = wq(weight3).reshape(out_f, in_f)
        x_neg = (ctx.x2d / s_neg.reshape(1)).round_().clamp_(-n_levels, 0) * s_neg.reshape(1)
        target = ctx.y2d - torch.nn.functional.linear(x_neg, w_hat)
    if n_levels < 2 or n_levels % 2:
        raise NotImplementedError('twin-uniform search needs n_bits >= 2')
    sims = linear_err_a(ctx, weight3, bias, wq, cands, torch.zeros_like(cands), n_levels // 2, y2d=target.contiguous())
    return sims.reshape(-1)


def linear_err_log(ctx, weight3, bias, wq, aq, cs, cq):
    """linear.py:856-890 (cs None: base-only search at the quantizer's current scale) and :898-931 -> [1, P]."""
    n_V, rows, in_f = weight3.shape
    out_f = n_V * rows
    P = cq.shape[-1]
    dev = weight3.device
    nl = aq.n_levels
    Bm, s_w, colsum = _fixed_weight_operand(weight3, wq, False, ctx)
    q1 = cq.detach().reshape(-1).to(torch.int64).contiguous()
    if cs is None:
        c1 = _f32(aq.scale).reshape(1).expand(P).contiguous()
    else:
        c1 = _f32(cs).reshape(-1)
    shift = _f32(aq.shift).reshape(1)
    mtab = search_table_ints(nl, dev)
    ka = ops.kpad(in_f)

    def gen(u0, nu, out):
        ops.gen_log_cand(ctx.x2d, u0, nu, c1, q1, P, shift, mtab, nl, out)

    rs = (_pad128(c1).double() / (4 * nl - 2)).float().contiguous()
    b = _f32(bias).double() if bias is not None else torch.zeros(out_f, device=dev, dtype=torch.float64)
    cb = (b - shift.double() * s_w.double() * colsum.double()).float().contiguous()
    ntok = ctx.x2d.shape[0]
    res = None
    passes = _lin_fused_passes()
    if out_f % 4 == 0 and passes is not None:
        res = ops.lin_fused_cand_gemm_err(ctx.x2d, Bm, out_f, ctx.y2d, rs, s_w.contiguous(), cb, nl, P, c1, cq=q1,
                                          shift=shift, mtab=mtab, max_passes=passes)
    if res is None:
        res = run_cand_gemm(gen, ntok, ka, ntok, Bm, 0, out_f, ctx.y2d, out_f, rs, None, 1 << 62, 1, s_w, cb,
                            k_true=in_f)
    res = adist.all_reduce_sum(res.sum(dim=0, keepdim=True))
    return (res[:, :P] / -((ctx.tok_per_sample * out_f))).float()


# ================================================================================================
# MatMul family.  A [B,H,S,Kd] @ Bop [B,H,Kd,S2]  (matmul.py:48-56)
# ================================================================================================
class MatMulCtx:
    def __init__(self, A, B, raw_out):
        self.raw_input, self.raw_out = [A, B], raw_out
        A, B, raw_out = _f32(A), _f32(B), _f32(raw_out)
        self.Bn, self.H, self.S1, self.Kd = A.shape
        adist.check_equal_shards(self.Bn, 'matmul raw_input')
        self.S2 = B.shape[-1]
        self.A2d = A.reshape(-1, self.Kd)                                   # rows (b,h,s1)
        self.Bt2d = B.transpose(-2, -1).contiguous().reshape(-1, self.Kd)   # rows (b,h,s2)
        self.y2d = raw_out.reshape(-1, self.S2)                             # rows (b,h,s1), cols s2
        self._yT = None
        self._raw_out = raw_out

    @property
    def yT2d(self):
        if self._yT is None:
            self._yT = self._raw_out.transpose(-2, -1).contiguous().reshape(-1, self.S1)  # rows (b,h,s2), cols s1
        return self._yT


def _head_params(q, H):
    s, z = uniform_operand_params(q)
    if s.numel() == 1:
        s, z = s.expand(H).contiguous(), z.expand(H).contiguous()
    return s, z


def _matmul_reduce(res, ctx, P, head_channel_wise, pool_heads, n_cols_total):
    """res [B*H, 128] FP64 sums -> similarities in the reference's layout."""
    res = res.view(ctx.Bn, ctx.H, ops.P_TILE).sum(dim=0)          # [H, 128]
    res = adist.all_reduce_sum(res)
    if head_channel_wise and not pool_heads:
        return (res[:, :P] / -(n_cols_total)).t().float().contiguous()      # [P, H]
    tot = res.sum(dim=0)
    return (tot[:P] / -((n_cols_total * ctx.H))).float()                    # [P]


# False sends every attention sweep through generator -> workspace -> GEMM: the path the fused kernel is tested against
FUSED = True


@functools.lru_cache(maxsize=1024)
def _fused_upc(groups, ug, K, N):
    """units per CTA of the fused kernel: a CTA stays inside one group (it loads the group's fixed operand once), all
    CTAs do equal work, so the launch takes ceil(CTAs / 148) rounds of the largest CTA."""
    unit_cost = 10 * K + 10 * N            # worker-warp clocks per unit: generation ~ K, error arithmetic ~ N
    best = None
    for cpg in range(1, min(ug, 16) + 1):
        upc = math.ceil(ug / cpg)
        ctas = groups * math.ceil(ug / upc)
        cost = math.ceil(ctas / NUM_SMS) * (upc * unit_cost + CTA_FIXED_COST)
        if best is None or cost < best[0]:
            best = (cost, upc)
    return best[1]


def _use_fused(K, N, i8, log, n_levels):
    """The fused generator + GEMM kernel is taken where it measured faster than generator -> workspace -> GEMM
    (DeiT-S, 128 images: QK^T sweeps 1.95 vs 2.44 ms, P.V base search 5.3 vs 5.8 ms); for a uniform candidate side with
    a long reduction (P.V value sweep, K = 197) its 14 worker warps are short of issue slots (2.3 vs 1.9 ms)."""
    return FUSED and ops.fused_plan(K, N, i8, log, n_levels) is not None and (log or K <= 128)


def _run_fused(x2d, K, Bm, N, U, UG, y, ldy, rs, H, n_levels, P, i8=False, **cand):
    """all units of an attention sweep in ONE launch of the fused generator + GEMM kernel -> [U/UG, 128] FP64"""
    upc = _fused_upc(U // UG, UG, K, N)
    part = ops.fused_cand_gemm_err(x2d, K, Bm, N, U, UG, N, y, ldy, rs, UG, H, upc, n_levels, P, i8=i8, **cand)
    return part.view(U // UG, -1, ops.P_TILE).sum(dim=1)


def matmul_err_A(ctx, Bq, cs, cz, n_levels_A, head_channel_wise):
    """matmul.py:135-163: candidates on A, fixed quantised B -> [P, H] (or [P])."""
    P = cs.shape[0]
    H = ctx.H
    c2, z2 = _cand2d(cs, cz)                                     # [P, H] or [P, 1]
    gs = 1 if c2.shape[1] == H else 0
    i8 = False       # bf16 operands: at K = 64 an int8 row is as long, and the fused int8 producer measured slower
    fused = _use_fused(ctx.Kd, ctx.S2, i8, False, n_levels_A)
    Bm, sB = _fixed_B_operand(ctx, Bq, i8)
    ka = ops.kpad(ctx.Kd)

    def gen(u0, nu, out):
        ops.gen_uniform_cand(ctx.A2d, u0, nu, c2, z2, P, c2.shape[1], gs, ctx.S1, H, n_levels_A, out)

    cfull = c2 if gs else c2.expand(P, H)
    rs = (_pad128(cfull.t().contiguous()).double() * sB.double().reshape(H, 1)).float().contiguous()   # [H,128]
    U = ctx.Bn * H * ctx.S1
    if fused:
        res = _run_fused(ctx.A2d, ctx.Kd, Bm, ctx.S2, U, ctx.S1, ctx.y2d, ctx.S2, rs, H, n_levels_A, P, i8=i8,
                         cs=c2, cz=z2, pstride=c2.shape[1], gstride=gs, g_div=ctx.S1, g_mod=H)
    else:
        res = run_cand_gemm(gen, U, ka, ctx.S1, Bm, ctx.S2, ctx.S2, ctx.y2d, ctx.S2, rs, None, ctx.S1, H,
                            k_true=ctx.Kd)
    return _matmul_reduce(res, ctx, P, head_channel_wise, False, ctx.S1 * ctx.S2)


def _fixed_B_operand(ctx, Bq, i8=False):
    """quant_input_B(B), transposed rows (b,h,s2), as a bf16 (or int8) operand; returns (Bm, per-head scale [H])."""
    H = ctx.H

    def build():
        sB, zB = _head_params(Bq, H)
        Bm, _ = ops.gen_uniform_fixed(ctx.Bt2d, sB, zB, ctx.S2, H, Bq.n_levels, i8=i8)
        return Bm, sB
    return _cached_fixed(ctx, 'B', (Bq.n_levels, bool(i8)) + _pkey(Bq.scale, Bq.zero_point), build)


def _fixed_A_operand(ctx, Aq, i8=False):
    """quant_input_A(A) as a bf16 (or int8) operand, rows (b,h,s1); returns (Bm, per-head scale FP64 [H], krep)."""
    H = ctx.H
    if _is_adalog(Aq):
        def build_log():
            nl = Aq.n_levels
            m2 = torch.round(_f32(Aq.table2) * (4 * nl - 2))
            Bm = ops.gen_log_fixed(ctx.A2d, Aq.scale, Aq.q, None, Aq.table1, m2, nl)
            return Bm, (_f32(Aq.scale).double().reshape(1) / (4 * nl - 2)).expand(H), 1
        return _cached_fixed(ctx, 'A', ('log', Aq.n_levels) + _pkey(Aq.scale, Aq.q, Aq.table1, Aq.table2), build_log)
    if getattr(Aq, 'is_log', False):
        # post_softmax_quantizer 'log2' / 'logsqrt2' (matmul.py:307-310): per-tensor scale, values 2^-k [x sqrt(2)]
        return _generic_fixed_operand(Aq, ctx.A2d), torch.ones(H, dtype=torch.float64, device=ctx.A2d.device), 3

    def build_uniform():
        sA, zA = _head_params(Aq, H)
        Bm, _ = ops.gen_uniform_fixed(ctx.A2d, sA, zA, ctx.S1, H, Aq.n_levels, i8=i8)
        return Bm, sA.double(), 1
    return _cached_fixed(ctx, 'A', ('uniform', Aq.n_levels, bool(i8)) + _pkey(Aq.scale, Aq.zero_point), build_uniform)


def matmul_err_B(ctx, Aq, cs, cz, n_levels_B, head_channel_wise):
    """matmul.py:173-201: candidates on B (its rows are the columns of the product), fixed quantised A."""
    P = cs.shape[0]
    H = ctx.H
    c2, z2 = _cand2d(cs, cz)
    gs = 1 if c2.shape[1] == H else 0
    i8 = False
    Bm, sA, krep = _fixed_A_operand(ctx, Aq, i8)
    fused = krep == 1 and _use_fused(ctx.Kd, ctx.S1, i8, False, n_levels_B)
    ka = krep * ops.kpad(ctx.Kd)

    def gen(u0, nu, out):
        ops.gen_uniform_cand(ctx.Bt2d, u0, nu, c2, z2, P, c2.shape[1], gs, ctx.S2, H, n_levels_B, out, krep)

    cfull = c2 if gs else c2.expand(P, H)
    rs = (_pad128(cfull.t().contiguous()).double() * sA.reshape(H, 1)).float().contiguous()
    U = ctx.Bn * H * ctx.S2
    if fused:
        res = _run_fused(ctx.Bt2d, ctx.Kd, Bm, ctx.S1, U, ctx.S2, ctx.yT2d, ctx.S1, rs, H, n_levels_B, P, i8=i8,
                         cs=c2, cz=z2, pstride=c2.shape[1], gstride=gs, g_div=ctx.S2, g_mod=H)
    else:
        res = run_cand_gemm(gen, U, ka, ctx.S2, Bm, ctx.S1, ctx.S1, ctx.yT2d, ctx.S1, rs, None, ctx.S2, H,
                            k_true=ctx.Kd)
    return _matmul_reduce(res, ctx, P, head_channel_wise, False, ctx.S1 * ctx.S2)


def matmul_err_A_log_base(ctx, Bq, cq, n_levels_A):
    """matmul.py:321-351: candidate log bases on the post-softmax operand, all heads pooled -> [P, 1]."""
    P = cq.shape[0]
    H = ctx.H
    dev = ctx.A2d.device
    q1 = cq.detach().reshape(-1).to(torch.int64).contiguous()
    Bm, sB = _fixed_B_operand(ctx, Bq)
    mtab = search_table_ints(n_levels_A, dev)
    ka = ops.kpad(ctx.Kd)

    def gen(u0, nu, out):
        ops.gen_log_cand(ctx.A2d, u0, nu, None, q1, P, None, mtab, n_levels_A, out)

    rs = (sB.double().reshape(H, 1) / (4 * n_levels_A - 2)).expand(H, ops.P_TILE).float().contiguous()
    U = ctx.Bn * H * ctx.S1
    if _use_fused(ctx.Kd, ctx.S2, False, True, n_levels_A):
        res = _run_fused(ctx.A2d, ctx.Kd, Bm, ctx.S2, U, ctx.S1, ctx.y2d, ctx.S2, rs, H, n_levels_A, P,
                         cq=q1, mtab=mtab, g_div=ctx.S1, g_mod=H)
    else:
        res = run_cand_gemm(gen, U, ka, ctx.S1, Bm, ctx.S2, ctx.S2, ctx.y2d, ctx.S2, rs, None, ctx.S1, H,
                            k_true=ctx.Kd)
    return _matmul_reduce(res, ctx, P, True, True, ctx.S1 * ctx.S2).reshape(P, 1)


# ================================================================================================
# Conv (patch embedding: kernel == stride, no padding) -- conv.py:226-256 with raw FP32 input (a_bit >= 8)
# ================================================================================================
class ConvCtx:
    def __init__(self, raw_input, raw_out, kernel_size):
        self.raw_input, self.raw_out = raw_input, raw_out
        x, y = _f32(raw_input), _f32(raw_out)
        Bn, ic, Hh, Ww = x.shape
        kh, kw = kernel_size
        oh, ow = Hh // kh, Ww // kw
        patches = x.reshape(Bn, ic, oh, kh, ow, kw).permute(0, 2, 4, 1, 3, 5).reshape(Bn * oh * ow, ic * kh * kw)
        self.n_samples = Bn
        adist.check_equal_shards(Bn, 'conv raw_input')
        self.pos_per_sample = oh * ow
        self.x3 = ops.gen_split3(patches.contiguous())                 # [tokens, 3*ka]
        oc = y.shape[1]
        self.yT = y.permute(1, 0, 2, 3).reshape(oc, -1).contiguous()   # [oc, tokens]
        self.K = ic * kh * kw


def conv_err_w(ctx, weight2d, bias, cs, cz, n_levels_w):
    """conv.py:226-256 -> similarities [P, oc]."""
    oc, K = weight2d.shape
    P = cs.shape[0]
    dev = weight2d.device
    c2, z2 = _cand2d(cs, cz)                                       # [P, oc]
    W2d = _f32(weight2d)
    ka = 3 * ops.kpad(K)

    def gen(u0, nu, out):
        ops.gen_uniform_cand(W2d, u0, nu, c2, z2, P, oc, 1, 1, oc, n_levels_w, out, 3)

    rs = _pad128(c2.t().contiguous()).contiguous()
    b = _f32(bias) if bias is not None else torch.zeros(oc, device=dev)
    rb = b.reshape(-1, 1).expand(oc, ops.P_TILE).contiguous()
    ntok = ctx.yT.shape[1]
    res = run_cand_gemm(gen, oc, ka, 1, ctx.x3, 0, ntok, ctx.yT, ntok, rs, rb, 1, oc, k_true=K)
    res = adist.all_reduce_sum(res)
    return (res[:, :P] / -(ctx.pos_per_sample)).t().float().contiguous()
