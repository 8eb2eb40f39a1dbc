"""Quantised nn.Linear family with the reference's class API (quant_layers/linear.py).

Same class names, constructor signatures, attributes (`mode`, `calibrated`, `raw_input`, `raw_out`, `tmp_input`,
`tmp_out`, `w_quantizer`, `a_quantizer`, `n_V`, `crb_rows`, `prev_layer`) and state_dict layout, so
utils/calibrator.py, utils/wrap_net.py, test_quant.py and the reference's BRECQ code drive them unchanged.
What differs is underneath: every `_search_best_*` evaluation is one fused device sweep (adalog_b200/sweep.py ->
libadalog_b200.so) over HBM-resident calibration tensors instead of a Python loop over 32-sample batches and
candidate chunks, and the refinement loop is the shared driver in _fpcs.py.
"""
import torch
import torch.nn as nn
import torch.nn.functional as F

from .. import _const, sweep
from ..quantizers.uniform import UniformQuantizer, TwinUniformQuantizer
from ..quantizers.logarithm import ShiftAdaLogQuantizer, ShiftLog2Quantizer, ShiftLogSqrt2Quantizer
from ..utils import dist as adist
from ..quantizers._ste import assign
from . import _fpcs

__all__ = ['MinMaxQuantLinear', 'PTQSLQuantLinear', 'PTQSLBatchingQuantLinear', 'AsymmetricallyBatchingQuantLinear',
           'AsymmetricallyChannelWiseBatchingQuantLinear', 'PostGeluTwinUniformBatchingQuantLinear',
           'PostGeluLogBasedBatchingQuantLinear']

GELU_MIN = 0.16997124254703522     # -min GELU(x); the post-GELU shift (reference linear.py:749)


class MinMaxQuantLinear(nn.Linear):
    """reference: quant_layers/linear.py:8-61"""

    def __init__(self, in_features: int, out_features: int, bias: bool = True, mode="raw", w_bit=8, a_bit=8):
        super().__init__(in_features, out_features, bias)
        self.mode = mode
        self.w_quantizer = UniformQuantizer(n_bits=w_bit, symmetric=True, channel_wise=False)
        self.a_quantizer = UniformQuantizer(n_bits=a_bit, symmetric=True, channel_wise=False)
        self.raw_input = None
        self.raw_out = None
        self.tmp_input = None
        self.tmp_out = None
        self.calibrated = False

    def forward(self, x):
        if self.mode == 'raw':
            return F.linear(x, self.weight, self.bias)
        if self.mode == 'quant_forward':
            return self.quant_forward(x)
        if self.mode == 'debug_only_quant_weight':
            return self.debug_only_quant_weight(x)
        if self.mode == 'debug_only_quant_act':
            return self.debug_only_quant_act(x)
        raise NotImplementedError

    def quant_weight_bias(self):
        return self.w_quantizer(self.weight), self.bias if self.bias is not None else None

    def quant_input(self, x):
        return self.a_quantizer(x)

    def quant_forward(self, x):
        assert self.calibrated, f"Module should be calibrated before run quant_forward for {self}"
        w_sim, bias_sim = self.quant_weight_bias()
        return F.linear(self.quant_input(x), w_sim, bias_sim)

    def debug_only_quant_weight(self, x):
        w_sim, bias_sim = self.quant_weight_bias()
        return F.linear(x, w_sim, bias_sim)

    def debug_only_quant_act(self, x):
        return F.linear(self.quant_input(x), self.weight, self.bias)


class PTQSLQuantLinear(MinMaxQuantLinear):
    """reference: quant_layers/linear.py:64-92 (row-block weight quantisation, n_V sub-matrices)"""

    # tensor-core inference forward (see quant_forward): opt-in, because the default forward is bit-identical to the
    # reference's F.linear(Q_a(x), Q_w(W), b) and calibration of later layers consumes it; enable per model with
    # utils.wrap_net.set_tensor_core_forward(model, True)
    tc_forward = False

    def __init__(self, in_features: int, out_features: int, bias: bool = True, mode="raw", w_bit=8, a_bit=8,
                 search_round=1, eq_n=100, n_V=1):
        super().__init__(in_features, out_features, bias=bias, mode=mode, w_bit=w_bit, a_bit=a_bit)
        self.w_quantizer = UniformQuantizer(n_bits=w_bit, symmetric=True, channel_wise=True)
        self.a_quantizer = UniformQuantizer(n_bits=a_bit, symmetric=True, channel_wise=False)
        self.search_round = search_round
        self.eq_n = eq_n
        self.parallel_eq_n = eq_n
        self.n_V = n_V
        self.crb_rows = out_features // n_V
        self.w_quantizer.scale = nn.Parameter(torch.zeros((n_V, self.crb_rows, 1)))
        self.a_quantizer.scale = nn.Parameter(torch.zeros((1)))

    def _get_similarity(self, tensor_raw, tensor_sim):
        return -(tensor_raw - tensor_sim) ** 2

    def _weight3(self):
        return self.weight.view(self.n_V, self.crb_rows, self.in_features)

    def quant_weight_bias(self):
        w_sim = self.w_quantizer(self._weight3()).view(self.out_features, self.in_features)
        return w_sim, self.bias if self.bias is not None else None

    def quant_forward(self, x):
        """reference linear.py:46-51 with :90-92: F.linear(Q_a(x), Q_w(W), b), bit-identical to the reference's
        composition (the quantizers are the sm_100a kernels, the product is FP32).  With `tc_forward` enabled
        (set_tensor_core_forward; inference only: no grad, no training_mode) the same product is ONE exact integer
        GEMM on the tensor cores with the dequantisation in its epilogue
        (sweep.linear_quant_forward; weight operand cached until the weight or its quantizer changes): equal to the
        FP32 composition to FP32 rounding (<= 2e-5 of the output range, tests/test_gpu_gemm.py), not bit for bit."""
        assert self.calibrated, f"Module should be calibrated before run quant_forward for {self}"
        if (self.tc_forward and x.is_cuda and x.dtype == torch.float32 and not torch.is_grad_enabled()
                and not self.w_quantizer.training_mode and not self.a_quantizer.training_mode
                and self.w_quantizer.n_bits < 32 and self.a_quantizer.n_bits < 32):
            cache = self.__dict__.setdefault('_tc_cache', {})
            x2d = x.reshape(-1, self.in_features)
            if not x2d.is_contiguous():
                x2d = x2d.contiguous()
            out = sweep.linear_quant_forward(x2d, self._weight3(), self.bias, self.w_quantizer, self.a_quantizer, cache)
            if out is not None:
                return out.view(*x.shape[:-1], self.out_features)
        w_sim, bias_sim = self.quant_weight_bias()
        return F.linear(self.quant_input(x), w_sim, bias_sim)


class PTQSLBatchingQuantLinear(PTQSLQuantLinear):
    """reference: quant_layers/linear.py:95-235.  The symmetric PTQ4ViT-style search of this base class is dead
    code in the reference (it dereferences an undefined name at linear.py:171); only its constructor and
    `_initialize_calib_parameters` are inherited by the live classes below."""

    def __init__(self, in_features: int, out_features: int, bias: bool = True, mode="raw", w_bit=8, a_bit=8,
                 calib_batch_size=32, search_round=1, eq_n=100, n_V=1):
        super().__init__(in_features, out_features, bias=bias, mode=mode, w_bit=w_bit, a_bit=a_bit,
                         search_round=search_round, eq_n=eq_n, n_V=n_V)
        self.calib_batch_size = calib_batch_size

    def _initialize_calib_parameters(self):
        """reference linear.py:111-121.  The calibration tensors are moved to (and stay in) HBM; candidate chunking
        is decided by the bf16 workspace in sweep.run_cand_gemm, so parallel_eq_n is informational only."""
        dev = self.weight.device
        sweep.require_cuda(dev)
        self.calib_size = self.raw_input.shape[0]
        self.parallel_eq_n = self.eq_n
        self._ctx = sweep.LinearCtx(self.raw_input.to(dev), self.raw_out.to(dev), self.out_features)

    def hyperparameter_searching(self):
        raise NotImplementedError('the symmetric PTQSL search is unreachable in the reference (linear.py:171 uses an '
                                  'undefined name); use the Asymmetrically* classes')


class AsymmetricallyBatchingQuantLinear(PTQSLBatchingQuantLinear):
    """reference: quant_layers/linear.py:238-545 (proj, head; qkv/fc1/reduction after reparam)"""

    def __init__(self, in_features: int, out_features: int, bias: bool = True, mode="raw", w_bit=8, a_bit=8,
                 calib_batch_size=32, search_round=1, eq_n=100, n_V=1, fpcs=False, steps=4):
        super().__init__(in_features, out_features, bias=bias, mode=mode, w_bit=w_bit, a_bit=a_bit,
                         calib_batch_size=calib_batch_size, search_round=search_round, eq_n=eq_n, n_V=n_V)
        self.fpcs = fpcs
        self.steps = steps
        del self.a_quantizer, self.w_quantizer
        self.w_quantizer = UniformQuantizer(n_bits=w_bit, symmetric=False, channel_wise=True)
        self.a_quantizer = UniformQuantizer(n_bits=a_bit, symmetric=False, channel_wise=False)
        self.a_quantizer.scale = nn.Parameter(torch.zeros((1)))
        self.a_quantizer.zero_point = nn.Parameter(torch.zeros((1)))
        self.w_quantizer.scale = nn.Parameter(torch.zeros((n_V, self.crb_rows, 1)))
        self.w_quantizer.zero_point = nn.Parameter(torch.zeros((n_V, self.crb_rows, 1)))

    # ------------------------------------------------------------------ selection helpers
    def _scored(self, fn, cs, cz, axis):
        """score <=128 candidates per device pass and concatenate along the candidate axis"""
        P = cs.shape[axis]
        parts = []
        for p0, p1 in _fpcs.candidate_chunks(P):
            sl = (slice(p0, p1),) if axis == 0 else (Ellipsis, slice(p0, p1))
            parts.append(fn(cs[sl], cz[sl]))
        return parts[0] if len(parts) == 1 else torch.cat(parts, dim=axis)

    def _store_w(self, cs, cz, idx):
        assign(self.w_quantizer.scale, torch.gather(cs, dim=0, index=idx).squeeze(0))
        assign(self.w_quantizer.zero_point, torch.gather(cz, dim=0, index=idx).squeeze(0))

    def _store_a(self, cs, cz, idx):
        assign(self.a_quantizer.scale, torch.gather(cs, dim=-1, index=idx).squeeze(-1))
        assign(self.a_quantizer.zero_point, torch.gather(cz, dim=-1, index=idx).squeeze(-1))

    # ------------------------------------------------------------------ the four evaluations
    def _search_best_w_scale_self(self, weight_scale_candidates, weight_zero_point_candidates, topk=1):
        """reference linear.py:296-318"""
        nl = self.w_quantizer.n_levels
        sims = self._scored(lambda s, z: sweep.linear_err_w_self(self._weight3(), s, z, nl),
                            weight_scale_candidates, weight_zero_point_candidates, 0)
        _, best = torch.topk(sims, k=topk, dim=0)
        best = best.reshape(topk, self.n_V, -1, 1)
        if topk == 1:
            self._store_w(weight_scale_candidates, weight_zero_point_candidates, best)
            self.w_quantizer.inited = True
        return best.squeeze(0)

    def _search_best_a_scale_self(self, input_scale_candidates, input_zero_point_candidates, topk=1):
        """reference linear.py:320-353"""
        nl, cw = self.a_quantizer.n_levels, self.a_quantizer.channel_wise
        sims = self._scored(lambda s, z: sweep.linear_err_a_self(self._ctx, s, z, nl, cw),
                            input_scale_candidates, input_zero_point_candidates, -1)
        _, best = torch.topk(sims, k=topk, dim=-1)
        if topk == 1:
            self._store_a(input_scale_candidates, input_zero_point_candidates, best)
            self.a_quantizer.inited = True
        return best

    def _search_best_w_scale(self, weight_scale_candidates, weight_zero_point_candidates, topk=1):
        """reference linear.py:355-392"""
        nl = self.w_quantizer.n_levels
        sims = self._scored(lambda s, z: sweep.linear_err_w(self._ctx, self._weight3(), self.bias, self.a_quantizer,
                                                            s, z, nl),
                            weight_scale_candidates, weight_zero_point_candidates, 0)
        _, best = torch.topk(sims, k=topk, dim=0)
        best = best.reshape(topk, self.n_V, -1, 1)
        if topk == 1:
            self._store_w(weight_scale_candidates, weight_zero_point_candidates, best)
        return best.squeeze(0)

    def _search_best_a_scale(self, input_scale_candidates, input_zero_point_candidates, topk=1):
        """reference linear.py:394-430"""
        nl = self.a_quantizer.n_levels
        sims = self._scored(lambda s, z: sweep.linear_err_a(self._ctx, self._weight3(), self.bias, self.w_quantizer,
                                                            s, z, nl),
                            input_scale_candidates, input_zero_point_candidates, -1)
        _, best = torch.topk(sims, k=topk, dim=-1)
        if topk == 1:
            self._store_a(input_scale_candidates, input_zero_point_candidates, best)
        return best

    # ------------------------------------------------------------------ candidate seeding
    def calculate_percentile_weight_candidates(self, l=0.9, r=1.0):
        """reference linear.py:432-451"""
        nl = self.w_quantizer.n_levels
        num_zp = min(16, nl)
        num_scale = int(self.eq_n / num_zp)
        pct = torch.tensor([l, r])
        w3 = self._weight3()
        up, lo = _fpcs.quantile_pair(w3, pct, -1, local=True)        # weights are replicated, not sharded
        up, lo = up.unsqueeze(-1), lo.unsqueeze(-1)
        return _fpcs.percentile_grid(up[0:1] - lo[0:1], up[1:] - lo[1:], nl, num_zp, num_scale, 0, 3)

    def calculate_percentile_activation_candidates(self, l=0.9, r=1.0):
        """reference linear.py:453-481.  Under data parallelism the order statistics are taken over the
        all-gathered activations so every rank seeds the same grid as a single process would."""
        nl = self.a_quantizer.n_levels
        num_zp = min(16, nl * 2)
        num_scale = int(self.eq_n / num_zp)
        pct = torch.tensor([l, r])
        # the calibration input of a module does not change between its search rounds: sort it once
        key = (bool(self.a_quantizer.channel_wise), l, r)
        cache = self._ctx.__dict__.setdefault('_pct_cache', {})
        if key not in cache:
            x = self._ctx.x2d                      # this rank's samples; the helpers select across ranks exactly
            if self.a_quantizer.channel_wise:
                up, lo = _fpcs.quantile_pair(x.reshape(-1, self.in_features), pct, 0)
            else:
                up, lo = _fpcs.chunked_quantile(x.reshape(1, 1, -1), pct)
            cache[key] = (up.transpose(0, 1), lo.transpose(0, 1))    # [C|1, 2]
        up, lo = cache[key]
        scales, zps = _fpcs.percentile_grid(up[:, 0:1] - lo[:, 0:1], up[:, 1:] - lo[:, 1:], nl, num_zp, num_scale, -1)
        return scales.clamp(min=1e-4), zps

    # ------------------------------------------------------------------ FPCS drivers
    def weight_fpcs(self, fpcs_width=16, steps=6, search_strategy=None):
        """reference linear.py:483-502"""
        cs, cz = self.calculate_percentile_weight_candidates()
        _fpcs.search(cs, cz, lambda s, z, k: search_strategy(self, s, z, topk=k), 0, self.eq_n, fpcs_width, steps)

    def activation_fpcs(self, fpcs_width=16, steps=6, search_strategy=None):
        """reference linear.py:504-523"""
        cs, cz = self.calculate_percentile_activation_candidates()
        _fpcs.search(cs, cz, lambda s, z, k: search_strategy(self, s, z, topk=k), -1, self.eq_n, fpcs_width, steps,
                     floor=1e-4)

    def _finish(self):
        self.calibrated = True
        del self.raw_input, self.raw_out
        self._ctx = None

    def hyperparameter_searching(self):
        """reference linear.py:525-545"""
        cls = AsymmetricallyBatchingQuantLinear
        self._initialize_calib_parameters()
        if self.fpcs:
            self.weight_fpcs(steps=self.steps, search_strategy=cls._search_best_w_scale_self)
            self.activation_fpcs(steps=self.steps, search_strategy=cls._search_best_a_scale_self)
        else:
            w_cs, w_cz = self.calculate_percentile_weight_candidates()
            a_cs, a_cz = self.calculate_percentile_activation_candidates()
            self._search_best_w_scale_self(w_cs, w_cz)
            self._search_best_a_scale_self(a_cs, a_cz)
        for _ in range(self.search_round):
            if self.fpcs:
                self.weight_fpcs(steps=self.steps, search_strategy=cls._search_best_w_scale)
                self.activation_fpcs(steps=self.steps, search_strategy=cls._search_best_a_scale)
            else:
                self._search_best_w_scale(w_cs, w_cz)
                self._search_best_a_scale(a_cs, a_cz)
        self._finish()
        return None


class AsymmetricallyChannelWiseBatchingQuantLinear(AsymmetricallyBatchingQuantLinear):
    """reference: quant_layers/linear.py:548-621 (qkv, fc1, Swin reduction): per-channel activation search,
    then scale reparameterisation into the preceding LayerNorm and the per-tensor search."""

    def __init__(self, in_features: int, out_features: int, bias: bool = True, mode="raw", w_bit=8, a_bit=8,
                 calib_batch_size=None, search_round=1, eq_n=100, n_V=1, fpcs=False, steps=4):
        super().__init__(in_features, out_features, bias=bias, mode=mode, w_bit=w_bit, a_bit=a_bit,
                         calib_batch_size=calib_batch_size, search_round=search_round, eq_n=eq_n, n_V=n_V, fpcs=fpcs,
                         steps=steps)
        del self.a_quantizer
        self.a_quantizer = UniformQuantizer(n_bits=a_bit, symmetric=False, channel_wise=True)
        self.a_quantizer.scale = nn.Parameter(torch.zeros((in_features)))
        self.a_quantizer.zero_point = nn.Parameter(torch.zeros((in_features)))
        self._prev_layer = None

    def __setattr__(self, name, value):
        # keep the LayerNorm out of _modules / state_dict (reference linear.py:571-583)
        if name == "prev_layer":
            self.__dict__['_prev_layer'] = value
        else:
            super().__setattr__(name, value)

    @property
    def prev_layer(self):
        return self._prev_layer

    def hyperparameter_searching(self):
        """reference linear.py:585-594"""
        assert self.a_quantizer.channel_wise and self.w_quantizer.channel_wise
        self._initialize_calib_parameters()
        if self.fpcs:
            self.activation_fpcs(steps=self.steps,
                                 search_strategy=AsymmetricallyBatchingQuantLinear._search_best_a_scale_self)
        else:
            a_cs, a_cz = self.calculate_percentile_activation_candidates()
            self._search_best_a_scale_self(a_cs, a_cz)
        self.calibrated = True

    def reparam_step1(self):
        """reference linear.py:596-612"""
        self.calibrated = False
        aq = self.a_quantizer
        channel_min = -aq.zero_point * aq.scale
        target_scale = torch.mean(aq.scale).view(1)
        target_zero_point = torch.mean(aq.zero_point).round().view(1)
        target_min = -target_zero_point * target_scale
        r = aq.scale / target_scale
        b = channel_min / r - target_min
        self.prev_layer.weight.data = self.prev_layer.weight.data / r
        self.prev_layer.bias.data = self.prev_layer.bias.data / r.view(-1) - b
        self.weight.data = self.weight.data * r.view(1, -1)
        folded = torch.mm(self.weight.data, b.reshape(-1, 1)).reshape(-1)
        if self.bias is not None:
            self.bias.data = self.bias.data + folded
        else:
            self.bias = nn.Parameter(torch.zeros(self.out_features))
            self.bias.data = folded
        return r, b, target_scale, target_zero_point

    def reparam(self):
        """reference linear.py:614-621"""
        r, b, target_scale, target_zero_point = self.reparam_step1()
        self.raw_input = (self.raw_input.to(r.device) / r - b)
        del self.a_quantizer.scale, self.a_quantizer.zero_point
        self.a_quantizer.channel_wise = False
        self.a_quantizer.scale = nn.Parameter(target_scale)
        self.a_quantizer.zero_point = nn.Parameter(target_zero_point)
        AsymmetricallyBatchingQuantLinear.hyperparameter_searching(self)


class PostGeluTwinUniformBatchingQuantLinear(AsymmetricallyBatchingQuantLinear):
    """reference: quant_layers/linear.py:624-721 (PTQ4ViT twin-uniform baseline, post_gelu_quantizer='ptq4vit'): a
    positive-range scale searched over 29 power-of-two multiples of the fixed negative-range scale."""

    def __init__(self, in_features: int, out_features: int, bias: bool = True, mode="raw", w_bit=8, a_bit=8,
                 calib_batch_size=None, search_round=1, eq_n=100, n_V=1, fpcs=False, steps=4):
        super().__init__(in_features, out_features, bias=bias, mode=mode, w_bit=w_bit, a_bit=a_bit,
                         calib_batch_size=calib_batch_size, search_round=search_round, eq_n=eq_n, n_V=n_V, fpcs=fpcs,
                         steps=steps)
        self.a_quantizer = TwinUniformQuantizer(n_bits=a_bit, symmetric=False, channel_wise=False)
        self.a_quantizer.scale = nn.Parameter(torch.zeros((2, 1)))

    def _initialize_activation_scale(self):
        """reference linear.py:647-662: positive scale from the largest |x| (max over the 32-sample batches = global
        max; all-reduced under data parallelism), negative scale = |min GELU| / n_levels"""
        nl = self.a_quantizer.n_levels
        dev = self.weight.device
        amax = adist.all_reduce_max(self._ctx.x2d.abs().max().view(1))
        pos = (amax / (nl - 0.5)).view(1)
        neg = torch.tensor(GELU_MIN / nl, device=dev).view(1)
        assign(self.a_quantizer.scale, torch.stack([pos, neg]))
        self.a_quantizer.inited = True

    def _search_best_a_scale(self, input_scale_candidates):
        """reference linear.py:664-696: only the first shape[-1] - 1 candidates are scored (:665-666) and the winner is
        taken with argmax (first maximum), not topk"""
        n = input_scale_candidates.shape[-1] - 1
        sims = sweep.linear_err_a_twin(self._ctx, self._weight3(), self.bias, self.w_quantizer,
                                       self.a_quantizer.scale[1].detach(), input_scale_candidates[:, :n].contiguous(),
                                       self.a_quantizer.n_levels)
        best = sims.argmax(dim=0, keepdim=True).reshape(1, -1)
        new_pos = torch.gather(input_scale_candidates, dim=-1, index=best).squeeze(-1)
        assign(self.a_quantizer.scale, torch.stack([new_pos, self.a_quantizer.scale[1].detach().clone()]))
        return best.squeeze(0)

    def hyperparameter_searching(self):
        """reference linear.py:698-721"""
        cls = AsymmetricallyBatchingQuantLinear
        self._initialize_calib_parameters()
        self._initialize_activation_scale()
        if self.fpcs:
            self.weight_fpcs(steps=self.steps, search_strategy=cls._search_best_w_scale_self)
        else:
            self._search_best_w_scale_self(*self.calculate_percentile_weight_candidates())
        # in PTQ4ViT, delta_r2 = delta_r1 * 2^m
        cands = (torch.tensor([(2 ** i) for i in range(-5, 25)]).to(self.weight.device).view(1, -1)
                 * self.a_quantizer.scale[1].detach().unsqueeze(-1))
        for _ in range(self.search_round):
            self._search_best_a_scale(cands)
            if self.fpcs:
                self.weight_fpcs(steps=self.steps, search_strategy=cls._search_best_w_scale)
            else:
                self._search_best_w_scale(*self.calculate_percentile_weight_candidates())
        self._finish()
        return None


class PostGeluLogBasedBatchingQuantLinear(AsymmetricallyBatchingQuantLinear):
    """reference: quant_layers/linear.py:724-1006 (fc2): shifted AdaLog activation quantizer, joint scale x base FPCS"""

    def __init__(self, in_features: int, out_features: int, bias: bool = True, mode="raw", w_bit=8, a_bit=8,
                 calib_batch_size=None, search_round=1, eq_n=100, n_V=1, quantizer='adalog', fpcs=False, steps=4):
        super().__init__(in_features, out_features, bias=bias, mode=mode, w_bit=w_bit, a_bit=a_bit,
                         calib_batch_size=calib_batch_size, search_round=search_round, eq_n=eq_n, n_V=n_V, fpcs=fpcs,
                         steps=steps)
        del self.a_quantizer
        self.a_quantizer = ShiftAdaLogQuantizer(n_bits=a_bit, symmetric=False, channel_wise=False)
        self.a_quantizer.scale = nn.Parameter(torch.zeros((1)))
        assign(self.a_quantizer.shift, torch.tensor(GELU_MIN))
        # search LUT (reference linear.py:750-752), kept for API parity; the kernels use its integer numerators
        self.table = torch.tensor([2 ** (-j / self.a_quantizer.r) for j in range(120)])
        self.table_scale = 1. / (4 * self.a_quantizer.n_levels - 2)
        self.table = torch.round(self.table / self.table_scale) * self.table_scale
        tmp_cls = {'log2': ShiftLog2Quantizer, 'logsqrt2': ShiftLogSqrt2Quantizer}.get(quantizer)
        if tmp_cls is not None:
            self.tmp_quantizer = tmp_cls(n_bits=a_bit, symmetric=False, channel_wise=False)
            self.tmp_quantizer.scale = nn.Parameter(torch.zeros((1)))
            assign(self.tmp_quantizer.shift, torch.tensor(GELU_MIN))

    @staticmethod
    def positive_percentile(tensor, q, dim=0):
        """reference linear.py:763-798: rank ceil(count*q)-1 among the positive entries (full sort; the exact
        radix-select replacement is SURVEY.md section 8f rank 2)"""
        positive = torch.where(tensor > 0, tensor, torch.full((), float('nan'), device=tensor.device))
        ordered, _ = positive.sort(dim=dim)
        counts = (~torch.isnan(ordered)).sum(dim=dim, keepdim=True).float()
        q = q.reshape(*([q.numel()] + [1] * tensor.ndim))
        ranks = ((counts * q).ceil().long() - 1).clamp(min=0)
        wide = ordered.unsqueeze(0).expand(q.shape[0], *ordered.shape)
        result = torch.gather(wide, dim + 1, ranks).squeeze(dim + 1)
        result.masked_fill_(torch.isnan(result), 0)
        return result

    @staticmethod
    def _positive_percentile_dist(x_local, q):
        """positive_percentile of the concatenation of all ranks' shards (1-D), without gathering them: global count of
        positive entries, then the exact element of rank ceil(count*q)-1 among them (utils/dist.py kth_values)."""
        pos = torch.where(x_local > 0, x_local, torch.full_like(x_local, float('inf')))
        srt, _ = pos.sort()
        counts = adist.all_reduce_sum((x_local > 0).sum().to(torch.int64).view(1)).float()
        ranks = ((counts * q).ceil().long() - 1).clamp(min=0)
        vals = adist.kth_values(srt.view(1, -1), ranks.view(-1)).view(-1)
        return torch.where(torch.isinf(vals) | (counts <= 0), torch.zeros_like(vals), vals)

    @staticmethod
    def _positive_percentile_select(x_local, q):
        """positive_percentile (of the concatenation of all ranks' shards under data parallelism) by exact radix
        selection instead of a full sort (csrc/select_kernels.cu): count the positive entries, then the element of rank
        ceil(count*q)-1 among them; entries <= 0 are keyed as +inf inside the kernel."""
        from .. import ops
        counts = adist.all_reduce_sum((x_local > 0).sum().to(torch.int64).view(1)).float()
        ranks = ((counts * q).ceil().long() - 1).clamp(min=0)
        vals = ops.select_kth(x_local.view(1, -1), ranks.view(-1), positive_only=True,
                              reduce_hist=adist.all_reduce_sum if adist.active() else None).view(-1)
        return torch.where(torch.isinf(vals) | (counts <= 0), torch.zeros_like(vals), vals)

    def calculate_percentile_activation_candidates(self, l=0.9, r=1.0):
        """reference linear.py:800-814"""
        # the calibration input does not change between search rounds: one selection per module
        cache = self._ctx.__dict__.setdefault('_pct_cache', {})
        if ('pos', l, r) not in cache:
            x = self._ctx.x2d.reshape(-1)
            q = _const.floats((l, r), x.device)
            if x.is_cuda and x.numel() >= _fpcs.SELECT_MIN_N:
                cache[('pos', l, r)] = self._positive_percentile_select(x, q)
            else:
                cache[('pos', l, r)] = (self._positive_percentile_dist(x, q) if adist.active()
                                        else self.positive_percentile(x, q))
        cand = cache[('pos', l, r)] + self.a_quantizer.shift.item()
        cand = cand.unsqueeze(0)
        ramp = _const.ramp(self.eq_n, cand.device).view(1, -1)
        return cand, cand[:, 0:1] + (cand[:, 1:] - cand[:, 0:1]) * ramp

    def _log_scored(self, cs, cq):
        P = cq.shape[-1]
        parts = []
        for p0, p1 in _fpcs.candidate_chunks(P):
            parts.append(sweep.linear_err_log(self._ctx, self._weight3(), self.bias, self.w_quantizer, self.a_quantizer,
                                              None if cs is None else cs[:, p0:p1], cq[:, p0:p1]))
        return parts[0] if len(parts) == 1 else torch.cat(parts, dim=-1)

    def _q_grid(self):
        return _const.int_range(10, 11 + self.eq_n, self.weight.device).view(1, -1)

    def _search_best_a_scale(self, input_scale_candidates, topk=1):
        """reference linear.py:816-854 (scale-only search at the current base; the fpcs=False path)"""
        P = input_scale_candidates.shape[-1]
        sims = self._log_scored(input_scale_candidates, self.a_quantizer.q.view(1, 1).expand(1, P))
        _, best = torch.topk(sims, k=topk, dim=-1)
        if topk == 1:
            assign(self.a_quantizer.scale, torch.gather(input_scale_candidates, dim=-1, index=best).squeeze(-1))
            self.a_quantizer.update_table()
        return best

    def _search_best_log_base(self, q_candidates=None, topk=1):
        """reference linear.py:856-896 (only the first eq_n of the 129 listed bases are scored)"""
        if q_candidates is None:
            q_candidates = self._q_grid()
        sims = self._log_scored(None, q_candidates[:, :self.eq_n])
        _, best = torch.topk(sims, k=topk, dim=-1)
        if topk == 1:
            assign(self.a_quantizer.q, torch.gather(q_candidates, dim=-1, index=best).view(*self.a_quantizer.q.shape))
            self.a_quantizer.update_table()
        return best

    def _search_best_scale_logbase(self, input_scale_candidates, q_candidates, topk=1):
        """reference linear.py:898-939"""
        sims = self._log_scored(input_scale_candidates, q_candidates)
        _, best = torch.topk(sims, k=topk, dim=-1)
        if topk == 1:
            assign(self.a_quantizer.scale, torch.gather(input_scale_candidates, dim=-1, index=best).squeeze(-1))
            assign(self.a_quantizer.q, torch.gather(q_candidates, dim=-1, index=best).view(*self.a_quantizer.q.shape))
            self.a_quantizer.update_table()
        return best

    def activation_fpcs(self, ud_candidates, base_num=8, scale_num=16, fpcs_width=32, steps=6):
        """reference linear.py:941-967: top-8 bases x 16 scales -> top-32 -> (steps-1) refinements of 4 points"""
        dev = self.weight.device
        q_all = self._q_grid()
        q_best = self._search_best_log_base(q_all, topk=base_num)
        ramp = _const.ramp(scale_num, dev).view(1, -1)
        cs = ud_candidates[:, 0:1] + (ud_candidates[:, 1:] - ud_candidates[:, 0:1]) * ramp
        delta = cs[:, 1:2] - cs[:, 0:1]
        cs = cs.repeat(1, base_num)
        cq = torch.gather(q_all, dim=-1, index=q_best).repeat_interleave(scale_num, dim=-1)
        _fpcs.refine(cs, cq, delta, lambda s, q, k: self._search_best_scale_logbase(s, q, topk=k), -1,
                     int(self.eq_n / fpcs_width), fpcs_width, steps)

    def hyperparameter_searching(self):
        """reference linear.py:969-997"""
        cls = AsymmetricallyBatchingQuantLinear
        self._initialize_calib_parameters()
        if self.fpcs:
            self.weight_fpcs(steps=self.steps, search_strategy=cls._search_best_w_scale_self)
        else:
            w_cs, w_cz = self.calculate_percentile_weight_candidates()
            self._search_best_w_scale_self(w_cs, w_cz)
        ud, a_cs = self.calculate_percentile_activation_candidates()
        assign(self.a_quantizer.scale, a_cs[:, -2])
        self.a_quantizer.inited = True
        for _ in range(self.search_round):
            if self.fpcs:
                self.activation_fpcs(ud_candidates=ud, steps=self.steps)
                self.weight_fpcs(steps=self.steps, search_strategy=cls._search_best_w_scale)
            else:
                self._search_best_log_base()
                self._search_best_a_scale(a_cs)
                w_cs, w_cz = self.calculate_percentile_weight_candidates()
                self._search_best_w_scale(w_cs, w_cz)
        if hasattr(self, 'tmp_quantizer'):
            assign(self.tmp_quantizer.scale, self.a_quantizer.scale.data)
            self.tmp_quantizer.inited = True
            self.a_quantizer = self.tmp_quantizer
            del self.tmp_quantizer
        self._finish()

    def reparam_bias(self):
        """reference linear.py:999-1006: fold -shift * W_hat^T into the bias"""
        if self.a_quantizer.bias_reparamed:
            return
        x_ = torch.full((1, self.in_features), -self.a_quantizer.shift.item(), device=self.weight.device)
        w_sim, bias_sim = self.quant_weight_bias()
        assign(self.bias, bias_sim + (x_ @ w_sim.transpose(0, 1)).squeeze())
        assign(self.a_quantizer.bias_reparamed, torch.tensor(True))
