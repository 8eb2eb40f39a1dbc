"""Calibration driver with the reference's API (utils/calibrator.py): QuantCalibrator(model, loader).batching_quant_calib().

Same protocol per module -- capture raw input/output of the still-FP32 model over the calibration set, run
hyperparameter_searching(), reparam() where a preceding LayerNorm is attached, finally flip every module to
'quant_forward' -- but the captured tensors stay in HBM (no .cpu() round trip per batch, reference :14-28) where the
device sweeps consume them directly.  Under torch.distributed each rank captures its own shard of the loader.
"""
import time

import torch

from ..quant_layers import MinMaxQuantConv2d, MinMaxQuantLinear, MinMaxQuantMatMul
from . import models as _zoo

try:
    from tqdm import tqdm
except Exception:  # noqa: BLE001
    tqdm = None


class QuantCalibrator:
    def __init__(self, model, calib_loader):
        self.model = model
        self.calib_loader = calib_loader
        self.progress = True
        # timing (set by the caller): synchronise around capture / search of every module and keep the seconds in
        # self.timings[name] = (capture_s, search_s) -- for profiling only (adds two device syncs per module)
        self.timing = False
        self.timings = {}
        # Block-resume capture (SURVEY.md section 8f rank 1): the reference re-runs the WHOLE model over the
        # calibration set for every module (74 full forwards for a ViT).  A module inside a transformer block only
        # needs that block re-run on the block's own input, which cannot change while the block is being calibrated
        # (reparam rewrites the block's LayerNorm/linear, i.e. what comes after the input).  So the input of each
        # block is captured once with one full forward and the block alone is replayed per module: same kernels on
        # the same tensors, hence bit-identical captures, at 1/4 of the forward work.
        self.block_types = (_zoo.Block, _zoo.SwinTransformerBlock)
        self._cached_block = None
        self._cached_inputs = None

    # hooks keep device tensors (detached), reference :14-28
    def single_input_forward_hook(self, module, inp, outp):
        if module.tmp_input is None:
            module.tmp_input = []
        module.tmp_input.append(inp[0].detach())

    def double_input_forward_hook(self, module, inp, outp):
        if module.tmp_input is None:
            module.tmp_input = [[], []]
        module.tmp_input[0].append(inp[0].detach())
        module.tmp_input[1].append(inp[1].detach())

    def outp_forward_hook(self, module, inp, outp):
        if module.tmp_out is None:
            module.tmp_out = []
        module.tmp_out.append(outp.detach())

    def _tick(self):
        if not self.timing:
            return 0.0
        torch.cuda.synchronize()
        return time.perf_counter()

    def _pending(self):
        return [(n, m) for n, m in self.model.named_modules() if hasattr(m, 'calibrated') and not m.calibrated]

    def _enclosing_block(self, name):
        """the innermost ancestor of `name` that is a replayable transformer block, or None"""
        parts = name.split('.')
        for cut in range(len(parts) - 1, 0, -1):
            anc = self._by_name.get('.'.join(parts[:cut]))
            if isinstance(anc, self.block_types):
                return anc
        return None

    def _is_successor(self, prev, block):
        """True when `block` directly follows `prev` inside the same nn.Sequential"""
        if prev is None:
            return False
        pn, bn = self._name_of.get(prev), self._name_of.get(block)
        if pn is None or bn is None:
            return False
        pp, _, pi = pn.rpartition('.')
        bp, _, bi = bn.rpartition('.')
        return (pp == bp and pi.isdigit() and bi.isdigit() and int(bi) == int(pi) + 1
                and isinstance(self._by_name.get(pp), torch.nn.Sequential))

    def _run_forwards(self, name, device):
        block = self._enclosing_block(name)
        with torch.no_grad():
            if block is None:
                self._cached_block = self._cached_inputs = None
                for inp, _ in self.calib_loader:
                    self.model(inp.to(device))
                return
            if block is not self._cached_block:
                if self._is_successor(self._cached_block, block):
                    # consecutive children of one nn.Sequential: the next block's input is this block's output under
                    # the (now final) weights -- exactly what the full forward would recompute
                    self._cached_inputs = [self._cached_block(x).detach() for x in self._cached_inputs]
                    self._cached_block = block
                else:
                    grabbed = []
                    h = block.register_forward_pre_hook(lambda m, args: grabbed.append(args[0].detach()))
                    for inp, _ in self.calib_loader:      # this pass also serves the first module of the block
                        self.model(inp.to(device))
                    h.remove()
                    self._cached_block, self._cached_inputs = block, grabbed
                    return
            for x in self._cached_inputs:
                block(x)

    def _capture(self, name, module, device):
        hooks = [module.register_forward_hook(self.outp_forward_hook)]
        if isinstance(module, (MinMaxQuantLinear, MinMaxQuantConv2d)):
            hooks.append(module.register_forward_hook(self.single_input_forward_hook))
        if isinstance(module, MinMaxQuantMatMul):
            hooks.append(module.register_forward_hook(self.double_input_forward_hook))
        self._run_forwards(name, device)
        module.raw_out = torch.cat(module.tmp_out, dim=0)
        if isinstance(module, MinMaxQuantMatMul):
            module.raw_input = [torch.cat(t, dim=0) for t in module.tmp_input]
        else:
            module.raw_input = torch.cat(module.tmp_input, dim=0)
        for h in hooks:
            h.remove()
        module.tmp_input = module.tmp_out = None

    def batching_quant_calib(self):
        """reference calibrator.py:30-67"""
        device = next(self.model.parameters()).device
        self._by_name = dict(self.model.named_modules())
        self._name_of = {m: n for n, m in self._by_name.items() if isinstance(m, self.block_types)}
        pending = self._pending()
        bar = tqdm(total=len(pending)) if (tqdm is not None and self.progress) else None
        for name, module in self.model.named_modules():
            if not hasattr(module, 'calibrated') or module.calibrated:
                continue
            if bar is not None:
                bar.set_description(f"calibrating {name}")
            t0 = self._tick()
            self._capture(name, module, device)
            t1 = self._tick()
            with torch.no_grad():
                module.hyperparameter_searching()
                if hasattr(module, 'prev_layer') and module.prev_layer is not None:
                    if bar is not None:
                        bar.set_description(f"reparaming {name}")
                    module.reparam()
            if self.timing:
                self.timings[name] = (t1 - t0, self._tick() - t1)
            if bar is not None:
                bar.update()
        if bar is not None:
            bar.close()
        self._cached_block = self._cached_inputs = None
        for _, module in self.model.named_modules():
            if hasattr(module, 'mode'):
                module.mode = "quant_forward"
