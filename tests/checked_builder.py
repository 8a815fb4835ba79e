"""Test-only Builder that verifies EVERY launch of a lowered network in situ: after each op runs
on the GPU, the same op is recomputed with torch fp32 ops (bf16 storage, tests/cpu_builder.
Bf16Builder) FROM THE KERNEL'S OWN INPUT BUFFERS and compared with the kernel's output.  Feeding
each reference the actual inputs removes the error amplification of the (ill-conditioned)
synthetic networks, so the tolerance is just bf16 output rounding + accumulation order."""
from __future__ import annotations

import torch

from oct_segmentation_b200.engine.builder import Builder
from tests.cpu_builder import Bf16Builder, _nchw


def _rel(a, b):
    return ((a.float() - b.float()).norm() / b.float().norm().clamp_min(1e-6)).item()


class CheckedBuilder(Builder):
    def __init__(self, device, N):
        super().__init__(device, N, reuse=False)     # the references re-read inputs that would otherwise be dead
        self.ref = Bf16Builder(N, device)
        self.checks = []
        self._pools = {}        # '<name>.se' -> SE partial-sum buffer [N][slots][C] of that block
        self._pool_snap = {}    # '<name>' -> its contents just before the SE launches

    def stem(self, x, in_dtype, w, b, **k):
        out = super().stem(x, in_dtype, w, b, **k)
        self.checks.append((k['name'], lambda: _nchw(self.ref.stem(x, in_dtype, w, b, **k)), lambda: _nchw(out)))
        return out

    def maxpool(self, x, **k):
        out = super().maxpool(x, **k)
        self.checks.append((k['name'], lambda: _nchw(self.ref.maxpool(x, **k)), lambda: _nchw(out)))
        return out

    def conv(self, srcs, w, b, **k):
        out = super().conv(srcs, w, b, **k)
        if out is not None:
            self.checks.append((k['name'], lambda: _nchw(self.ref.conv(srcs, w, b, **k)), lambda: _nchw(out)))
        else:
            real = k['out_tensor']

            def ref_fn():
                kk = dict(k)
                kk['out_tensor'] = torch.zeros_like(real, dtype=torch.float32)
                kk['out_mode'] = 'f32_nchw'
                self.ref.conv(srcs, w, b, **kk)
                return kk['out_tensor']
            if k.get('out_mode') == 'u8_nchw':
                self.checks.append((k['name'] + '[mask]', lambda: (ref_fn() > 0).float(), lambda: real.float()))
            else:
                self.checks.append((k['name'], ref_fn, lambda: real))
        return out

    def dwconv(self, x, w, b, **k):
        out = super().dwconv(x, w, b, **k)
        pool = k['pool']

        def ref_fn():
            kk = dict(k)
            kk['pool'] = torch.zeros_like(pool)
            r = _nchw(self.ref.dwconv(x, w, b, **kk))
            self._last_pool_err = _rel(pool.sum(1), kk['pool'].sum(1))
            return r
        self.checks.append((k['name'], ref_fn, lambda: _nchw(out)))
        return out

    def se_project(self, x, pool, w1, b1, w2, b2, wp, bp, **k):
        out = super().se_project(x, pool, w1, b1, w2, b2, wp, bp, **k)
        self._pools[k['name'] + '.se'] = pool
        self.checks.append((k['name'],
                            lambda: _nchw(self.ref.se_project(x, self._pool_snap[k['name']], w1, b1, w2, b2, wp, bp, **k)),
                            lambda: _nchw(out)))
        return out

    @torch.no_grad()
    def run_checked(self):
        """Runs the op list one launch at a time; returns [(name, rel_l2)]."""
        self.finalize()
        checks = {}
        for name, r, g in self.checks:          # a split conv registers its inner launch, then the whole op: keep the latter
            checks[name.replace('[mask]', '')] = (name, r, g)
        errs = []
        for op_name, op in zip(self.op_names, self.ops):
            if op_name in self._pools:
                self._pool_snap[op_name[:-3]] = self._pools[op_name].clone()
            op()
            torch.cuda.synchronize()
            if op_name not in checks:               # helper launches (SE gate) are covered by their consumer
                continue
            name, ref_fn, got_fn = checks[op_name]
            want, got = ref_fn(), got_fn()
            assert torch.isfinite(got).all(), f'{name}: non-finite output'
            errs.append((name, _rel(got, want)))
        return errs
