"""ORACLE (test infrastructure) — the calls a TokenFlow driver makes into the hook module, the UNet and
the scheduler, as plain values.

The reference drivers (run_tokenflow_pnp.py / run_tokenflow_sdedit.py, class TokenFlow) import the hook
functions from `tokenflow_utils` and call them, the UNet and the scheduler in a fixed order.  `Recorder`
logs every such call: a hook's name with its scalar arguments (timesteps, flags, batch indices; modules
and paths are left out), and for each UNet call and scheduler step the timestep, the tensor shapes and
a position-weighted checksum of the tensors, so that the same values in other places do not pass.
oracle/gen_golden.py records the unmodified reference driver running on this repo's drop-in hooks into
tests/golden/driver_protocol.json; the tests run `TokenFlowEditor` under a recorder and compare.
"""
from __future__ import annotations

import functools

import numpy as np
import torch

HOOKS = ("register_extended_attention_pnp", "register_conv_injection", "register_extended_attention",
         "set_tokenflow", "load_source_latents_t", "register_time", "register_pivotal", "register_batch_idx")


def checksum(t: torch.Tensor):
    """[sum(v*w), sum(|v|*w)] in float64 with fixed weights w in [1, 2) that vary with the position."""
    v = t.detach().reshape(-1).double().cpu().numpy()
    i = np.arange(v.size, dtype=np.int64)
    w = 1.0 + ((i * 7919) % 1009) / 1009.0
    return [float(v @ w), float(np.abs(v) @ w)]


def _plain(a):
    if isinstance(a, torch.Tensor):
        return int(a) if a.dim() == 0 else [int(v) for v in a.reshape(-1).tolist()]
    if isinstance(a, (bool, int)):
        return a
    if isinstance(a, (list, tuple)):
        return [_plain(v) for v in a]
    return None


class Recorder:
    def __init__(self):
        self.events = []

    def wrap(self, name, fn):
        @functools.wraps(fn)
        def call(*args, **kwargs):
            self.events.append([name] + [p for p in map(_plain, args) if p is not None])
            return fn(*args, **kwargs)
        return call

    def patch_globals(self, namespace: dict):
        """Record the hook functions a driver module calls through its globals."""
        for name in HOOKS:
            if name in namespace:
                namespace[name] = self.wrap(name, namespace[name])

    def hooks(self, module):
        """A stand-in for the hook module that records the calls to HOOKS and passes everything else on."""
        rec = self

        class _Hooks:
            def __getattr__(self, name):
                fn = getattr(module, name)
                return rec.wrap(name, fn) if name in HOOKS else fn
        return _Hooks()

    def watch_unet(self, unet: torch.nn.Module):
        def pre(_mod, args, kwargs):
            sample, t = args[0], args[1]
            ctx = kwargs["encoder_hidden_states"]
            self.events.append(["unet", int(t), list(sample.shape), checksum(sample), list(ctx.shape), checksum(ctx)])
        return unet.register_forward_pre_hook(pre, with_kwargs=True)

    def watch_scheduler(self, scheduler):
        step = scheduler.step

        def recorded(model_output, t, sample, *a, **k):
            self.events.append(["scheduler.step", int(t), list(sample.shape), checksum(model_output), checksum(sample)])
            return step(model_output, t, sample, *a, **k)
        scheduler.step = recorded
        return scheduler


def assert_same(got, want, rtol=1e-4):
    """Same calls in the same order with the same scalar arguments and shapes; checksums within `rtol` of
    the weighted absolute sum (the UNet numerics may differ in the last bits between machines)."""
    assert len(got) == len(want), (len(got), len(want))
    for n, (g, w) in enumerate(zip(got, want)):
        assert len(g) == len(w) and g[0] == w[0], (n, g[:2], w[:2])
        for a, b in zip(g[1:], w[1:]):
            if isinstance(b, list) and len(b) == 2 and all(isinstance(x, float) for x in b):
                assert abs(a[0] - b[0]) <= rtol * b[1] + 1e-9 and abs(a[1] - b[1]) <= rtol * b[1] + 1e-9, (n, g[0], a, b)
            else:
                assert a == b, (n, g[0], a, b)
