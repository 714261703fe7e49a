"""CPU tier: this repo's drop-in `tokenflow_utils` / `util` modules against the UNMODIFIED reference drivers
(run_tokenflow_pnp.py and run_tokenflow_sdedit.py, class `TokenFlow`).  oracle/gen_golden.py ran the drivers'
own `init_method` and `batched_denoise_step` on the drop-in hooks and stored in tests/golden/driver_protocol.json
the names they import from the drop-ins and every call they make into the hooks, the UNet and the scheduler
(oracle/protocol.py); their result equalled the golden produced by the reference hooks.  Here
`tokenflow_b200/editor.py` must export what the drivers import, make the same calls in the same order on the
same values, and reach the same result, which shows both that the hooks are a drop-in under the reference's own
caller and that the editor mirrors that caller.  The oracle ops stand in for the CUDA kernels (no GPU here)."""
import json
import os

import pytest
import torch

from oracle import protocol
from oracle.oracle_ops import OracleOps
from tokenflow_b200 import sd_unet
from tokenflow_b200 import tokenflow_utils as tfu
from tokenflow_b200.editor import TokenFlowEditor, synthetic_inputs, write_latents_dir
from tokenflow_b200.scheduler import DDIMScheduler


@pytest.mark.parametrize("mode,driver,golden", [("pnp", "run_tokenflow_pnp.py", "unet_c1_pnp.pt"),
                                                ("sdedit", "run_tokenflow_sdedit.py", "unet_c1_sdedit.pt")])
def test_unmodified_reference_driver_on_dropin_hooks(mode, driver, golden, golden_dir, tmp_path):
    c = torch.load(os.path.join(golden_dir, golden), weights_only=False)
    with open(os.path.join(golden_dir, "driver_protocol.json")) as f:
        want = json.load(f)[driver]
    import tokenflow_utils as dropin_tf                          # top-level drop-in modules of this repo
    import util as dropin_util
    for name in want["imports"]["tokenflow_utils"]:
        assert hasattr(dropin_tf, name), name
    for name in want["imports"]["util"]:
        assert callable(getattr(dropin_util, name, None)), name
    for name in protocol.HOOKS:                                  # `from tokenflow_utils import *` binds OUR hooks
        assert getattr(dropin_tf, name) is getattr(tfu, name), name

    cfg = dict(c["config"])
    assert cfg["mode"] == mode
    unet = sd_unet.build_unet("tiny", seed=c["seed"])
    x, text, pnp, src = synthetic_inputs(cfg["n_frames"], c["latent"], unet.config.cross_attention_dim,
                                         cfg["n_timesteps"], seed=c["seed"], ctx_len=c["ctx_len"])
    cfg["latents_path"] = write_latents_dir(str(tmp_path), src)   # the drivers read source latents from disk
    rec = protocol.Recorder()
    tfu._install_ops_for_testing(OracleOps())
    ed = TokenFlowEditor(unet, rec.watch_scheduler(DDIMScheduler()), rec.hooks(tfu), cfg, text, pnp)
    rec.watch_unet(unet)
    ed.init_method()
    assert [int(t) for t in ed.scheduler.timesteps] == c["timesteps"]
    torch.manual_seed(c["seed"])
    steps = []
    out = ed.sample_loop(x, on_step=lambda i, t, z: steps.append(z.clone()))
    protocol.assert_same(rec.events, want["events"])
    assert len(steps) == len(c["steps"])
    for i, (got, ref) in enumerate(zip(steps, c["steps"])):
        assert torch.allclose(got, ref, atol=2e-4, rtol=1e-4), f"step {i}"
    assert torch.allclose(out, c["out"], atol=2e-4, rtol=1e-4)
