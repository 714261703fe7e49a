"""CPU tier: this package's hook layer (tokenflow_b200.tokenflow_utils) with the oracle ops installed,
against golden vectors produced by the unmodified reference hooks — i.e. the host logic / plumbing
of the drop-in, with no GPU compute.  BASELINE config C1 in miniature."""
import os

import pytest
import torch
import torch.nn as nn

from oracle import golden
from oracle.oracle_ops import OracleOps
from tokenflow_b200 import sd_unet
from tokenflow_b200 import tokenflow_utils as tfu
from tokenflow_b200.editor import TokenFlowEditor, synthetic_inputs
from tokenflow_b200.scheduler import DDIMScheduler


def _load(golden_dir, name):
    return torch.load(os.path.join(golden_dir, name), weights_only=False)


class _OneBlockUNet(nn.Module):
    def __init__(self, block):
        super().__init__()
        self.block = block
        site = nn.Module()
        site.transformer_blocks = nn.ModuleList([block])
        ups = []
        for _ in range(4):
            u = nn.Module()
            u.attentions = nn.ModuleList([site, site, site])
            ups.append(u)
        self.up_blocks = nn.ModuleList(ups)


class _Wrap(nn.Module):
    def __init__(self, unet):
        super().__init__()
        self.unet = unet


def test_public_surface_matches_reference_names():
    for name in ("register_pivotal", "register_batch_idx", "register_time", "load_source_latents_t",
                 "register_conv_injection", "register_extended_attention_pnp", "register_extended_attention",
                 "make_tokenflow_attention_block", "set_tokenflow", "isinstance_str", "batch_cosine_sim"):
        assert callable(getattr(tfu, name)), name
    import tokenflow_utils as top          # the drop-in module name the reference drivers import
    import util as top_util
    assert top.set_tokenflow is tfu.set_tokenflow
    assert callable(top_util.seed_everything) and callable(top_util.save_video)


def test_no_fallback_without_gpu():
    """The product op path must fail loudly, not fall back, when there is no CUDA device."""
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from tokenflow_b200.ops import TokenflowB200Error
    tfu._install_ops_for_testing(None)
    with pytest.raises(TokenflowB200Error):
        tfu._ops()


def test_attention_closure_matches_reference(golden_dir):
    tfu._install_ops_for_testing(OracleOps())
    for c in golden.load_ext_attn(golden_dir):
        block = sd_unet.BasicTransformerBlock(c["dim"], c["heads"], c["dim"] // c["heads"], 32).eval()
        block.attn1.load_state_dict(c["state_dict"])
        model = _Wrap(_OneBlockUNet(block))
        if c["pnp"]:
            tfu.register_extended_attention_pnp(model, torch.tensor(c["schedule"]))
            block.attn1.t = c["t"]
        else:
            tfu.register_extended_attention(model)
        with torch.no_grad():
            out = block.attn1(c["x"])
        assert torch.allclose(out, c["out"], atol=2e-6, rtol=1e-5), c["name"]


def test_tokenflow_block_matches_reference(golden_dir):
    tfu._install_ops_for_testing(OracleOps())
    c = golden.load_block_passes(golden_dir)
    block = sd_unet.BasicTransformerBlock(c["dim"], c["heads"], c["dim"] // c["heads"], c["ctx"]).eval()
    block.load_state_dict(c["state_dict"])
    model = _Wrap(_OneBlockUNet(block))
    tfu.register_extended_attention(model)
    tfu.set_tokenflow(model.unet)
    assert tfu.isinstance_str(block, "TokenFlowBlock") and tfu.isinstance_str(block, "BasicTransformerBlock")
    with torch.no_grad():
        tfu.register_pivotal(model, True)
        out = block(c["pivotal"]["hidden"], encoder_hidden_states=c["pivotal"]["ctx"])
        assert torch.allclose(out, c["pivotal"]["out"], atol=1e-5, rtol=1e-5)
        assert torch.allclose(block.pivot_hidden_states, c["pivotal"]["pivot_hidden_states"], atol=1e-6)
        assert torch.allclose(block.kf_attn_output, c["pivotal"]["kf_attn_output"], atol=2e-6, rtol=1e-5)
        tfu.register_pivotal(model, False)
        for fr in c["frames"]:
            tfu.register_batch_idx(model, fr["batch_idx"])
            out = block(fr["hidden"], encoder_hidden_states=fr["ctx"])
            idx_a, idx_b = block._tf_nn_idx
            assert torch.equal(idx_a.reshape(-1).long(), fr["idx1"])
            if fr["idx2"] is not None:
                assert torch.equal(idx_b.reshape(-1).long(), fr["idx2"])
            assert torch.allclose(out, fr["out"], atol=1e-5, rtol=1e-5)


def test_frame_table_equals_batch_idx(golden_dir):
    """register_frame_table (per-frame keyframes/weights) reproduces register_batch_idx."""
    tfu._install_ops_for_testing(OracleOps())
    c = golden.load_block_passes(golden_dir)
    block = sd_unet.BasicTransformerBlock(c["dim"], c["heads"], c["dim"] // c["heads"], c["ctx"]).eval()
    block.load_state_dict(c["state_dict"])
    model = _Wrap(_OneBlockUNet(block))
    tfu.register_extended_attention(model)
    tfu.set_tokenflow(model.unet)
    from tokenflow_b200.ops import blend_weights
    with torch.no_grad():
        tfu.register_pivotal(model, True)
        block(c["pivotal"]["hidden"], encoder_hidden_states=c["pivotal"]["ctx"])
        tfu.register_pivotal(model, False)
        fr = c["frames"][2]
        B = c["B"]
        tfu.register_frame_table(model, [2] * B, [1] * B, blend_weights(B))
        out = block(fr["hidden"], encoder_hidden_states=fr["ctx"])
        assert torch.allclose(out, fr["out"], atol=1e-5, rtol=1e-5)


@pytest.mark.parametrize("name", ["unet_c1_pnp.pt", "unet_c1_sdedit.pt"])
def test_unet_edit_matches_reference(golden_dir, name):
    """Full SD-topology UNet (toy width), 4 frames, B=2: PnP (2 steps) and SDEdit (truncated
    schedule) loops through this package's hooks == through the reference's hooks."""
    tfu._install_ops_for_testing(OracleOps())
    c = _load(golden_dir, name)
    cfg = c["config"]
    unet = sd_unet.build_unet("tiny", seed=c["seed"])
    x, text, pnp, src = synthetic_inputs(cfg["n_frames"], c["latent"], unet.config.cross_attention_dim,
                                         cfg["n_timesteps"], seed=c["seed"], ctx_len=c["ctx_len"])
    assert torch.equal(x, c["x0"])
    ed = TokenFlowEditor(unet, DDIMScheduler(), tfu, cfg, text, pnp, source_latents=lambda t: src[t])
    ed.init_method()
    assert [int(t) for t in ed.scheduler.timesteps] == c["timesteps"]
    torch.manual_seed(c["seed"])
    steps = []
    out = ed.sample_loop(x, on_step=lambda i, t, z: steps.append(z.clone()))
    assert ed.keyframe_log == c["keyframes"]
    for got, want in zip(steps, c["steps"]):
        assert torch.allclose(got, want, atol=2e-4, rtol=1e-4)
    assert torch.allclose(out, c["out"], atol=2e-4, rtol=1e-4)


def test_registration_finds_sd_topology():
    unet = sd_unet.build_unet("tiny")
    model = _Wrap(unet)
    blocks = tfu._transformer_blocks(model)
    assert len(blocks) == 16                       # 5 per resolution x 3 + mid (SURVEY.md §8)
    tfu.register_extended_attention_pnp(model, torch.tensor([981, 961]))
    injected = [b for b in blocks if len(b.attn1.injection_schedule) > 0]
    assert len(injected) == 8                      # decoder blocks 4-11 (reference :208-214)
    tfu.register_time(model, 981)
    assert all(b.attn1.t == 981 and b.attn2.t == 981 for b in blocks)
    assert unet.up_blocks[1].resnets[1].t == 981
    tfu.register_pivotal(model, True)
    tfu.register_batch_idx(model, 3)
    assert all(b.pivotal_pass is True and b.batch_idx == 3 for b in blocks)


def test_schedule_membership_matches_reference_semantics():
    m = nn.Module()
    m.injection_schedule = torch.tensor([981, 961])
    m.t = 961
    assert tfu._in_schedule(m)
    m.t = 1
    assert not tfu._in_schedule(m)
    m.t = 1000                                     # reference: `or self.t == 1000`
    assert tfu._in_schedule(m)
    m.injection_schedule = []
    m.t = 981
    assert not tfu._in_schedule(m)
    m.injection_schedule = None
    m.t = 1000
    assert not tfu._in_schedule(m)


def test_load_source_latents(tmp_path):
    from tokenflow_b200.editor import write_latents_dir
    src = {981: torch.randn(4, 4, 8, 8), 961: torch.randn(4, 4, 8, 8)}
    lat = write_latents_dir(str(tmp_path), src)
    assert torch.equal(tfu.load_source_latents_t(981, lat), src[981])
    assert torch.equal(tfu.load_source_latents_t(torch.tensor(961), lat), src[961])
    with pytest.raises(AssertionError):
        tfu.load_source_latents_t(1, lat)


def test_frames_per_pass_equals_reference_schedule(golden_dir):
    """All frames in one frame pass (per-frame keyframe table) == the reference's per-batch passes."""
    tfu._install_ops_for_testing(OracleOps())
    c = _load(golden_dir, "unet_c1_pnp.pt")
    cfg = dict(c["config"], frames_per_pass=c["config"]["n_frames"])
    unet = sd_unet.build_unet("tiny", seed=c["seed"])
    x, text, pnp, src = synthetic_inputs(cfg["n_frames"], c["latent"], unet.config.cross_attention_dim,
                                         cfg["n_timesteps"], seed=c["seed"], ctx_len=c["ctx_len"])
    ed = TokenFlowEditor(unet, DDIMScheduler(), tfu, cfg, text, pnp, source_latents=lambda t: src[t])
    ed.init_method()
    torch.manual_seed(c["seed"])
    out = ed.sample_loop(x)
    assert ed.keyframe_log == c["keyframes"]
    assert torch.allclose(out, c["out"], atol=2e-4, rtol=1e-4)


@pytest.mark.parametrize("name", ["unet_c1_pnp.pt", "unet_c1_sdedit.pt"])
def test_fused_pass_equals_reference_schedule(golden_dir, name):
    """ONE UNet call per step ([pivotal samples | all frames]) == the reference's pivotal pass + N/B frame
    passes, including the PnP conv-feature injection on both parts of the batch."""
    tfu._install_ops_for_testing(OracleOps())
    c = _load(golden_dir, name)
    cfg = dict(c["config"], fused_pass=True)
    unet = sd_unet.build_unet("tiny", seed=c["seed"])
    x, text, pnp, src = synthetic_inputs(cfg["n_frames"], c["latent"], unet.config.cross_attention_dim,
                                         cfg["n_timesteps"], seed=c["seed"], ctx_len=c["ctx_len"])
    ed = TokenFlowEditor(unet, DDIMScheduler(), tfu, cfg, text, pnp, source_latents=lambda t: src[t])
    ed.init_method()
    torch.manual_seed(c["seed"])
    steps = []
    out = ed.sample_loop(x, on_step=lambda i, t, z: steps.append(z.clone()))
    assert ed.keyframe_log == c["keyframes"]
    for got, want in zip(steps, c["steps"]):
        assert torch.allclose(got, want, atol=2e-4, rtol=1e-4)
    assert torch.allclose(out, c["out"], atol=2e-4, rtol=1e-4)
    assert all(getattr(b, "_tf_fused", 0) == 0 for b in tfu._transformer_blocks(ed))   # mode restored
