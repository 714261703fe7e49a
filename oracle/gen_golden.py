"""ORACLE (test infrastructure) — generate tests/golden/ by running the UNMODIFIED reference hooks
(tokenflow_utils.py, imported through oracle/ref_shim.py) and drivers on seeded inputs.

Run where the reference tree exists:   TOKENFLOW_REFERENCE_DIR=<path> python -m oracle.gen_golden
The reference ships no golden vectors of its own (SURVEY.md §4); these files are the pin for the
oracle and for the CUDA path.  Everything is fp32 on CPU (the reference's CPU-runnable configuration,
BASELINE config C1), deterministic in the seeds below.  No file exceeds 1 MB (oracle/golden.py).
"""
from __future__ import annotations

import os
import sys

import torch
import torch.nn as nn

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if REPO not in sys.path:
    sys.path.insert(0, REPO)

from oracle import golden, protocol  # noqa: E402
from oracle.ref_shim import load_driver, load_reference  # noqa: E402
from tokenflow_b200 import sd_unet  # noqa: E402
from tokenflow_b200.editor import TokenFlowEditor, synthetic_inputs  # noqa: E402
from tokenflow_b200.scheduler import DDIMScheduler  # noqa: E402

GOLDEN_DIR = os.path.join(REPO, "tests", "golden")


class _Wrap(nn.Module):
    """`model` as the reference hooks see it: something with `.unet` whose module tree they walk."""

    def __init__(self, unet):
        super().__init__()
        self.unet = unet


class _OneBlockUNet(nn.Module):
    """Just enough `unet` for register_extended_attention*: one transformer block reachable through
    named_modules(); the hard-coded decoder sites are the same block."""

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


def attention_case(ref, name, n, S, dim, heads, pnp, t, schedule, seed):
    torch.manual_seed(seed)
    block = sd_unet.BasicTransformerBlock(dim, heads, dim // heads, cross_attention_dim=32).eval()
    model = _Wrap(_OneBlockUNet(block))
    if pnp:
        ref.register_extended_attention_pnp(model, schedule)
        block.attn1.t = t
    else:
        ref.register_extended_attention(model)
    x = torch.randn(3 * n, S, dim)
    with torch.no_grad():
        out = block.attn1(x)
        q, k, v = block.attn1.to_q(x), block.attn1.to_k(x), block.attn1.to_v(x)
    inject = bool(pnp and (t in schedule or t == 1000))
    return {"name": name, "n": n, "S": S, "dim": dim, "heads": heads, "pnp": pnp, "t": t,
            "schedule": list(schedule), "inject": inject, "seed": seed,
            "state_dict": {k_: v_.clone() for k_, v_ in block.attn1.state_dict().items()},
            "x": x, "q": q, "k": k, "v": v, "out": out}


def block_case(ref, ref_util, seed=7, K=3, B=4, S=40, dim=64, heads=4, ctx=32):
    """Pivotal pass over K keyframes, then frame passes for batches 0..K-1 (B frames each)."""
    torch.manual_seed(seed)
    block = sd_unet.BasicTransformerBlock(dim, heads, dim // heads, cross_attention_dim=ctx).eval()
    # non-trivial LayerNorm affine so norm1 is not the identity scaling
    for ln in (block.norm1, block.norm2, block.norm3):
        ln.weight.data.uniform_(0.5, 1.5)
        ln.bias.data.uniform_(-0.2, 0.2)
    state = {k_: v_.clone() for k_, v_ in block.state_dict().items()}
    model = _Wrap(_OneBlockUNet(block))
    ref.register_extended_attention(model)
    ref.set_tokenflow(model.unet)
    piv_h = torch.randn(3 * K, S, dim)
    piv_ctx = torch.randn(3 * K, 5, ctx)
    case = {"K": K, "B": B, "S": S, "dim": dim, "heads": heads, "ctx": ctx, "seed": seed, "state_dict": state,
            "pivotal": {"hidden": piv_h, "ctx": piv_ctx}, "frames": []}
    with torch.no_grad():
        ref.register_pivotal(model, True)
        case["pivotal"]["out"] = block(piv_h, encoder_hidden_states=piv_ctx)
        case["pivotal"]["pivot_hidden_states"] = block.pivot_hidden_states.clone()
        case["pivotal"]["kf_attn_output"] = block.kf_attn_output.clone()
        ref.register_pivotal(model, False)
        for i in range(K):
            # video-like queries: keyframe tokens + noise, so the NN field is not uniform noise
            base = piv_h[:K][i].unsqueeze(0).repeat(B, 1, 1)
            src = base[:, torch.randperm(S)] + 0.3 * torch.randn(B, S, dim)
            h = torch.cat([src, torch.randn(2 * B, S, dim)])
            c = torch.randn(3 * B, 5, ctx)
            ref.register_batch_idx(model, i)
            out = block(h, encoder_hidden_states=c)
            # the NN indices the reference computed inside (recomputed with its own helper)
            norm = block.norm1(h).view(3, B, S, dim)
            kfs = [i] + ([i - 1] if i > 0 else [])
            sim = ref_util.batch_cosine_sim(norm[0].reshape(-1, dim),
                                            block.pivot_hidden_states[0][kfs].reshape(-1, dim))
            if len(kfs) == 2:
                s1, s2 = sim.chunk(2, dim=1)
                idx1, idx2 = s1.argmax(-1), s2.argmax(-1)
            else:
                idx1, idx2 = sim.argmax(-1), None
            case["frames"].append({"batch_idx": i, "hidden": h, "ctx": c, "out": out, "idx1": idx1, "idx2": idx2})
    return case


def unet_case(ref, mode, seed=1, n_frames=4, batch_size=2, n_timesteps=2, latent=16):
    """BASELINE config C1 in miniature: SD topology at toy width, 4 frames, B=2, 2 DDIM steps."""
    unet = sd_unet.build_unet("tiny", seed=seed)
    cfg = {"n_frames": n_frames, "batch_size": batch_size, "n_timesteps": n_timesteps, "guidance_scale": 7.5,
           "mode": mode, "pnp_attn_t": 0.5, "pnp_f_t": 0.8, "start": 0.9}
    x, text, pnp, src = synthetic_inputs(n_frames, latent, unet.config.cross_attention_dim, n_timesteps, seed=seed,
                                         ctx_len=7)
    ed = TokenFlowEditor(unet, DDIMScheduler(), ref, cfg, text, pnp, source_latents=lambda t: src[t])
    ed.init_method()
    torch.manual_seed(seed)           # keyframe draws come from the global CPU generator
    steps = []
    out = ed.sample_loop(x, on_step=lambda i, t, z: steps.append(z.clone()))
    return {"mode": mode, "config": cfg, "seed": seed, "latent": latent, "ctx_len": 7,
            "timesteps": [int(t) for t in ed.scheduler.timesteps], "keyframes": ed.keyframe_log,
            "x0": x, "steps": steps, "out": out}


# the cases of the live comparisons in tests/test_reference_live.py: (seed, n, S, dim, heads, pnp, inject)
LIVE_ATTENTION = [(101, 2, 24, 32, 2, False, False), (102, 4, 20, 64, 4, True, True), (103, 4, 20, 64, 4, True, False),
                  (104, 13, 8, 32, 4, True, True)]


def live_cases(ref, ref_util):
    """The reference's attention output for small blocks (K=13 takes the reference's per-frame loop), and its
    cosine-similarity / isinstance_str helpers."""
    attn = {}
    for seed, n, S, dim, heads, pnp, inject in LIVE_ATTENTION:
        torch.manual_seed(seed)
        block = sd_unet.BasicTransformerBlock(dim, heads, dim // heads, 16).eval()
        model = _Wrap(_OneBlockUNet(block))
        if pnp:
            ref.register_extended_attention_pnp(model, [981] if inject else [])
            block.attn1.t = 981
        else:
            ref.register_extended_attention(model)
        x = torch.randn(3 * n, S, dim)
        with torch.no_grad():
            out = block.attn1(x)
        attn[seed] = {"n": n, "S": S, "dim": dim, "heads": heads, "inject": inject, "x": x,
                      "state_dict": {k_: v_.clone() for k_, v_ in block.attn1.state_dict().items()}, "out": out}
    torch.manual_seed(5)
    x, y = torch.randn(50, 24), torch.randn(30, 24)
    blk = sd_unet.BasicTransformerBlock(16, 2, 8, 8)
    names = ("BasicTransformerBlock", "Module", "Attention", "object")
    return {"attention": attn, "cosine_sim": {"x": x, "y": y, "out": ref_util.batch_cosine_sim(x, y)},
            "isinstance_str": {name: ref_util.isinstance_str(blk, name) for name in names}}


def driver_protocol(filename, c):
    """The unmodified reference driver's TokenFlow.init_method / batched_denoise_step on this repo's drop-in hooks
    (oracle ops), on the inputs of the unet_c1 golden `c`: the names it imports from the drop-in modules and the
    calls it makes (oracle/protocol.py).  Its __init__ (Stable Diffusion, VAE, CLIP, video files) is bypassed;
    the result must equal `c`, which the reference hooks produced through TokenFlowEditor."""
    import tempfile
    import warnings
    import tokenflow_utils as dropin_tf
    import util as dropin_util
    from oracle.oracle_ops import OracleOps
    from tokenflow_b200 import tokenflow_utils as tfu
    from tokenflow_b200.editor import write_latents_dir
    mod = load_driver(filename, DDIMScheduler)
    ns = vars(mod)
    with open(mod.__file__) as f:
        code = [compile(f.read(), mod.__file__, "exec")]
    used = set()
    while code:                                              # every name the driver's code refers to
        co = code.pop()
        used.update(co.co_names)
        code.extend(k for k in co.co_consts if hasattr(k, "co_names"))
    imports = {m.__name__: sorted(n for n in used if n in ns and ns[n] is getattr(m, n, None))
               for m in (dropin_tf, dropin_util)}
    assert ns["register_pivotal"] is tfu.register_pivotal
    rec = protocol.Recorder()
    rec.patch_globals(ns)
    cfg = c["config"]
    unet = sd_unet.build_unet("tiny", seed=c["seed"])
    x, text, pnp, src = synthetic_inputs(cfg["n_frames"], c["latent"], unet.config.cross_attention_dim,
                                         cfg["n_timesteps"], seed=c["seed"], ctx_len=c["ctx_len"])
    tfu._install_ops_for_testing(OracleOps())
    try:
        with tempfile.TemporaryDirectory() as tmp:
            ed = mod.TokenFlow.__new__(mod.TokenFlow)
            nn.Module.__init__(ed)
            ed.config = {k_: cfg[k_] for k_ in ("batch_size", "guidance_scale", "n_frames", "n_timesteps")}
            ed.device = "cpu"
            ed.sd_version = "1.5"
            ed.unet = unet
            ed.scheduler = rec.watch_scheduler(DDIMScheduler())
            ed.scheduler.set_timesteps(cfg["n_timesteps"], device="cpu")
            if cfg["mode"] == "sdedit":                          # run_tokenflow_sdedit.py:57
                ed.scheduler.timesteps = ed.scheduler.timesteps[int(1 - cfg["start"] * cfg["n_timesteps"]):]
            ed.latents_path = write_latents_dir(tmp, src)
            ed.text_embeds = text
            ed.pnp_guidance_embeds = pnp
            rec.watch_unet(unet)
            if cfg["mode"] == "pnp":                             # run_tokenflow_pnp.py:253-256
                ed.init_method(conv_injection_t=int(cfg["n_timesteps"] * cfg["pnp_f_t"]),
                               qk_injection_t=int(cfg["n_timesteps"] * cfg["pnp_attn_t"]))
            else:                                                # run_tokenflow_sdedit.py:191-193
                ed.init_method()
            assert [int(t) for t in ed.scheduler.timesteps] == c["timesteps"]
            torch.manual_seed(c["seed"])
            indices = torch.arange(cfg["n_frames"])
            with warnings.catch_warnings():
                warnings.simplefilter("ignore")                  # the driver's cuda autocast decorator on a CPU box
                for i, t in enumerate(ed.scheduler.timesteps):   # the body of sample_loop (:266-267), VAE decode omitted
                    x = ed.batched_denoise_step(x, t, indices)
                    assert torch.allclose(x, c["steps"][i], atol=2e-4, rtol=1e-4), f"step {i}"
    finally:
        tfu._install_ops_for_testing(None)
    return {"imports": imports, "events": rec.events}


def main():
    import json
    ref, ref_util = load_reference()
    os.makedirs(GOLDEN_DIR, exist_ok=True)
    attn = [
        attention_case(ref, "sdedit_n3", 3, 48, 64, 4, False, 0, [], seed=11),
        attention_case(ref, "pnp_n3_inject", 3, 48, 64, 4, True, 981, [981, 961], seed=12),
        attention_case(ref, "pnp_n3_noinject", 3, 48, 64, 4, True, 1, [981, 961], seed=13),
        attention_case(ref, "pnp_n3_t1000", 3, 24, 32, 2, True, 1000, [981], seed=14),
        attention_case(ref, "pnp_n13_loop", 13, 16, 32, 2, True, 981, [981], seed=15),    # K>12 per-frame loop
        attention_case(ref, "sdedit_n2_d40", 2, 32, 80, 2, False, 0, [], seed=16),        # head dim 40
    ]
    golden.save_ext_attn(GOLDEN_DIR, attn)
    golden.save_block_passes(GOLDEN_DIR, block_case(ref, ref_util))
    unet_c1 = {"pnp": unet_case(ref, "pnp"), "sdedit": unet_case(ref, "sdedit", n_timesteps=10)}
    for mode, c in unet_c1.items():
        torch.save(c, os.path.join(GOLDEN_DIR, f"unet_c1_{mode}.pt"))
    torch.save(live_cases(ref, ref_util), os.path.join(GOLDEN_DIR, "reference_live.pt"))
    drivers = {"run_tokenflow_pnp.py": driver_protocol("run_tokenflow_pnp.py", unet_c1["pnp"]),
               "run_tokenflow_sdedit.py": driver_protocol("run_tokenflow_sdedit.py", unet_c1["sdedit"])}
    with open(os.path.join(GOLDEN_DIR, "driver_protocol.json"), "w") as f:
        json.dump(drivers, f, indent=None, separators=(",", ":"))
        f.write("\n")
    for root, _, files in sorted(os.walk(GOLDEN_DIR)):
        for f in sorted(files):
            path = os.path.join(root, f)
            size = os.path.getsize(path)
            assert size < 1 << 20, (path, size)
            print(os.path.relpath(path, GOLDEN_DIR), size)


if __name__ == "__main__":
    main()
