"""GPU tier (-m gpu), round 2: the fused norm1 kernel, the fused CFG+DDIM kernel, chunked launches beyond the
per-launch table sizes, the CUDA-graphed step, the hook layer at the SD1.5 top-level shape against the
reference's GPU arithmetic, strict-dtype edits, and the NCCL path on two GPUs (when two are visible)."""
import os
import socket
import subprocess
import sys

import pytest
import torch

from oracle import tokenflow_oracle as O
from oracle.oracle_ops import OracleOps
from tokenflow_b200 import sd_unet
from tokenflow_b200 import tokenflow_utils as tfu
from tokenflow_b200.editor import TokenFlowEditor, synthetic_inputs
from tokenflow_b200.scheduler import DDIMScheduler

pytestmark = pytest.mark.gpu
REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def ops():
    from tokenflow_b200.ops import CudaOps
    return CudaOps()


# ------------------------------------------------------------------------------------------------
# tf_layernorm_rows: norm1 -> (fp16 QKV operand, fp16 unit rows of the source samples)
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("b,S,dim,n_unit", [(3, 64, 40, 1), (15, 1024, 320, 5), (6, 256, 1280, 2), (4, 100, 640, 4)])
def test_layernorm_rows(ops, b, S, dim, n_unit):
    torch.manual_seed(b * S + dim)
    norm = torch.nn.LayerNorm(dim).cuda().half()
    with torch.no_grad():
        norm.weight.uniform_(0.5, 1.5)
        norm.bias.uniform_(-0.3, 0.3)
    x = (torch.randn(b, S, dim, device="cuda") * 2 + 0.3).half()
    y, unit = ops.layernorm_rows(x, norm, n_unit)
    with torch.autocast("cuda", dtype=torch.float16):
        y32 = norm(x)                                     # autocast: fp32 LayerNorm, the reference's norm1 output
    assert y32.dtype == torch.float32
    want_y = y32.half()                                   # the operand autocast hands the to_q/k/v GEMMs
    assert y.dtype == torch.float16 and y.shape == x.shape
    assert (y.float() - want_y.float()).abs().max().item() <= 4e-3          # <= 1 fp16 ulp at |y| < 8
    assert (y != want_y).float().mean().item() < 5e-3                       # last-ulp rounding of the fp32 statistics only
    want_u = ops.unit_rows(y32[:n_unit])
    assert unit.shape == (n_unit, S, dim)
    assert (unit.float() - want_u.float()).abs().max().item() <= 1e-3
    assert (unit != want_u).float().mean().item() < 5e-3
    # packed outputs: strided views of one buffer
    pack = torch.zeros(b, S, 3 * dim, device="cuda", dtype=torch.float16)
    y2, u2 = ops.layernorm_rows(x, norm, b, y_out=pack[..., :dim], unit_out=pack[..., 2 * dim:])
    assert torch.equal(pack[..., :dim], y) and torch.equal(pack[:n_unit, :, 2 * dim:], unit)
    assert pack[..., dim:2 * dim].abs().max().item() == 0


def test_layernorm_affine_cache_follows_weight_updates(ops):
    """ADVICE r1: the fp32 copies of norm1's affine parameters must follow in-place updates / reloads."""
    norm = torch.nn.LayerNorm(64).cuda().half()
    x = torch.randn(8, 64, device="cuda").half()
    a = ops.layernorm_unit_rows(x, norm).clone()
    with torch.no_grad():
        norm.bias.add_(1.0)                                # same Parameter object, new version
    b = ops.layernorm_unit_rows(x, norm)
    y = torch.nn.functional.layer_norm(x.float(), (64,), norm.weight.float(), norm.bias.float(), norm.eps)
    want = (y / y.norm(dim=-1, keepdim=True)).half()
    assert not torch.equal(a, b)
    assert (b.float() - want.float()).abs().max().item() <= 1e-3


# ------------------------------------------------------------------------------------------------
# tf_cfg_ddim: bit-identical to the eager expression (run_tokenflow_pnp.py:213-217)
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("step", [0, 7, 24, 49])
def test_cfg_ddim_bit_exact(ops, step):
    torch.manual_seed(step)
    sch = DDIMScheduler()
    sch.set_timesteps(50)
    unet = torch.nn.Linear(1, 1).cuda()                    # only a device carrier for the editor
    ed = TokenFlowEditor.__new__(TokenFlowEditor)
    torch.nn.Module.__init__(ed)
    ed.scheduler, ed.device = sch, torch.device("cuda")
    ed._t_host = [int(t) for t in sch.timesteps]
    coef = TokenFlowEditor._make_coef_table(ed)
    t = ed._t_host[step]
    x = torch.randn(5, 4, 64, 64, device="cuda").half()
    eps = torch.randn(10, 4, 64, 64, device="cuda").half().contiguous(memory_format=torch.channels_last)
    u, c = eps.chunk(2)
    g = 7.5
    want = sch.step(u + g * (c - u), t, x)["prev_sample"]
    got = ops.cfg_ddim(u, c, x, coef[step], g)
    assert got.dtype == torch.float16 and got.shape == x.shape
    assert torch.equal(got, want), (got.float() - want.float()).abs().max().item()


# ------------------------------------------------------------------------------------------------
# chunked launches: more frames / samples than one kernel's by-value tables hold
# ------------------------------------------------------------------------------------------------
def test_nn_field_and_propagate_200_frames(ops):
    """BASELINE C5 single-GPU shape class: F = 200 frames in one call (kMaxFrames = 64 per launch)."""
    torch.manual_seed(5)
    F, K, S, dim = 200, 25, 256, 320
    piv = torch.nn.functional.layer_norm(torch.randn(K, S, dim, device="cuda"), (dim,))
    x = torch.stack([piv[(f // 8)][torch.randperm(S, device="cuda")] for f in range(F)]) + 0.2 * torch.randn(F, S, dim, device="cuda")
    kf_a = [f // 8 for f in range(F)]
    kf_b = [(f // 8) - 1 if f >= 8 else -1 for f in range(F)]
    from tokenflow_b200.ops import blend_weights
    w = [blend_weights(8)[f % 8] for f in range(F)]
    xu, pu = ops.unit_rows(x), ops.unit_rows(piv)
    idx_a, idx_b = ops.nn_field(xu, pu, kf_a, kf_b)
    for f in (0, 63, 64, 65, 127, 128, 199):               # frames on both sides of every chunk boundary
        sim = (xu[f].double() @ pu[kf_a[f]].double().T).float().half()
        want = sim.argmax(-1)
        bad = idx_a[f].long() != want
        if bad.any():                                      # fp16 tie classes only
            gap = (sim[bad, want[bad]].float() - sim[bad, idx_a[f].long()[bad]].float()).abs().max().item()
            assert gap <= 1e-3 and bad.float().mean().item() < 0.01
    A = torch.randn(3, K, S, dim, device="cuda").half()
    res = torch.randn(3 * F, S, dim, device="cuda").half()
    got = ops.propagate(A, idx_a, idx_b, kf_a, kf_b, w, res)
    want = OracleOps().propagate(A, idx_a, idx_b, kf_a, kf_b, w, res).half()
    assert torch.equal(got, want)
    got32 = ops.propagate(A, idx_a, idx_b, kf_a, kf_b, w, res, out_dtype=torch.float32)
    want32 = OracleOps().propagate(A, idx_a, idx_b, kf_a, kf_b, w, res)
    assert got32.dtype == torch.float32 and torch.equal(got32, want32.float())


def test_ext_attn_more_samples_than_one_launch(ops):
    """n = 60 keyframes -> 180 (stream, keyframe) samples > kMaxAttnSamples = 160 per launch."""
    torch.manual_seed(6)
    n, S, heads, d = 60, 256, 2, 40
    dim = heads * d
    q, k, v = (torch.randn(3 * n, S, dim, device="cuda").half() for _ in range(3))
    got = ops.ext_attn(q, k, v, heads, d ** -0.5, False)
    table = [(0, 0, 0, 1), (n - 1, n - 1, n - 1, 1), (n, n, n, n), (2 * n - 1, n, n, n), (3 * n - 1, 2 * n, 2 * n, n)]
    want = OracleOps().ext_attn_table(q.float(), k.float(), v.float(), table, heads, d ** -0.5)
    for j, (smp, *_rest) in enumerate(table):
        assert (got[smp].float() - want[j]).abs().max().item() < 1e-3, smp


# ------------------------------------------------------------------------------------------------
# extended attention: a FULL (sample, head) slab at the C2 top-level shape, both kernels' variants
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("inject", [False, True])
def test_ext_attn_full_slab_c2_top_level(ops, inject):
    torch.manual_seed(11)
    n, S, heads, d = 5, 4096, 8, 40
    dim = heads * d
    q = torch.randn(3 * n, S, dim, device="cuda")
    k = (torch.randn(3 * n, S, dim, device="cuda") + 1.5 * q).half()        # peaked rows (video-like)
    q, v = q.half(), torch.randn(3 * n, S, dim, device="cuda").half()
    out = ops.ext_attn(q, k, v, heads, d ** -0.5, inject)
    for smp, head in ((n + 2, 3), (2 * n + 4, 7), (1, 0)):
        s_, f_ = divmod(smp, n)
        qs = f_ if (inject and s_ > 0) else smp
        qq = q[qs, :, head * d:(head + 1) * d].float()
        if s_ == 0:
            kk, vv = k[smp, :, head * d:(head + 1) * d].float(), v[smp, :, head * d:(head + 1) * d].float()
        else:
            k0 = 0 if inject else s_ * n
            kk = k[k0:k0 + n, :, head * d:(head + 1) * d].reshape(n * S, d).float()
            vv = v[s_ * n:(s_ + 1) * n, :, head * d:(head + 1) * d].reshape(n * S, d).float()
        ref = torch.softmax(qq @ kk.T * d ** -0.5, dim=-1) @ vv
        err = (out[smp, :, head * d:(head + 1) * d].float() - ref).abs().max().item()
        # every one of the 4096 query rows of the slab; peaked softmax rows carry |O| up to ~4, where the fp16
        # rounding of P (2^-11 relative) alone is 2e-3; rows are within 1e-3 of the fp16 grid of the exact output
        assert err < 2.5e-3, (smp, head, err)
        rel = ((out[smp, :, head * d:(head + 1) * d].float() - ref).norm() / ref.norm()).item()
        assert rel < 1e-3, (smp, head, rel)


# ------------------------------------------------------------------------------------------------
# paired samples (PnP q/k injection): one kernel computes S / P once per (uncond, cond) pair
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n,S,heads,d", [(3, 512, 2, 40), (5, 4096, 8, 40), (2, 320, 1, 24)])
def test_ext_attn_paired_kernel_equals_separate_samples(ops, monkeypatch, n, S, heads, d):
    """With injection the uncond and cond samples of a keyframe share q and k: the paired kernel (P [V_u | V_c] in one
    MMA) must reproduce what the per-sample kernel computes, and both must match the oracle."""
    torch.manual_seed(n * S + d)
    dim = heads * d
    q = torch.randn(3 * n, S, dim, device="cuda")
    k = (torch.randn(3 * n, S, dim, device="cuda") + 1.0 * q).half()
    q, v = q.half(), torch.randn(3 * n, S, dim, device="cuda").half()
    table = []
    for i in range(3 * n):
        s_, f_ = divmod(i, n)
        table.append((i, i, i, 1) if s_ == 0 else (f_, 0, s_ * n, n))            # injected: q, k of the source stream
    paired = ops.ext_attn_table(q, k, v, table, heads, d ** -0.5)
    launches0 = ops.launch_count()
    paired2 = ops.ext_attn(q, k, v, heads, d ** -0.5, True)
    assert ops.launch_count() - launches0 == 2                                    # one paired launch + the source samples
    assert torch.equal(paired, paired2)
    # the same samples one by one (a single-sample table cannot be paired)
    for i in (n, 2 * n - 1, 2 * n, 3 * n - 1, 0):
        single = ops.ext_attn_table(q, k, v, [table[i]], heads, d ** -0.5)[0]
        assert (single.float() - paired[i].float()).abs().max().item() < 1e-3, i
    want = OracleOps().ext_attn_table(q.float(), k.float(), v.float(), [table[n], table[3 * n - 1]], heads, d ** -0.5)
    assert (paired[n].float() - want[0]).abs().max().item() < 2.5e-3
    assert (paired[3 * n - 1].float() - want[1]).abs().max().item() < 2.5e-3
    assert ((paired[n].float() - want[0]).norm() / want[0].norm()).item() < 1e-3


@pytest.mark.parametrize("S,heads,d,n", [(4096, 8, 40, 5), (1024, 8, 80, 3), (256, 4, 160, 2), (576, 5, 64, 2), (64, 2, 40, 2)])
@pytest.mark.parametrize("inject", [False, True])
def test_ext_attn_query_row_ranges_tile_the_full_result(ops, S, heads, d, n, inject):
    """Multi-GPU token split: computing the query rows of all samples in G ranges and concatenating equals the
    full call, bit for bit (same kernel, same tiles)."""
    torch.manual_seed(S + d)
    dim = heads * d
    q, k, v = (torch.randn(3 * n, S, dim, device="cuda").half() for _ in range(3))
    table = []
    for i in range(3 * n):
        s_, f_ = divmod(i, n)
        table.append((i, i, i, 1) if s_ == 0 else ((f_, 0, s_ * n, n) if inject else (i, s_ * n, s_ * n, n)))
    full = ops.ext_attn_table(q, k, v, table, heads, d ** -0.5)
    for G in (2, 8):
        tiles = -(-S // 128)
        nrows = -(-tiles // G) * 128
        parts = [ops.ext_attn_table(q, k, v, table, heads, d ** -0.5, row0=r * nrows, nrows=nrows) for r in range(G)]
        got = torch.stack(parts).permute(1, 0, 2, 3).reshape(3 * n, G * nrows, dim)[:, :S]
        if nrows >= 256 or S <= 128:
            assert torch.equal(got, full), (G, (got.float() - full.float()).abs().max().item())
        else:      # a 128-row range runs the one-tile kernel where the full call runs a two-tile kernel: same math, other tiling
            assert (got.float() - full.float()).abs().max().item() < 1e-3, G


# ------------------------------------------------------------------------------------------------
# hook layer at the SD1.5 top-level shape vs the reference's GPU arithmetic (oracle ops under autocast)
# ------------------------------------------------------------------------------------------------
class _U(torch.nn.Module):
    def __init__(self, block):
        super().__init__()
        site = torch.nn.Module()
        site.transformer_blocks = torch.nn.ModuleList([block])
        ups = []
        for _ in range(4):
            u = torch.nn.Module()
            u.attentions = torch.nn.ModuleList([site, site, site])
            ups.append(u)
        self.up_blocks = torch.nn.ModuleList(ups)


class _W(torch.nn.Module):
    def __init__(self, unet):
        super().__init__()
        self.unet = unet


@pytest.mark.parametrize("inject", [False, True])
def test_block_sd15_top_level_shape_vs_reference_gpu_path(inject):
    """One SD1.5 top-level block (S = 4096, dim = 320, 8 heads x 40), K = 5 keyframes, B = 8 frames, PnP flavour with
    the q/k injection on / off: pivotal pass + frame passes 0 and 2, CUDA ops vs oracle ops under the same autocast.
    Every NN-index mismatch is classified against the oracle's own fp16 similarity values and counted."""

    def run(ops_obj):
        tfu._install_ops_for_testing(ops_obj)
        torch.manual_seed(3)
        block = sd_unet.BasicTransformerBlock(320, 8, 40, 768).cuda().half().eval()
        model = _W(_U(block))
        sched = [981, 961]
        tfu.register_extended_attention_pnp(model, sched)
        block.attn1.injection_schedule = sched
        tfu.set_tokenflow(model.unet)
        block.attn1.t = 981 if inject else 1
        K, B, S = 5, 8, 4096
        res = {}
        with torch.no_grad(), torch.autocast("cuda", dtype=torch.float16):
            h = torch.randn(3 * K, S, 320, device="cuda").half()
            ctx = torch.randn(3 * K, 77, 768, device="cuda").half()
            tfu.register_pivotal(model, True)
            res["piv"] = block(h, encoder_hidden_states=ctx).float()
            res["piv_unit_src"] = getattr(block, "_tf_pivot_unit", None)
            tfu.register_pivotal(model, False)
            for i in (0, 2):
                hf = (h[:K][i].unsqueeze(0).repeat(B, 1, 1) + 0.3 * torch.randn(B, S, 320, device="cuda").half())
                hf = torch.cat([hf, torch.randn(2 * B, S, 320, device="cuda").half()])
                tfu.register_batch_idx(model, i)
                res[f"out{i}"] = block(hf, encoder_hidden_states=torch.randn(3 * B, 77, 768, device="cuda").half()).float()
                res[f"idx{i}"] = tuple(None if t is None else t.long().reshape(B, S).clone() for t in block._tf_nn_idx)
                res[f"x{i}"] = hf[:B].clone()
        res["block"] = block
        return res

    want = run(OracleOps())
    got = run(None)
    # pivotal pass (extended attention + residual + cross-attn + FF), whole tensor
    assert torch.allclose(got["piv"], want["piv"], atol=4e-3, rtol=4e-3)
    total = mismatched = tie_class = 0
    for i in (0, 2):
        for which in (0, 1):
            g_idx, w_idx = got[f"idx{i}"][which], want[f"idx{i}"][which]
            if g_idx is None:
                assert w_idx is None
                continue
            bad = g_idx != w_idx
            total += g_idx.numel()
            mismatched += int(bad.sum())
            if bad.any():
                # the oracle's own similarity values (reference GPU arithmetic) at both candidates
                blk = want["block"]
                kf = i if which == 0 else i - 1
                with torch.autocast("cuda", dtype=torch.float16):
                    xn = blk.norm1(want[f"x{i}"])
                    pn = blk.pivot_hidden_states[0][kf]
                    sim = O.cosine_sim(xn.reshape(-1, 320), pn)                 # fp16 under autocast, like the reference
                rows = bad.reshape(-1).nonzero().squeeze(1)
                gap = (sim[rows, w_idx.reshape(-1)[rows]].float() - sim[rows, g_idx.reshape(-1)[rows]].float()).abs()
                tie_class += int((gap <= 2.0 ** -10).sum())                      # <= 1 fp16 ulp below 1.0
        # propagated output on the rows whose indices agree for both keyframes
        same = torch.ones_like(got[f"idx{i}"][0], dtype=torch.bool)
        for which in (0, 1):
            if got[f"idx{i}"][which] is not None:
                same &= got[f"idx{i}"][which] == want[f"idx{i}"][which]
        rows = same.reshape(1, -1).expand(3, -1).reshape(-1)
        g2, w2 = got[f"out{i}"].reshape(-1, 320)[rows], want[f"out{i}"].reshape(-1, 320)[rows]
        assert torch.allclose(g2, w2, atol=4e-3, rtol=4e-3)
    msg = f"NN indices: {mismatched} of {total} differ, {tie_class} of them inside an fp16 tie class"
    print(msg)
    assert mismatched == tie_class, msg                    # every mismatch is a <= 1-ulp tie in the reference's own values
    assert mismatched <= 5e-3 * total, msg


# ------------------------------------------------------------------------------------------------
# the CUDA-graphed fused step == the eager fused step, bit for bit, over all three injection variants
# ------------------------------------------------------------------------------------------------
def _editor(mode, steps, graph, n_frames=8, batch=2, latent=16, seed=1, strict=False):
    tfu._install_ops_for_testing(None)
    unet = sd_unet.build_unet("tiny", seed=seed, device="cuda", dtype=torch.float16)
    cfg = {"n_frames": n_frames, "batch_size": batch, "n_timesteps": steps, "guidance_scale": 7.5, "mode": mode,
           "pnp_attn_t": 0.5, "pnp_f_t": 0.8, "start": 0.9, "fused_pass": True, "cuda_graph": graph, "keyframe_seed": seed}
    x, text, pnp, src = synthetic_inputs(n_frames, latent, unet.config.cross_attention_dim, steps, seed=seed,
                                         device="cuda", dtype=torch.float16, ctx_len=7)
    ed = TokenFlowEditor(unet, DDIMScheduler(), tfu, cfg, text, pnp, source_latents=lambda t: src[t])
    ed.init_method()
    return ed, x


@pytest.mark.parametrize("mode,steps", [("pnp", 5), ("sdedit", 10)])
def test_cuda_graph_step_identical_to_eager(mode, steps):
    ed_e, x = _editor(mode, steps, graph=False)
    want = ed_e.sample_loop(x.clone())
    ed_g, x = _editor(mode, steps, graph=True)
    got = ed_g.sample_loop(x.clone())
    assert ed_g.keyframe_log == ed_e.keyframe_log
    if mode == "pnp":
        assert len(ed_g._graphs) == 3                      # q/k + conv injection, conv injection only, none
    assert all(e["replays"] >= 1 for e in ed_g._graphs.values())
    assert torch.equal(got, want), (got.float() - want.float()).abs().max().item()
    # per-launch event nodes of the graphs are readable when timing was on at capture
    ed_t, x = _editor(mode, steps, graph=True)             # (re-creates the global op object: enable timing after it)
    ops_ = tfu._ops()
    ops_.enable_timing(True)
    try:
        ed_t.step_index(x.clone(), 0)
        kt, n_steps = ed_t.graph_kernel_times()
        assert n_steps == 1
    finally:
        ops_.enable_timing(False)
    assert kt["tf_ext_attn"]["launches"] == 16 and kt["tf_ext_attn"]["ms"] > 0
    assert ed_t.graph_launches_per_step() >= 16 * 4


@pytest.mark.parametrize("graph", [False, True])
def test_dual_stream_step_matches_fused_step(graph):
    """The dual-stream schedule (pivotal pass on a side stream, frame pass on the current stream, per-block events)
    computes the same edit as the fused single call (body GEMMs / convs see other batch sizes: fp16 accumulation-order
    noise only), and its CUDA-graph replay equals its eager run bit for bit."""
    def run(dual, use_graph):
        ed, x = _editor("pnp", 5, graph=use_graph)
        ed.config["dual_stream"] = dual
        out = ed.sample_loop(x.clone())
        return out, ed.keyframe_log
    want, kf_w = run(False, False)
    got, kf_g = run(True, graph)
    assert kf_g == kf_w and torch.isfinite(got).all()
    rel = ((got.float() - want.float()).norm() / want.float().norm()).item()
    assert rel < 2e-2, rel
    if graph:
        eager, _ = run(True, False)
        assert torch.equal(got, eager)


def test_edit_with_strict_dtype(monkeypatch):
    """TOKENFLOW_B200_STRICT_DTYPE=1: the blended frame-pass output is the reference's promoted fp32; the edit
    still matches the reference GPU arithmetic."""
    import importlib.util
    spec = importlib.util.spec_from_file_location("_tf_gpu_hooks", os.path.join(REPO, "tests", "test_gpu_hooks.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    _run = mod._run
    want, kf_w, _ = _run(OracleOps(), "pnp", steps=2)
    monkeypatch.setenv("TOKENFLOW_B200_STRICT_DTYPE", "1")
    got, kf_g, _ = _run(None, "pnp", steps=2)
    assert kf_g == kf_w
    rel = (got - want).norm() / want.norm()
    assert rel.item() < 2e-2, rel.item()


# ------------------------------------------------------------------------------------------------
# the sharded CUDA path on ONE GPU: two "ranks" as two threads with an in-process all-gather
# ------------------------------------------------------------------------------------------------
class _ThreadWorld:
    """In-process stand-in for the communicator: rank threads meet at a barrier and concatenate their tensors
    (all ranks enqueue on the same default CUDA stream, so stream order makes the producers visible)."""

    def __init__(self, world):
        import threading
        self.world = world
        self.barrier = threading.Barrier(world, timeout=300)
        self.slots = [None] * world

    class _Rank:
        def __init__(self, parent, rank):
            self.parent, self.rank = parent, rank

        def all_gather(self, t):
            P = self.parent
            P.slots[self.rank] = t.contiguous()
            torch.cuda.current_stream().synchronize()      # rank threads may run on different (side) streams
            P.barrier.wait()
            out = torch.cat(list(P.slots))
            P.barrier.wait()
            return out

    def rank(self, r):
        return _ThreadWorld._Rank(self, r)


@pytest.mark.parametrize("token_split,dual", [(True, True), (True, False), (False, False)])
@pytest.mark.parametrize("world", [2, 4])
def test_sharded_cuda_path_in_one_process(world, token_split, dual):
    """The multi-GPU code path of the hooks on the CUDA kernels (packed q|k|v|unit gather, query-row split of the
    extended attention with the paired kernel, output re-assembly, sharded conv injection) with `world` rank threads
    on one GPU == the single-rank edit."""
    import threading
    steps, n_frames, batch = 4, 8, 2

    def edit(world_size, rank, comm, out, unet):
        try:
            cfg = {"n_frames": n_frames, "batch_size": batch, "n_timesteps": steps, "guidance_scale": 7.5, "mode": "pnp",
                   "pnp_attn_t": 0.5, "pnp_f_t": 0.8, "fused_pass": True, "cuda_graph": False, "keyframe_seed": 1,
                   "token_split": token_split, "dual_stream": dual and world_size > 1}
            x, text, pnp, src = synthetic_inputs(n_frames, 16, unet.config.cross_attention_dim, steps, seed=1,
                                                 device="cuda", dtype=torch.float16, ctx_len=7)
            ed = TokenFlowEditor(unet, DDIMScheduler(), tfu, cfg, text, pnp, source_latents=lambda t: src[t],
                                 world_size=world_size, rank=rank)
            if comm is not None:
                ed.attach_communicator(comm)
            ed.init_method()
            out[rank] = (ed.sample_loop(x).float(), ed.keyframe_log)
        except BaseException as ex:  # noqa: BLE001
            out[rank] = ex
            if comm is not None:
                comm.parent.barrier.abort()

    tfu._install_ops_for_testing(None)
    tfu._ops()                                              # one op object for all threads
    # the models are built one after the other in this thread: build_unet seeds the process-global CPU generator,
    # which rank threads would race for (separate processes each have their own)
    unets = [sd_unet.build_unet("tiny", seed=1, device="cuda", dtype=torch.float16) for _ in range(world + 1)]
    ref = {}
    edit(1, 0, None, ref, unets[world])
    assert not isinstance(ref[0], BaseException), ref[0]
    want, kf_want = ref[0]
    tw = _ThreadWorld(world)
    res = {}
    threads = [threading.Thread(target=edit, args=(world, r, tw.rank(r), res, unets[r])) for r in range(world)]
    for t in threads:
        t.start()
    for t in threads:
        t.join(timeout=600)
    for r in range(world):
        assert r in res and not isinstance(res[r], BaseException), res.get(r)
        got, kf = res[r]
        assert kf == kf_want
        assert torch.isfinite(got).all()
        rel = ((got - want).norm() / want.norm()).item()
        assert rel < 2e-2, (r, rel)
    assert torch.equal(res[0][0], res[1][0])               # every rank ends the step with the same latents


# ------------------------------------------------------------------------------------------------
# NCCL: two ranks on two GPUs == one rank  (skipped with fewer than two GPUs)
# ------------------------------------------------------------------------------------------------
_WORKER = r"""
import os, sys, json, torch
sys.path.insert(0, {repo!r})
import torch.distributed as dist
rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
torch.cuda.set_device(rank)
dist.init_process_group("nccl", device_id=torch.device("cuda", rank))
from tokenflow_b200 import sd_unet, tokenflow_utils as tfu
from tokenflow_b200.editor import TokenFlowEditor, synthetic_inputs
from tokenflow_b200.scheduler import DDIMScheduler
from tokenflow_b200.ops import Communicator
def edit(world, rank, graph, comm):
    unet = sd_unet.build_unet("tiny", seed=1, device="cuda", dtype=torch.float16)
    cfg = dict(n_frames=8, batch_size=2, n_timesteps=4, guidance_scale=7.5, mode="pnp", pnp_attn_t=0.5, pnp_f_t=0.8,
               fused_pass=True, cuda_graph=graph, keyframe_seed=1, check_keyframes=True)
    x, text, pnp, src = synthetic_inputs(8, 16, unet.config.cross_attention_dim, 4, seed=1, device="cuda", dtype=torch.float16, ctx_len=7)
    ed = TokenFlowEditor(unet, DDIMScheduler(), tfu, cfg, text, pnp, source_latents=lambda t: src[t], world_size=world, rank=rank)
    if comm is not None:
        ed.attach_communicator(comm)
    ed.init_method()
    return ed.sample_loop(x).float(), ed.keyframe_log
comm = Communicator(world, rank)
want, kf1 = edit(1, 0, False, None)
res = {{}}
for name, graph, c in (("capi_graph", True, comm), ("capi_eager", False, comm), ("torch_eager", False, None)):
    got, kf = edit(world, rank, graph, c)
    res[name] = dict(kf_equal=(kf == kf1), rel=float((got - want).norm() / want.norm()), finite=bool(torch.isfinite(got).all()))
comm.destroy()
if rank == 0:
    print("RESULT " + json.dumps(res), flush=True)
dist.destroy_process_group()
"""


def test_two_rank_nccl_edit_equals_single_rank(tmp_path):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    script = tmp_path / "worker.py"
    script.write_text(_WORKER.format(repo=REPO))
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
                        "--master-addr", "127.0.0.1", "--master-port", str(port), str(script)],
                       capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]
    import json
    line = [ln for ln in r.stdout.splitlines() if ln.startswith("RESULT ")][-1]
    res = json.loads(line[len("RESULT "):])
    for name, v in res.items():
        assert v["kf_equal"] and v["finite"], (name, v)
        assert v["rel"] < 2e-2, (name, v)                  # fp16 accumulation-order differences of the smaller batches
    assert res["capi_graph"]["rel"] == res["capi_eager"]["rel"]      # graph replay == eager, same kernels
