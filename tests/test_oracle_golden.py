"""CPU tier: the oracle restatement against the golden vectors the UNMODIFIED reference produced
(oracle/gen_golden.py), and against the independent numpy closed form."""
import numpy as np
import pytest
import torch

from oracle import closed_form as CF
from oracle import golden
from oracle import tokenflow_oracle as O


@pytest.fixture(scope="module")
def attn_cases(golden_dir):
    return golden.load_ext_attn(golden_dir)


@pytest.fixture(scope="module")
def block_case(golden_dir):
    return golden.load_block_passes(golden_dir)


def _to_out(case, o):
    w, b = case["state_dict"]["to_out.0.weight"], case["state_dict"]["to_out.0.bias"]
    return o @ w.T + b


def test_extended_attention_matches_reference(attn_cases):
    assert len(attn_cases) >= 6
    for c in attn_cases:
        scale = (c["dim"] // c["heads"]) ** -0.5
        o = O.extended_attention(c["q"], c["k"], c["v"], c["heads"], scale, inject=c["inject"])
        got = _to_out(c, o)
        assert torch.allclose(got, c["out"], atol=2e-6, rtol=1e-5), c["name"]


def test_injection_flag_matters(attn_cases):
    c = next(c for c in attn_cases if c["name"] == "pnp_n3_inject")
    scale = (c["dim"] // c["heads"]) ** -0.5
    o = _to_out(c, O.extended_attention(c["q"], c["k"], c["v"], c["heads"], scale, inject=False))
    assert not torch.allclose(o, c["out"], atol=1e-3)


def test_closed_form_matches_reference(attn_cases):
    for c in attn_cases:
        scale = (c["dim"] // c["heads"]) ** -0.5
        o = CF.extended_attention(c["q"].numpy(), c["k"].numpy(), c["v"].numpy(), c["heads"], scale, c["inject"])
        got = _to_out(c, torch.from_numpy(o).float())
        assert torch.allclose(got, c["out"], atol=5e-6, rtol=1e-5), c["name"]


def test_nn_field_matches_reference(block_case):
    piv = block_case["pivotal"]["pivot_hidden_states"]
    ln_w, ln_b = block_case["state_dict"]["norm1.weight"], block_case["state_dict"]["norm1.bias"]
    B, S, dim = block_case["B"], block_case["S"], block_case["dim"]
    for fr in block_case["frames"]:
        norm = torch.nn.functional.layer_norm(fr["hidden"], (dim,), ln_w, ln_b).view(3, B, S, dim)
        idx1, idx2 = O.nn_field(norm[0], piv[0], fr["batch_idx"])
        assert torch.equal(idx1, fr["idx1"])
        if fr["idx2"] is None:
            assert idx2 is None
        else:
            assert torch.equal(idx2, fr["idx2"])
        # independent closed form (fp64): identical indices on this data
        kf = fr["batch_idx"]
        cf1 = CF.nn_index(norm[0].reshape(-1, dim).numpy(), piv[0][kf].numpy())
        assert np.array_equal(cf1, fr["idx1"].numpy())


def test_blend_weights_table():
    # SURVEY.md §8(a5): B=8 → [.6225,.6514,.6792,.7058,.7311,.7109,.6971,.6869], independent of batch index
    w = O.blend_weights(3, 8)
    ref = torch.tensor([.6225, .6514, .6792, .7058, .7311, .7109, .6971, .6869])
    assert torch.allclose(w, ref, atol=5e-5)
    assert torch.allclose(O.blend_weights(1, 8), w)
    assert all(abs(CF.blend_weight(f, 8) - float(w[f])) < 1e-6 for f in range(8))


def test_block_self_attention_matches_reference(block_case):
    """Whole self-attention stage (pivotal + frame passes) of the reference block."""
    from tokenflow_b200 import sd_unet
    dim, heads, ctx = block_case["dim"], block_case["heads"], block_case["ctx"]
    block = sd_unet.BasicTransformerBlock(dim, heads, dim // heads, ctx).eval()
    block.load_state_dict(block_case["state_dict"])
    scale = (dim // heads) ** -0.5

    def attn1(x):
        a = block.attn1
        o = O.extended_attention(a.to_q(x), a.to_k(x), a.to_v(x), heads, scale, inject=False)
        return a.to_out[0](o)

    def rest(h, c):
        h = block.attn2(block.norm2(h), encoder_hidden_states=c) + h
        return block.ff(block.norm3(h)) + h

    st = O.BlockState()
    with torch.no_grad():
        p = block_case["pivotal"]
        h = O.block_self_attention(st, p["hidden"], block.norm1(p["hidden"]), True, 0, attn1)
        assert torch.allclose(st.kf_attn_output, p["kf_attn_output"], atol=2e-6, rtol=1e-5)
        assert torch.allclose(rest(h, p["ctx"]), p["out"], atol=1e-5, rtol=1e-5)
        for fr in block_case["frames"]:
            h = O.block_self_attention(st, fr["hidden"], block.norm1(fr["hidden"]), False, fr["batch_idx"], attn1)
            assert torch.allclose(rest(h, fr["ctx"]), fr["out"], atol=1e-5, rtol=1e-5)


def test_propagate_closed_form(block_case):
    K, B, S, dim = block_case["K"], block_case["B"], block_case["S"], block_case["dim"]
    A = block_case["pivotal"]["kf_attn_output"]
    for fr in block_case["frames"]:
        got = O.propagate(A, fr["idx1"], fr["idx2"], fr["batch_idx"], B)
        cf = CF.propagate(A.view(3, K, S, dim).numpy(), fr["idx1"].numpy(),
                          None if fr["idx2"] is None else fr["idx2"].numpy(), fr["batch_idx"], B)
        assert np.allclose(got.numpy(), cf, atol=1e-6)


def test_fp16_emulated_similarity_is_monotone_rounding():
    torch.manual_seed(0)
    x, y = torch.randn(64, 32), torch.randn(48, 32)
    s16 = O.nn_sim_fp16_emulated(x, y)
    s32 = O.cosine_sim(x, y)
    assert s16.dtype == torch.float16
    assert (s16.float() - s32).abs().max() < 2e-3
