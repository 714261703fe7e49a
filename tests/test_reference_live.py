"""CPU tier: the oracle against outputs of the UNMODIFIED reference hooks and helpers on fresh seeds,
stored in tests/golden/reference_live.pt by oracle/gen_golden.py (the reference's extended attention on
small blocks, its batch_cosine_sim and isinstance_str)."""
import os

import pytest
import torch

from oracle import tokenflow_oracle as O
from tokenflow_b200 import sd_unet


@pytest.fixture(scope="module")
def live(golden_dir):
    return torch.load(os.path.join(golden_dir, "reference_live.pt"), weights_only=False)


@pytest.mark.parametrize("seed,n,S,dim,heads,pnp,inject", [
    (101, 2, 24, 32, 2, False, False), (102, 4, 20, 64, 4, True, True), (103, 4, 20, 64, 4, True, False),
    (104, 13, 8, 32, 4, True, True)])
def test_live_extended_attention(live, seed, n, S, dim, heads, pnp, inject):
    c = live["attention"][seed]
    assert (c["n"], c["S"], c["dim"], c["heads"], c["inject"]) == (n, S, dim, heads, inject)
    block = sd_unet.BasicTransformerBlock(dim, heads, dim // heads, 16).eval()
    block.attn1.load_state_dict(c["state_dict"])
    x = c["x"]
    with torch.no_grad():
        a = block.attn1
        got = a.to_out[0](O.extended_attention(a.to_q(x), a.to_k(x), a.to_v(x), heads, a.scale, inject))
    assert torch.allclose(got, c["out"], atol=2e-6, rtol=1e-5)


def test_live_cosine_sim_and_isinstance_str(live):
    from tokenflow_b200.util import isinstance_str
    cs = live["cosine_sim"]
    # the same ops as the reference; bit-equal where the reference ran, and a BLAS built for another CPU
    # may order the 24-term dot products differently
    assert torch.allclose(O.cosine_sim(cs["x"], cs["y"]), cs["out"], atol=1e-6, rtol=0)
    blk = sd_unet.BasicTransformerBlock(16, 2, 8, 8)
    assert len(live["isinstance_str"]) == 4
    for name, want in live["isinstance_str"].items():
        assert isinstance_str(blk, name) == want
