"""GPU tier (-m gpu): the sm_100a kernels, called through the C ABI (tokenflow_b200.ops.CudaOps →
libtokenflow_b200.so), against the oracle on the same seeded inputs, against the committed golden
vectors, and — at BASELINE full sizes — through size-independent properties.

Tolerances (from BASELINE.json north_star): NN indices bit-exact; attention outputs within 1e-3
(fp16).  "Bit-exact" for the NN field means: equal to the argmax of the reference GPU arithmetic
(fp32 normalise → fp16 operands → fp32-accumulated dot → fp16 → first max).  The only admissible
deviation is inside a *tie class*: two candidates whose fp16 similarity differs by ≤ 1 fp16 ulp,
where the winner depends on the fp32 accumulation order of the GEMM (cuBLAS's own order is not
specified either).  Such rows are counted, bounded, and every one of them is checked.
"""
import pytest
import torch

from oracle import golden
from oracle import tokenflow_oracle as O
from oracle.oracle_ops import OracleOps

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ops():
    from tokenflow_b200.ops import CudaOps
    return CudaOps()


def _video_like(F, K, S, dim, seed, noise=0.3, device="cuda"):
    """pivot features ~ layer-normed noise; frame tokens = permuted keyframe tokens + noise
    (SURVEY.md §8d: iid features understate tie/locality effects)."""
    g = torch.Generator(device="cpu").manual_seed(seed)
    piv = torch.nn.functional.layer_norm(torch.randn(K, S, dim, generator=g), (dim,))
    x = torch.empty(F, S, dim)
    for f in range(F):
        x[f] = piv[f % K][torch.randperm(S, generator=g)] + noise * torch.randn(S, dim, generator=g)
    return x.to(device), piv.to(device)


# ------------------------------------------------------------------------------------------------
# unit rows
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("rows,dim", [(1, 8), (77, 40), (4096, 320), (1000, 1280)])
def test_unit_rows(ops, rows, dim):
    torch.manual_seed(rows + dim)
    x = torch.randn(rows, dim, device="cuda") * 3 + 0.5
    got = ops.unit_rows(x)
    want = (x / x.norm(dim=-1, keepdim=True)).half()
    assert got.dtype == torch.float16 and got.shape == x.shape
    diff = (got.float() - want.float()).abs()
    # identical up to the last-ulp rounding of the fp32 norm reduction order
    assert diff.max().item() <= 1e-3
    assert (got != want).float().mean().item() < 2e-3
    got16 = ops.unit_rows(x.half())
    assert (got16.float() - want.float()).abs().max().item() < 2e-3


@pytest.mark.parametrize("rows,dim", [(3, 8), (100, 40), (4096, 320), (2048, 640), (512, 1280)])
def test_layernorm_unit_rows(ops, rows, dim):
    """norm1 + row normalisation fused (frame pass): equals LayerNorm in fp32 followed by tf_unit_rows."""
    torch.manual_seed(rows + dim)
    norm = torch.nn.LayerNorm(dim).cuda().half()
    with torch.no_grad():
        norm.weight.uniform_(0.5, 1.5)
        norm.bias.uniform_(-0.3, 0.3)
    x = (torch.randn(rows, dim, device="cuda") * 2 + 0.3).half()
    got = ops.layernorm_unit_rows(x, norm)
    y = torch.nn.functional.layer_norm(x.float(), (dim,), norm.weight.float(), norm.bias.float(), norm.eps)
    want = (y / y.norm(dim=-1, keepdim=True)).half()
    assert got.dtype == torch.float16 and got.shape == x.shape
    assert (got.float() - want.float()).abs().max().item() <= 1e-3
    assert (got != want).float().mean().item() < 5e-3         # last-ulp rounding of the fp32 statistics only
    # strided source-stream view (first third of a [3B, S, dim] tensor)
    x3 = torch.cat([x, x * 2, x + 1]).view(3, rows, dim)
    assert torch.equal(ops.layernorm_unit_rows(x3[0], norm), got)


def test_unit_rows_empty(ops):
    assert ops.unit_rows(torch.empty(0, 64, device="cuda")).shape == (0, 64)


# ------------------------------------------------------------------------------------------------
# propagate: bit exact (same fp32 arithmetic as the reference expression)
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("F,K,S,dim,batch", [(2, 2, 16, 8, 1), (4, 3, 40, 64, 0), (4, 3, 40, 64, 2),
                                            (8, 5, 1024, 640, 3), (8, 5, 4096, 320, 4)])
@pytest.mark.parametrize("with_residual", [True, False])
def test_propagate_bit_exact(ops, F, K, S, dim, batch, with_residual):
    from tokenflow_b200.ops import blend_weights
    torch.manual_seed(F * 1000 + S)
    A = torch.randn(3, K, S, dim, device="cuda").half()
    idx_a = torch.randint(0, S, (F, S), device="cuda", dtype=torch.int32)
    idx_b = torch.randint(0, S, (F, S), device="cuda", dtype=torch.int32) if batch > 0 else None
    res = torch.randn(3 * F, S, dim, device="cuda").half() if with_residual else None
    kf_a, kf_b, w = [batch] * F, [batch - 1 if batch > 0 else -1] * F, blend_weights(F)
    ref = OracleOps().propagate(A, idx_a, idx_b, kf_a, kf_b, w, res)         # fp32 when blended
    got32 = ops.propagate(A, idx_a, idx_b, kf_a, kf_b, w, res, out_dtype=torch.float32)
    if ref.dtype == torch.float32:        # blended: the reference's promoted dtype, bit for bit
        assert torch.equal(got32, ref)
    else:                                 # batch 0: the reference stays in fp16 (fp32 add, one rounding)
        assert torch.equal(got32.half(), ref)
    got16 = ops.propagate(A, idx_a, idx_b, kf_a, kf_b, w, res)
    assert got16.dtype == torch.float16 and torch.equal(got16, ref.half())


def test_propagate_mixed_frame_table(ops):
    """Per-frame tables (frame-granular sharding): frames of different batches in one launch."""
    from tokenflow_b200.ops import blend_weights
    torch.manual_seed(3)
    K, S, dim, B = 4, 64, 32, 4
    A = torch.randn(3, K, S, dim, device="cuda").half()
    w = blend_weights(B)
    kf_a, kf_b, ww = [0, 1, 1, 3], [-1, 0, 0, 2], [1.0, w[0], w[3], w[2]]
    idx_a = torch.randint(0, S, (4, S), device="cuda", dtype=torch.int32)
    idx_b = torch.randint(0, S, (4, S), device="cuda", dtype=torch.int32)
    got = ops.propagate(A, idx_a, idx_b, kf_a, kf_b, ww, None, out_dtype=torch.float32)
    ref = OracleOps().propagate(A, idx_a, idx_b, kf_a, kf_b, ww, None)
    assert torch.equal(got, ref.float())


def test_propagate_identity_roundtrip(ops):
    """Size-independent property at the BASELINE C2 top-level shape: identity indices and a single
    keyframe reproduce the keyframe slab for every frame and stream."""
    K, S, dim, F = 5, 4096, 320, 8
    A = torch.randn(3, K, S, dim, device="cuda").half()
    ident = torch.arange(S, device="cuda", dtype=torch.int32).repeat(F, 1)
    out = ops.propagate(A, ident, None, [2] * F, [-1] * F, [1.0] * F, None).view(3, F, S, dim)
    assert torch.equal(out, A[:, 2:3].expand(3, F, S, dim))


# ------------------------------------------------------------------------------------------------
# NN field
# ------------------------------------------------------------------------------------------------
def _check_nn(ops, x, piv, kf_a, kf_b, max_tie_frac=5e-3):
    F, S, dim = x.shape
    xu, pu = ops.unit_rows(x), ops.unit_rows(piv)
    idx_a, idx_b = ops.nn_field(xu, pu, kf_a, kf_b)
    torch.cuda.synchronize()
    total, ties = 0, 0
    for f in range(F):
        for kf, idx in ((kf_a[f], idx_a), (kf_b[f], idx_b)):
            if kf < 0:
                continue
            # the kernel's own fp16 operands, dot products accumulated in fp64, rounded to fp16
            sim16 = (xu[f].double() @ pu[kf].double().T).float().half()
            want = sim16.argmax(dim=-1)
            got = idx[f].long()
            assert got.min() >= 0 and got.max() < S
            bad = (got != want).nonzero().flatten()
            total += S
            ties += bad.numel()
            if bad.numel():
                s_got = sim16[bad, got[bad]].float()
                s_want = sim16[bad, want[bad]].float()
                ulp = 2.0 ** (torch.floor(torch.log2(s_want.abs().clamp_min(1e-8))) - 10)
                assert ((s_want - s_got).abs() <= ulp * 1.001).all(), "NN index outside the tie class"
    assert ties <= max(2, int(max_tie_frac * total)), f"{ties}/{total} rows differ from the oracle"
    return idx_a, idx_b, ties, total


@pytest.mark.parametrize("F,K,S,dim", [
    (2, 2, 64, 32),        # tiny, partial tiles everywhere
    (3, 3, 144, 320),      # SD2.1 mid-level token count: 144 = 128 + 16
    (4, 3, 576, 320),      # cfg 0 (256-row tiles), S not a multiple of 256
    (4, 3, 1024, 640),     # cfg 1
    (4, 3, 256, 1280),     # cfg 2 (streamed A)
    (2, 2, 4, 16),         # S < 8 (toy UNet mid block)
])
def test_nn_field_vs_oracle(ops, F, K, S, dim):
    x, piv = _video_like(F, K, S, dim, seed=S + dim)
    kf_a = [min(f, K - 1) for f in range(F)]
    kf_b = [a - 1 for a in kf_a]                      # first frame: -1 (no second keyframe)
    _check_nn(ops, x, piv, kf_a, kf_b)


def test_nn_field_matches_cublas_path(ops):
    """The reference's own GPU arithmetic, executed here: fp16 cuBLAS GEMM (fp16 output) + argmax.  Every index that
    differs from cuBLAS's is classified against cuBLAS's OWN similarity values: both candidates must lie within 2 fp16
    ulp of each other (each fp32-accumulated dot rounds to fp16 at most one ulp apart between two accumulation orders),
    i.e. the row is a tie class whose winner the reference's GEMM does not pin either.  Counts are reported."""
    F, K, S, dim = 4, 2, 1024, 320
    x, piv = _video_like(F, K, S, dim, seed=9)
    xu, pu = ops.unit_rows(x), ops.unit_rows(piv)
    idx_a, idx_b = ops.nn_field(xu, pu, [1] * F, [0] * F)
    total = mism = tie_class = 0
    for idx, kf in ((idx_a, 1), (idx_b, 0)):
        sim = xu.view(-1, dim) @ pu[kf].T                       # fp16 cuBLAS output, like util.py:68 under autocast
        ref = sim.argmax(-1)
        got = idx.long().view(-1)
        bad = (got != ref).nonzero().squeeze(1)
        total += got.numel()
        mism += bad.numel()
        if bad.numel():
            gap = (sim[bad, ref[bad]].float() - sim[bad, got[bad]].float()).abs()
            tie_class += int((gap <= 2.0 ** -10).sum())         # 2 ulp of fp16 values in [0.5, 1]
    msg = f"NN field vs cuBLAS + argmax: {mism} of {total} indices differ, {tie_class} of them inside an fp16 tie class"
    print(msg)
    assert mism <= 0.005 * total, msg
    # all of them tie classes — up to the few rows where cuBLAS itself may be more than one ulp off the exactly rounded
    # dot (PyTorch lets it reduce split-K partial sums in fp16: allow_fp16_reduced_precision_reduction defaults to True)
    assert mism - tie_class <= 5e-4 * total, msg


def test_nn_field_first_index_on_exact_ties(ops):
    """Duplicate keyframe tokens: torch.argmax returns the first maximal index, so must we."""
    S, dim = 256, 64
    g = torch.Generator().manual_seed(1)
    base = torch.randn(S // 2, dim, generator=g)
    piv = torch.cat([base, base]).unsqueeze(0).cuda()           # token c and c + S/2 are identical
    x = (base[torch.randperm(S // 2, generator=g)]).repeat(2, 1).unsqueeze(0).cuda()
    idx_a, _ = ops.nn_field(ops.unit_rows(x), ops.unit_rows(piv), [0], [-1])
    assert idx_a.max().item() < S // 2                          # never the duplicate in the upper half


def test_nn_field_recovers_permutation_full_size(ops):
    """BASELINE C2 top level (F=8, S=4096, dim=320, K=5): frame tokens are an exact permutation of
    the keyframe tokens, so the NN field must invert the permutation (self-similarity is the max)."""
    F, K, S, dim = 8, 5, 4096, 320
    g = torch.Generator().manual_seed(4)
    piv = torch.randn(K, S, dim, generator=g).cuda()
    perms = [torch.randperm(S, generator=g) for _ in range(F)]
    kf_a = [3] * F
    kf_b = [2] * F
    x = torch.stack([piv[3][p.cuda()] for p in perms])
    idx_a, idx_b = ops.nn_field(ops.unit_rows(x), ops.unit_rows(piv), kf_a, kf_b)
    for f in range(F):
        assert torch.equal(idx_a[f].long().cpu(), perms[f])
    assert idx_b.min().item() >= 0 and idx_b.max().item() < S


# ------------------------------------------------------------------------------------------------
# extended attention
# ------------------------------------------------------------------------------------------------
def _attn_ref(q, k, v, heads, scale, inject):
    """fp32 oracle evaluated on the fp16-rounded inputs the kernel sees."""
    return O.extended_attention(q.float(), k.float(), v.float(), heads, scale, inject)


@pytest.mark.parametrize("n,S,heads,d,inject", [
    (1, 16, 1, 8, False),
    (2, 48, 2, 16, False),
    (3, 48, 4, 16, True),
    (2, 200, 2, 40, False),      # SD1.5 top-level head dim, ragged key tiles
    (3, 256, 2, 40, True),
    (2, 160, 2, 80, False),
    (3, 1024, 2, 80, True),      # SD1.5 middle level (two-half kernel), injected
    (2, 300, 2, 128, False),     # widest head dim of the two-half kernel, ragged key tiles
    (2, 384, 1, 96, False),
    (2, 96, 2, 160, True),
    (2, 144, 3, 64, False),      # SD2.1 head dim, 144 tokens
    (13, 16, 2, 16, True),       # K > 12 (the reference's per-frame loop path)
])
def test_ext_attn_vs_oracle(ops, n, S, heads, d, inject):
    torch.manual_seed(n * 100 + S + d)
    dim = heads * d
    q, k, v = (torch.randn(3 * n, S, dim, device="cuda").half() for _ in range(3))
    scale = d ** -0.5
    got = ops.ext_attn(q, k, v, heads, scale, inject)
    want = _attn_ref(q, k, v, heads, scale, inject)
    assert got.dtype == torch.float16 and got.shape == q.shape
    assert (got.float() - want).abs().max().item() < 1e-3         # north_star tolerance


def test_ext_attn_peaky_softmax(ops):
    """Large logits (running-max rescale path): scaled q so that the row max moves between tiles."""
    torch.manual_seed(0)
    n, S, heads, d = 2, 512, 2, 64
    q = (torch.randn(3 * n, S, heads * d, device="cuda") * 6).half()
    k = torch.randn(3 * n, S, heads * d, device="cuda").half()
    v = torch.randn(3 * n, S, heads * d, device="cuda").half()
    got = ops.ext_attn(q, k, v, heads, d ** -0.5, False)
    want = _attn_ref(q, k, v, heads, d ** -0.5, False)
    # near one-hot softmax: outputs approach raw |v| ~ 3, where one fp16 ulp is already 2e-3 —
    # the 1e-3 bound applies at unit magnitude and scales with the fp16 spacing above it
    assert torch.allclose(got.float(), want, atol=1e-3, rtol=1.5e-3)


def test_ext_attn_golden(ops, golden_dir):
    """Golden vectors of the unmodified reference (fp32 CPU) through the CUDA kernel (fp16)."""
    for c in golden.load_ext_attn(golden_dir):
        q, k, v = (c[t].cuda().half() for t in ("q", "k", "v"))
        scale = (c["dim"] // c["heads"]) ** -0.5
        o = ops.ext_attn(q, k, v, c["heads"], scale, c["inject"]).float().cpu()
        got = o @ c["state_dict"]["to_out.0.weight"].T + c["state_dict"]["to_out.0.bias"]
        assert (got - c["out"]).abs().max().item() < 3e-3, c["name"]   # fp16 inputs vs fp32 reference


def test_ext_attn_fused_qkv_stride(ops):
    """q,k,v as views of one fused [3n,S,3*dim] projection buffer (token stride 3*dim)."""
    torch.manual_seed(2)
    n, S, heads, d = 2, 64, 2, 40
    dim = heads * d
    qkv = torch.randn(3 * n, S, 3 * dim, device="cuda").half()
    q, k, v = qkv[..., :dim], qkv[..., dim:2 * dim], qkv[..., 2 * dim:]
    got = ops.ext_attn(q, k, v, heads, d ** -0.5, True)
    want = _attn_ref(q.contiguous(), k.contiguous(), v.contiguous(), heads, d ** -0.5, True)
    assert (got.float() - want).abs().max().item() < 1e-3


def test_ext_attn_uniform_values_full_size(ops):
    """BASELINE C2 top level (n=5, S=4096, h=8, d=40): with V constant per head-channel the output
    must equal that constant for any q/k (softmax rows sum to one) — checks masking, the row-sum and
    the 20 480-key streaming loop without an O(S²) oracle; plus sampled rows against SDPA."""
    n, S, heads, d = 5, 4096, 8, 40
    dim = heads * d
    torch.manual_seed(1)
    q = torch.randn(3 * n, S, dim, device="cuda").half()
    k = torch.randn(3 * n, S, dim, device="cuda").half()
    c = torch.randn(dim, device="cuda").half()
    v = c.expand(3 * n, S, dim).contiguous()
    got = ops.ext_attn(q, k, v, heads, d ** -0.5, False)
    assert (got.float() - c.float()).abs().max().item() < 2e-3
    # sampled rows vs torch SDPA in fp32 on random V
    v = torch.randn(3 * n, S, dim, device="cuda").half()
    got = ops.ext_attn(q, k, v, heads, d ** -0.5, False)
    rows = torch.tensor([0, 1, 777, 4095], device="cuda")
    for smp in (0, n + 2, 2 * n + 4):
        s = smp // n
        qq = q[smp, rows].view(len(rows), heads, d).permute(1, 0, 2).float()
        if s == 0:
            kk, vv = k[smp], v[smp]
        else:
            kk, vv = k[s * n:(s + 1) * n].reshape(n * S, dim), v[s * n:(s + 1) * n].reshape(n * S, dim)
        kk = kk.view(-1, heads, d).permute(1, 0, 2).float()
        vv = vv.view(-1, heads, d).permute(1, 0, 2).float()
        ref = torch.softmax(qq @ kk.transpose(1, 2) * d ** -0.5, dim=-1) @ vv
        ref = ref.permute(1, 0, 2).reshape(len(rows), dim)
        assert (got[smp, rows].float() - ref).abs().max().item() < 1e-3


# ------------------------------------------------------------------------------------------------
# other BASELINE configurations (C3: K = 10 keyframes; C4: SD2.1 shapes; C5: K > 12) and the sharded form
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n,S,heads,d", [
    (10, 256, 2, 40),      # C3: 80 frames / stride 8 -> 10 keyframes, 2560 keys per query here
    (5, 576, 2, 64),       # C4: SD2.1 head dim 64, 576 tokens (24x24 level of a 768^2 frame)
    (25, 64, 2, 40),       # C5 stride 8: 25 keyframes (the reference's K > 12 per-frame loop)
])
def test_ext_attn_other_configs(ops, n, S, heads, d):
    torch.manual_seed(n + S)
    dim = heads * d
    q, k, v = (torch.randn(3 * n, S, dim, device="cuda").half() for _ in range(3))
    for inject in (False, True):
        got = ops.ext_attn(q, k, v, heads, d ** -0.5, inject)
        want = _attn_ref(q, k, v, heads, d ** -0.5, inject)
        assert torch.allclose(got.float(), want, atol=1e-3, rtol=1.5e-3)


def test_ext_attn_table_matches_whole_pass(ops):
    """The sharded-pass entry point (per-sample q/k/v slab table) reproduces the whole-pass result
    rank by rank — the arithmetic behind tests/test_sharded_cpu.py, on the CUDA kernel."""
    from tokenflow_b200.tokenflow_utils import PivotalShard
    torch.manual_seed(5)
    K, S, heads, d = 5, 320, 2, 40
    dim = heads * d
    q, k, v = (torch.randn(3 * K, S, dim, device="cuda").half() for _ in range(3))
    for inject in (False, True):
        whole = ops.ext_attn(q, k, v, heads, d ** -0.5, inject)
        for G in (2, 8):
            m = -(-3 * K // G)
            pad = G * m - 3 * K
            padded = [torch.cat([t, t[-1:].expand(pad, S, dim)]) if pad else t for t in (q, k, v)]
            for r in range(G):
                sh = PivotalShard(G, r, K)
                q_local = padded[0][r * m:(r + 1) * m]
                q_src = padded[0] if inject else q_local
                out = ops.ext_attn_table(q_src, padded[1], padded[2], sh.attention_table(inject), heads, d ** -0.5)
                for j, i in enumerate(sh.slots):
                    if i < 3 * K:
                        if inject and i >= K:
                            # the whole pass pairs the uncond / cond sample of a keyframe (shared q, k: one kernel computes
                            # their probabilities once); a rank that holds only one of the two runs the per-sample kernel
                            assert (out[j].float() - whole[i].float()).abs().max().item() < 1e-3, (G, r, j)
                        else:
                            assert torch.equal(out[j], whole[i]), (G, r, j)


def test_nn_field_sd21_token_counts(ops):
    """C4: 768^2 frames -> 9216 tokens at the top level (and 2304 one level down)."""
    for S, dim in ((9216, 320), (2304, 640)):
        x, piv = _video_like(2, 2, S, dim, seed=S)
        _check_nn(ops, x, piv, [1, 1], [0, -1])


def test_propagate_many_frames_one_launch(ops):
    """All 40 frames of C2 in one launch (per-frame table spanning 5 batches) == 5 per-batch launches."""
    from tokenflow_b200.ops import blend_weights
    torch.manual_seed(11)
    N, B, K, S, dim = 40, 8, 5, 256, 320
    A = torch.randn(3, K, S, dim, device="cuda").half()
    idx_a = torch.randint(0, S, (N, S), device="cuda", dtype=torch.int32)
    idx_b = torch.randint(0, S, (N, S), device="cuda", dtype=torch.int32)
    res = torch.randn(3, N, S, dim, device="cuda").half()
    w = blend_weights(B)
    kf_a = [g // B for g in range(N)]
    kf_b = [g // B - 1 if g >= B else -1 for g in range(N)]
    ww = [w[g % B] for g in range(N)]
    one = ops.propagate(A, idx_a, idx_b, kf_a, kf_b, ww, res.view(3 * N, S, dim)).view(3, N, S, dim)
    for i in range(K):
        sl = slice(i * B, (i + 1) * B)
        part = ops.propagate(A, idx_a[sl], idx_b[sl] if i > 0 else None, kf_a[sl], kf_b[sl], ww[sl],
                             res[:, sl].reshape(3 * B, S, dim)).view(3, B, S, dim)
        assert torch.equal(one[:, sl], part)
