"""The decoder's fused cross-attention (cross_attn.cuh, etude_k_cross_attn): K|V projected inside the attention kernel per
frame of 256 encoder tokens.  Checked against the two-kernel path it replaces (gemm_bstat K|V + attention4), against fp64,
with an exact routing probe, and for the workspace it no longer needs."""
import pytest
import torch

pytestmark = pytest.mark.gpu

import gpu_diag as D  # noqa: E402  (tests/ is on sys.path via conftest)
from conftest import report  # noqa: E402
from etude_b200 import _lib  # noqa: E402
from test_decoder_kernels_gpu import _key_vec, _query_vec, attention_bound  # noqa: E402

P, stream = D.P, D.stream
bf = lambda t: t.to(torch.bfloat16)
LAYERS = ("decoder.layer_zero_freq.encoder_attention", "decoder.layers_freq.0.encoder_attention",
          "decoder.layers_freq.1.encoder_attention")
N_FRAMES = [1, 2, 37, 16384]   # 16 384 frames = the 32-window batch of bench.py


@pytest.fixture(scope="module")
def sd():
    from oracle import model as omodel
    return omodel.init_state_dict(0)


def head_major(wk, wv, bk, bv):
    """[Wk_h; Wv_h] of every head, 128 rows each (the layout etude_k_cross_attn takes)."""
    w = torch.cat([torch.cat([wk[64 * h:64 * h + 64], wv[64 * h:64 * h + 64]]) for h in range(4)]).contiguous()
    b = torch.cat([torch.cat([bk[64 * h:64 * h + 64], bv[64 * h:64 * h + 64]]) for h in range(4)]).contiguous()
    return w, b


def fused(x, w_hm, b_hm, q, q_stride, n_frames):
    out = torch.full((n_frames * 88, 256), float("nan"), dtype=torch.bfloat16, device="cuda")
    _lib.check(_lib.load().etude_k_cross_attn(P(x), P(w_hm), P(b_hm), P(q), q.shape[0], q_stride, n_frames, P(out), stream()),
               "etude_k_cross_attn")
    torch.cuda.synchronize()
    return out


def two_kernel(x, wkv, bkv, q, q_stride, n_frames):
    """The replaced path: gemm_bstat writes K|V [tokens, 512] (K then V), attention4 reads it back.  Returns (out, kv)."""
    lib = _lib.load()
    kv = torch.empty((n_frames * 256, 512), dtype=torch.bfloat16, device="cuda")
    _lib.check(lib.etude_k_gemm(P(x), P(wkv), P(bkv), n_frames * 256, 512, 256, 0, P(kv), None, 0, None, None, None, stream()), "etude_k_gemm")
    out = torch.full((n_frames * 88, 256), float("nan"), dtype=torch.bfloat16, device="cuda")
    _lib.check(lib.etude_k_attention(P(q), q.shape[0], 256, 0, q_stride, P(kv), 512, 0, 256, n_frames, 88, 256, P(out), None, stream()),
               "etude_k_attention")
    torch.cuda.synchronize()
    return out, kv


def layer_inputs(sd, layer, n_frames, seed, wscale=1.0):
    """Encoder output rows (unit variance, like the LayerNorm output), the layer's K|V weights and its queries as forward_impl
    feeds them: layer 0 the shared q0 table (128 rows, 88 valid), layers 1-2 88 rows per frame."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    pre = LAYERS[layer]
    x = bf(torch.randn(n_frames * 256, 256, generator=g, device="cuda"))
    wk, wv = sd[f"{pre}.fc_k.weight"].cuda() * wscale, sd[f"{pre}.fc_v.weight"].cuda() * wscale
    bk, bv = sd[f"{pre}.fc_k.bias"].cuda(), sd[f"{pre}.fc_v.bias"].cuda()
    wq, bq = sd[f"{pre}.fc_q.weight"].cuda() * wscale, sd[f"{pre}.fc_q.bias"].cuda()
    if layer == 0:
        q = bf(sd["decoder.pos_embedding_freq.weight"].cuda() @ wq.T + bq)
        q, stride = torch.cat([q, torch.zeros(40, 256, dtype=torch.bfloat16, device="cuda")]).contiguous(), 0
    else:
        q, stride = bf(bf(torch.randn(n_frames * 88, 256, generator=g, device="cuda")).float() @ wq.T + bq), 88
    return x, bf(torch.cat([wk, wv])).contiguous(), torch.cat([bk, bv]).float().contiguous(), q, stride


@pytest.mark.parametrize("n_frames", N_FRAMES)
@pytest.mark.parametrize("layer", [0, 1, 2])
def test_cross_attn_vs_two_kernel_path_and_fp64(sd, layer, n_frames):
    """Fused against (a) the gemm_bstat + attention4 path on the same seeded checkpoint weights, reported as the maximum
    difference, and (b) fp64 attention over the K|V that gemm_bstat rounds, within test_decoder_kernels_gpu.attention_bound.
    The fused projection has the same rounding point (fp32 accumulation of the 256 products, + fp32 bias, one bf16 rounding),
    so its K|V can differ from gemm_bstat's only where the two tensor-core accumulation orders round apart; the bound is
    therefore widened by the effect of one bf16 unit on every K and V element: |dS| <= u sum_d |q_d k_d| on the scores
    (scale 1/8 and the softmax's Lipschitz factor 2 in max-norm) and u |v| on the values:
        err <= bound + u (max_k |v| + 2 / 8 max_k sum_d |q_d k_d| max_k |v|)."""
    x, wkv, bkv, q, stride = layer_inputs(sd, layer, n_frames, seed=100 * layer + n_frames)
    w_hm, b_hm = head_major(wkv[:256], wkv[256:], bkv[:256], bkv[256:])
    got = fused(x, w_hm, b_hm, q, stride, n_frames)
    ref, kv = two_kernel(x, wkv, bkv, q, stride, n_frames)
    diff = (got.float() - ref.float()).abs()
    diff = torch.where(torch.isnan(diff), torch.full_like(diff, float("inf")), diff)
    n_diff = int((got.view(torch.int16) != ref.view(torch.int16)).sum())
    worst = 0.0
    slab = 1024
    for f0 in range(0, n_frames, slab):
        f1 = min(n_frames, f0 + slab)
        n = f1 - f0
        qv = (q[:88].reshape(1, 88, 4, 64).expand(n, 88, 4, 64) if stride == 0 else q[f0 * 88:f1 * 88].reshape(n, 88, 4, 64))
        kk = kv[f0 * 256:f1 * 256, :256].reshape(n, 256, 4, 64)
        vv = kv[f0 * 256:f1 * 256, 256:].reshape(n, 256, 4, 64)
        o, bound, _, _, _ = attention_bound(qv, kk, vv)
        qk = torch.einsum("sqhd,skhd->shqk", qv.double().abs(), kk.double().abs()).amax(-1)          # [s, h, q]
        vmax = vv.double().abs().amax(1)                                                             # [s, h, 64]
        extra = 2.0 ** -8 * (vmax.unsqueeze(1) * (1 + 2.0 / 8.0 * qk.permute(0, 2, 1).unsqueeze(-1)))  # [s, q, h, 64]
        err = (got[f0 * 88:f1 * 88].view(n, 88, 4, 64).double() - o).abs()
        err = torch.where(torch.isnan(err), torch.full_like(err, float("inf")), err)
        worst = max(worst, (err / (bound + extra)).max().item())
    report(f"cross_attn layer={layer} n_frames={n_frames}", max_diff_vs_two_kernel=diff.max().item(), elems_differing=n_diff,
           err_over_bound=worst)
    assert worst <= 1.0, worst


@pytest.mark.parametrize("n_frames", [1, 37, 300])
@pytest.mark.parametrize("q_shared", [False, True])
def test_cross_attn_exact_routing(n_frames, q_shared):
    """Weights that select channel slices with zero bias make K_h and V_h exact slices of x (one product
    per output, fp32-exact), so the r6a routing probe applies: every key of a frame gets a distinct base-8 code, a query's
    score is exactly 0 on its target key and <= -1024 on every other, P is exactly one-hot and each output row must equal the
    target key's V row bit for bit.  K_h dims 0-4 read channels 0-4 (the code), dims 5-63 zero channels; V of head h reads channels 128 + (32 h + d) mod 128 (random bf16 values).  The targets
    include the first and last key of both 128-key blocks; with q_shared one query table (and one code order) serves every frame."""
    g = torch.Generator().manual_seed(7 + n_frames + 100 * q_shared)
    x = torch.zeros(n_frames * 256, 256, dtype=torch.float64)
    perms = [torch.randperm(512, generator=g)[:256] for _ in range(1 if q_shared else n_frames)]
    codes = torch.stack(perms * n_frames if q_shared else perms)                                          # [F, 256] distinct
    x[:, 128:] = torch.randn(n_frames * 256, 128, generator=g).to(torch.bfloat16).double()
    kvec = _key_vec(codes.reshape(-1))                                                                   # [F*256, 64]
    x[:, :5] = kvec[:, :5]
    w = torch.zeros(512, 256, dtype=torch.float64)
    vcols = []
    for h in range(4):
        for d in range(5):
            w[128 * h + d, d] = 1.0                    # K_h dims 0-4: the code; dims 5-63 read zero channels
        cols = [128 + (32 * h + d) % 128 for d in range(64)]
        vcols.append(cols)
        for d in range(64):
            w[128 * h + 64 + d, cols[d]] = 1.0
    nq = 1 if q_shared else n_frames
    tg = torch.randint(0, 256, (nq, 4, 88), generator=g)
    edge = torch.tensor([0, 127, 128, 255])
    tg[:, :, :4] = edge
    q = torch.zeros(nq * 88 if not q_shared else 128, 256, dtype=torch.float64)
    for f in range(nq):
        for h in range(4):
            q[f * 88:f * 88 + 88, 64 * h:64 * h + 64] = _query_vec(codes[f, tg[f, h]])
    xd, wd = bf(x).cuda(), bf(w).cuda()
    qd = bf(q).cuda()
    got = fused(xd, wd, torch.zeros(512, device="cuda"), qd, 0 if q_shared else 88, n_frames)
    exp = torch.empty(n_frames * 88, 256, dtype=torch.bfloat16)
    xb = bf(x)
    for f in range(n_frames):
        tf = tg[0 if q_shared else f]
        for h in range(4):
            exp[f * 88:f * 88 + 88, 64 * h:64 * h + 64] = xb[f * 256 + tf[h]][:, vcols[h]]
    mism = int((got.view(torch.int16) != exp.cuda().view(torch.int16)).sum())
    report(f"cross_attn_exact_routing n_frames={n_frames} q_shared={q_shared}", mismatches=mism)
    assert mism == 0


def test_workspace_shrinks_by_the_cross_kv(sd):
    """With the K|V projected inside the attention kernel the workspace keeps only layer 2's K|V (512 columns, for the
    attention-probabilities output) and no encoder Q|K|V buffer: per 512-frame window 256 * 512 * 2 * (1536 + 768 - 512)
    bytes = 0.47 GB less than before (15 GB at 32 windows)."""
    from test_decoder_kernels_gpu import _engine
    eng = _engine(sd, 512)
    try:
        b32 = int(eng.lib.etude_workspace_bytes(eng._h, 32))
    finally:
        eng.close()
    NT, ND = 512 * 256, 512 * 88
    dec = ND * 2 * (256 + 768 + 256 + 256 + 256)
    old = 32 * (NT * 2 * (256 + 768 + 256 + 1536) + dec) + 1024
    new = 32 * (NT * 2 * (256 + 256 + 512) + dec) + 1024
    report("cross_attn_workspace", bytes_32_windows=b32, before=old, saved=old - b32)
    assert b32 == new, (b32, new)
