"""Decoder-side kernels in the configurations forward_impl launches (etude_b200/csrc/api.cu), each against a plain torch
fp64 reference fed the same bf16 operands, with elementwise tolerances derived from the kernel's rounding points, plus exact
probes whose answer is known bit for bit.

Rounding units used below: u = 2^-8 (bf16 round to nearest, 8-bit significand), 2^-24 (fp32 round to nearest).  Tensor-core accumulation
over K products is bounded as K * 2^-23 * sum |a_k b_k| (one unit of 2^-23 per addition allows for truncating adders)."""
import ctypes

import pytest
import torch

pytestmark = pytest.mark.gpu

import gpu_diag as D  # noqa: E402  (tests/ is on sys.path via conftest)
from conftest import report  # noqa: E402
from etude_b200 import _lib  # noqa: E402

P, stream = D.P, D.stream
U_BF16 = 2.0 ** -8
LOG2E = 1.4426950408889634
SCALE = LOG2E / 8.0          # the kernels' score scale in the log2 domain (1 / sqrt(64) * log2(e))
bf = lambda t: t.to(torch.bfloat16)


def gamma_mma(k):
    return k * 2.0 ** -23


@pytest.fixture(scope="module")
def sd():
    from oracle import model as omodel
    return omodel.init_state_dict(0)


def _engine(sd, n_frame, max_windows=1):
    from etude_b200.engine import Engine
    from etude_b200.weights import pack_state_dict
    s = dict(sd)
    s["decoder.pos_embedding_time.weight"] = s["decoder.pos_embedding_time.weight"][:n_frame].clone()
    blob, _ = pack_state_dict(s, strict=True, n_frame=n_frame)
    return Engine(blob, torch.device("cuda", torch.cuda.current_device()), max_windows=max_windows)


@pytest.fixture(scope="module")
def engines(sd):
    e = {512: _engine(sd, 512), 128: _engine(sd, 128)}
    yield e
    for x in e.values():
        x.close()


# ============================================================================================================ attention
# (name, q_ld, q_seq_stride (None: = Lq), q table rows (None: n_seq * Lq), kv_ld, k_col0, v_col0, Lq, Lk, production n_seq)
ATTN_CASES = {
    "dec_layer0_cross": (256, 0, 128, 1536, 0, 256, 88, 256, 1024),
    "dec_self": (768, None, None, 768, 256, 512, 88, 88, 1024),
    "dec_cross_l1": (256, None, None, 1536, 512, 768, 88, 256, 1024),
    "dec_cross_l2": (256, None, None, 1536, 1024, 1280, 88, 256, 1024),
    "time_512": (768, None, None, 768, 256, 512, 512, 512, 176),
    "time_128": (768, None, None, 768, 256, 512, 128, 128, 176),
}
# (case, kernel): attention4 for every launch of forward_impl; attention2 (+ probabilities) for the 9-tuple's layer-2 cross
ATTN_RUNS = [(c, 4) for c in ATTN_CASES] + [("dec_cross_l2", 2)]
N_SEQS = ["1", "2", "37", "38", "prod"]   # 4 * 37 = 148 work items = one per SM


def _n_seq(case, tag):
    return ATTN_CASES[case][8] if tag == "prod" else int(tag)


def _buffers(case, n_seq, fill):
    """Q and K|V buffers laid out like forward_impl's: returns (q_buf, kv_buf, shared) where shared = Q and K|V are one buffer."""
    q_ld, stride, q_rows, kv_ld, k0, v0, Lq, Lk, _ = ATTN_CASES[case]
    shared = q_ld == 768
    kv = fill(n_seq * Lk, kv_ld)
    q = kv if shared else fill(q_rows if q_rows else n_seq * Lq, q_ld)
    return q, kv, shared


def _launch(case, q, kv, n_seq, kernel, out=None):
    q_ld, stride, q_rows, kv_ld, k0, v0, Lq, Lk, _ = ATTN_CASES[case]
    lib = _lib.load()
    out = torch.full((n_seq * Lq, 256), float("nan"), dtype=torch.bfloat16, device="cuda") if out is None else out
    probs = torch.full((n_seq, 4, Lq, Lk), float("nan"), device="cuda") if kernel == 2 else None
    _lib.check(lib.etude_k_attention(P(q), q.shape[0], q_ld, 0, Lq if stride is None else stride, P(kv), kv_ld, k0, v0, n_seq, Lq, Lk,
                                     P(out), P(probs), stream()), "etude_k_attention")
    torch.cuda.synchronize()
    return out, probs


def _qkv_views(case, q, kv, n_seq):
    """[S, L, 4, 64] views of Q, K, V as the kernel reads them (the layer-0 table broadcast over sequences)."""
    q_ld, stride, q_rows, kv_ld, k0, v0, Lq, Lk, _ = ATTN_CASES[case]
    if stride == 0:
        qv = q[:Lq].reshape(1, Lq, 4, 64).expand(n_seq, Lq, 4, 64)
    else:
        qv = q[: n_seq * Lq, :256].reshape(n_seq, Lq, 4, 64)
    kk = kv[:, k0:k0 + 256].reshape(n_seq, Lk, 4, 64)
    vv = kv[:, v0:v0 + 256].reshape(n_seq, Lk, 4, 64)
    return qv, kk, vv


# ---------------------------------------------------------------------------------------------------- exact routing probe
def _key_vec(code):
    a, b, c = (code >> 6).double(), ((code >> 3) & 7).double(), (code & 7).double()
    v = torch.zeros(code.shape + (64,), dtype=torch.float64)
    v[..., 0], v[..., 1], v[..., 2], v[..., 3], v[..., 4] = a, b, c, a * a + b * b + c * c, 1.0
    return v


def _query_vec(code):
    a, b, c = (code >> 6).double(), ((code >> 3) & 7).double(), (code & 7).double()
    v = torch.zeros(code.shape + (64,), dtype=torch.float64)
    v[..., 0], v[..., 1], v[..., 2], v[..., 3], v[..., 4] = 2048 * a, 2048 * b, 2048 * c, -1024.0, -1024 * (a * a + b * b + c * c)
    return v


def _boundary_keys(Lk):
    return sorted({0, Lk - 1} | {x for j in range(1, (Lk + 127) // 128) for x in (128 * j - 1, 128 * j)})


def _probe(case, n_seq, seed):
    """Q / K codes in base 8 (code = 64a + 8b + c) with q.k = -1024 ((a-A)^2 + (b-B)^2 + (c-C)^2): exactly 0 for the target key,
    <= -1024 for every other key.  Every term is a bf16-exact integer and every fp32 partial sum is an exact multiple of 1024,
    so the scores are exact; ex2.approx.ftz of <= -1024 * log2(e) / 8 < -126 is 0, and so is pow2_int of a block reference
    that far below, so P is exactly one-hot and the output row must be the target V row bit for bit (the drain multiplies by
    1 / l = 1 - 2^-24 at worst, which rounds back to the same bf16 value).  Returns (q, kv, expected out, targets)."""
    q_ld, stride, q_rows, kv_ld, k0, v0, Lq, Lk, _ = ATTN_CASES[case]
    g = torch.Generator().manual_seed(seed)
    H = 4
    # targets: a per-(sequence, head) choice of distinct keys that always includes the first and last key of every KV block,
    # spread over random query rows (Lq == Lk: a permutation, so every query tile has targets)
    r = torch.rand(n_seq, H, Lk, generator=g)
    r[..., _boundary_keys(Lk)] -= 2.0
    tp = r.argsort(-1)                                    # boundary keys first
    qperm = torch.rand(n_seq, H, Lq, generator=g).argsort(-1)
    targets = tp[..., :Lq].gather(-1, qperm)              # [S, H, Lq]
    if stride == 0:
        # layer 0: one Q table for every sequence, so the key codes vary per sequence instead
        qcodes = torch.rand(1, H, 512, generator=g).argsort(-1)[..., :Lq].expand(n_seq, H, Lq)
    elif Lk == 88:
        # every sequence uses the same 88 codes, so each key of sequence s + 1 (and each zero-filled key past the last sequence,
        # which scores exactly 0) ties with the target of some query row of sequence s if the 96-key tile's mask leaks it
        c88 = torch.randperm(512, generator=g)[:88]
        qcodes = c88[torch.rand(n_seq, H, 88, generator=g).argsort(-1)]
    else:
        qcodes = torch.rand(n_seq, H, 512, generator=g).argsort(-1)[..., :Lq]
    # key codes: kc[tp[k]] = codeset[k], with codeset[qperm[i]] = qcodes[i] so that kc[targets[i]] = qcodes[i]
    codeset = torch.empty(n_seq, H, Lk, dtype=torch.int64)
    codeset[..., :Lq] = qcodes.gather(-1, qperm.argsort(-1))
    if Lk > Lq:
        used = torch.zeros(n_seq, H, 512).scatter_(-1, qcodes.contiguous(), 1.0)
        codeset[..., Lq:] = (torch.rand(n_seq, H, 512, generator=g) + 2.0 * used).argsort(-1)[..., :Lk - Lq]
    kc = torch.empty_like(codeset).scatter_(-1, tp, codeset)
    assert torch.equal(kc.gather(-1, targets), qcodes)
    # V rows: codes of (sequence, key, head) in the first three columns of each head, random bf16 elsewhere
    v = torch.randn(n_seq, Lk, H, 64, generator=g, dtype=torch.float64)
    v[..., 0] = (torch.arange(n_seq) % 256)[:, None, None]
    v[..., 1] = (torch.arange(Lk) % 256)[None, :, None]
    v[..., 2] = (torch.arange(Lk) // 256)[None, :, None] + 4 * torch.arange(H)[None, None, :]
    noise = lambda rows, cols: torch.randn(rows, cols, generator=g, dtype=torch.float64)   # unused columns: noise
    q, kv, shared = _buffers(case, n_seq, noise)
    kv[:, k0:k0 + 256] = _key_vec(kc).permute(0, 2, 1, 3).reshape(n_seq * Lk, 256)
    kv[:, v0:v0 + 256] = v.reshape(n_seq * Lk, 256)
    qv = _query_vec(qcodes).permute(0, 2, 1, 3)             # [S, Lq, H, 64]
    if stride == 0:
        q[:Lq] = qv[0].reshape(Lq, 256)
    else:
        q[:, :256] = qv.reshape(n_seq * Lq, 256)
    expect = v.permute(0, 2, 1, 3).gather(2, targets[..., None].expand(n_seq, H, Lq, 64)).permute(0, 2, 1, 3).reshape(n_seq * Lq, 256)
    dev = lambda t: bf(t).cuda()
    kv_d = dev(kv)
    q_d = kv_d if shared else dev(q)
    return q_d, kv_d, dev(expect), targets.cuda()


@pytest.mark.parametrize("tag", N_SEQS)
@pytest.mark.parametrize("case,kernel", ATTN_RUNS, ids=[f"{c}-attention{k}" for c, k in ATTN_RUNS])
def test_attention_exact_routing(case, kernel, tag):
    """Every query row scores 0 against one target key and <= -1024 against all others (see _probe): the output must be the
    target V row bit for bit, and attention2's probabilities exactly one-hot.  Targets cover the first and last key of every
    KV block and every query tile; for Lk = 88 every key of the next sequence and every zero-filled key past the last one
    would tie with some row's target if the 96-key tile's mask let it in."""
    n_seq = _n_seq(case, tag)
    q, kv, expect, targets = _probe(case, n_seq, seed=1000 + n_seq)
    out, probs = _launch(case, q, kv, n_seq, kernel)
    Lq, Lk = ATTN_CASES[case][6], ATTN_CASES[case][7]
    bad = (out.view(torch.int16) != expect.view(torch.int16)).view(n_seq, Lq, 4, 64).any(-1)
    n_bad = int(bad.sum())
    if probs is not None:
        one_hot = torch.zeros_like(probs).scatter_(-1, targets[..., None], 1.0)
        n_bad_p = int((probs != one_hot).any(-1).sum())
    else:
        n_bad_p = 0
    report(f"decoder_attention_exact_routing {case} attention{kernel} n_seq={n_seq}", wrong_rows=n_bad, wrong_prob_rows=n_bad_p)
    assert n_bad == 0, f"{n_bad} (row, head) outputs differ; first (seq, row, head): {bad.nonzero()[:5].tolist()}"
    assert n_bad_p == 0


# ---------------------------------------------------------------------------------------------------- realistic inputs
def _projection(sd, prefix, parts):
    w = torch.cat([sd[f"{prefix}.{p}.weight"] for p in parts])
    b = torch.cat([sd[f"{prefix}.{p}.bias"] for p in parts])
    return w.cuda(), b.cuda()


def _realistic(case, n_seq, sd, wscale, seed):
    """Q, K, V the way the model makes them: bf16(bf16(x) W^T + b) with the seeded checkpoint's weights (times wscale) and
    unit-variance rows x (LayerNorm outputs); the time axis feeds x = bf16(16 z + pos_embedding_time) like the transpose."""
    q_ld, stride, q_rows, kv_ld, k0, v0, Lq, Lk, _ = ATTN_CASES[case]
    g = torch.Generator(device="cuda").manual_seed(seed)
    rnd = lambda rows: torch.randn(rows, 256, generator=g, device="cuda")
    proj = lambda x, w, b: bf(bf(x).float() @ (w * wscale).T + b)
    if case.startswith("time"):
        pos = sd["decoder.pos_embedding_time.weight"][:Lq].cuda()
        x = (16 * rnd(n_seq * Lq).view(n_seq, Lq, 256) + pos).view(-1, 256)
        qkv = proj(x, *_projection(sd, "decoder.layers_time.0.self_attention", ("fc_q", "fc_k", "fc_v")))
        return qkv, qkv
    if case == "dec_self":
        qkv = proj(rnd(n_seq * 88), *_projection(sd, "decoder.layers_freq.0.self_attention", ("fc_q", "fc_k", "fc_v")))
        return qkv, qkv
    enc = rnd(n_seq * 256)
    kv = torch.cat([proj(enc, *_projection(sd, p, ("fc_k", "fc_v"))) for p in
                    ("decoder.layer_zero_freq.encoder_attention", "decoder.layers_freq.0.encoder_attention",
                     "decoder.layers_freq.1.encoder_attention")], 1).contiguous()
    if case == "dec_layer0_cross":
        q = proj(sd["decoder.pos_embedding_freq.weight"].cuda(), *_projection(sd, "decoder.layer_zero_freq.encoder_attention", ("fc_q",)))
        return torch.cat([q, torch.zeros(128 - 88, 256, dtype=torch.bfloat16, device="cuda")]).contiguous(), kv
    layer = "0" if case == "dec_cross_l1" else "1"
    q = proj(rnd(n_seq * 88), *_projection(sd, f"decoder.layers_freq.{layer}.encoder_attention", ("fc_q",)))
    return q, kv


def attention_bound(q, k, v):
    """fp64 reference and elementwise error bound of the kernel's output (and of attention2's fp32 probabilities).
    Per key j of a row: the fp32 score carries at most 64 * 2^-23 * sum_d |q_d k_jd| (tensor-core accumulation), and the
    exponent argument s * scale - m picks up the scale's and the FMA's roundings, 2^-23 |s * scale|, and ex2.approx its
    2^-22: exponent error d_j = scale 64 2^-23 sum|q k| + 2^-23 |s scale| + 2^-22, so e_j is off by a factor within
    [2^-d_j, 2^d_j].  l sums the unrounded e: p_j = e_j / l is off by at most p_j (Dup_j + Dup) / (1 - Dlo) with
    Dup_j = 2^d_j - 1, Dup = sum p Dup, Dlo = sum p (1 - 2^-d).  P = bf16(e) adds u = 2^-8 per key, P V accumulates Lk
    products (Lk 2^-23), 1 / l is good to 2^-23, ftz / pow2_int underflow drops at most Lk 2^-126 of weight, and the output
    is rounded to bf16 once more:
        err <= (1 + u) A + u |o|,  A = sum_j |v_j| (p_j (u + (Lk + 1) 2^-23) + dp_j) + Lk 2^-125 max|v|.
    Probabilities (fp32, not rounded to bf16): |dp_j| <= p_j (Dup_j + Dup) / (1 - Dlo) + p_j 2^-22 + 2^-126."""
    q, k, v = q.double(), k.double(), v.double()
    s = torch.einsum("sqhd,skhd->shqk", q, k)
    sabs = torch.einsum("sqhd,skhd->shqk", q.abs(), k.abs())
    p = torch.softmax(s / 8.0, dim=-1)
    Lk = k.shape[1]
    d = SCALE * gamma_mma(64) * sabs + 2.0 ** -23 * (s * SCALE).abs() + 2.0 ** -22
    Dup, Dlo = torch.exp2(d) - 1, 1 - torch.exp2(-d)
    dp = p * (Dup + (p * Dup).sum(-1, keepdim=True)) / (1 - (p * Dlo).sum(-1, keepdim=True))
    o = torch.einsum("shqk,skhd->sqhd", p, v)
    A = torch.einsum("shqk,skhd->sqhd", p * (U_BF16 + (Lk + 1) * 2.0 ** -23) + dp, v.abs()) + Lk * 2.0 ** -125 * v.abs().amax(1, keepdim=True)
    bound = (1 + U_BF16) * A + U_BF16 * o.abs()
    pbound = dp + p * 2.0 ** -22 + 2.0 ** -126
    return o, bound, p, pbound, (s * SCALE).abs().amax().item()


@pytest.mark.parametrize("wscale", [1.0, 4.0])
@pytest.mark.parametrize("tag", N_SEQS)
@pytest.mark.parametrize("case,kernel", ATTN_RUNS, ids=[f"{c}-attention{k}" for c, k in ATTN_RUNS])
def test_attention_realistic_vs_fp64(case, kernel, tag, wscale, sd):
    """Model-built Q / K / V (checkpoint weights, x4 for near one-hot rows) against fp64 within attention_bound, every row."""
    n_seq = _n_seq(case, tag)
    q, kv = _realistic(case, n_seq, sd, wscale, seed=int(2000 + n_seq + 10 * wscale))
    out, probs = _launch(case, q, kv, n_seq, kernel)
    qv, kk, vv = _qkv_views(case, q, kv, n_seq)
    Lq, Lk = ATTN_CASES[case][6], ATTN_CASES[case][7]
    got = out.view(n_seq, Lq, 4, 64)
    worst, worst_p, regime, err_max = 0.0, 0.0, 0.0, 0.0
    slab = max(1, (1 << 22) // (Lq * Lk))
    for s0 in range(0, n_seq, slab):
        s1 = min(n_seq, s0 + slab)
        o, bound, p, pbound, reg = attention_bound(qv[s0:s1], kk[s0:s1], vv[s0:s1])
        err = (got[s0:s1].double() - o).abs()
        err = torch.where(torch.isnan(err), torch.full_like(err, float("inf")), err)
        worst = max(worst, (err / bound).max().item())
        err_max = max(err_max, err.max().item())
        regime = max(regime, reg)
        if probs is not None:
            ep = (probs[s0:s1].double() - p).abs()
            ep = torch.where(torch.isnan(ep), torch.full_like(ep, float("inf")), ep)
            worst_p = max(worst_p, (ep / pbound).max().item())
    report(f"decoder_attention_vs_fp64 {case} attention{kernel} n_seq={n_seq} wscale={wscale:g}", err_over_bound=worst,
           probs_err_over_bound=worst_p, out_maxabs=err_max, max_abs_score_log2=regime)
    assert worst <= 1.0, worst
    assert worst_p <= 1.0, worst_p


# ============================================================================================================ heads
def _heads_weights(sd, dom, ties=None):
    w = torch.zeros(144, 256)
    b = torch.zeros(144)
    for i, n in enumerate(("onset", "offset", "mpe")):
        w[i] = sd[f"decoder.fc_{n}_{dom}.weight"][0]
        b[i] = sd[f"decoder.fc_{n}_{dom}.bias"][0]
    w[3:131] = sd[f"decoder.fc_velocity_{dom}.weight"]
    b[3:131] = sd[f"decoder.fc_velocity_{dom}.bias"]
    w *= 3.0    # logits of a few units, like a trained model's heads
    if ties == "pair":        # velocity columns 5 and 70 identical and ahead of all others
        w[3 + 70] = w[3 + 5]
        b[3 + 5] = b[3 + 70] = 20.0
    elif ties == "all":       # all 128 velocity columns identical
        w[3:131] = w[3]
        b[3:131] = b[3]
    return bf(w).cuda(), b.float().cuda()


def _run_heads(eng, x, w, b, nw, time_major, out_row, keep, n_rows, with_logits):
    lib = eng.lib
    rolls = [torch.full((n_rows, 88), float("nan"), device="cuda") for _ in range(3)] + \
            [torch.full((n_rows, 88), -1, dtype=torch.int8, device="cuda")]
    logits = torch.full((x.shape[0], 128), float("nan"), device="cuda") if with_logits else None
    arr = (ctypes.c_void_p * 4)(*[t.data_ptr() for t in rolls])
    _lib.check(lib.etude_k_heads(eng._h, P(x), P(w), P(b), nw, int(time_major), _lib.i64_array(out_row), keep[0], keep[1], arr,
                                 P(logits), stream()), "etude_k_heads")
    torch.cuda.synchronize()
    return rolls, logits


HEADS_CASES = [(512, nw, tm, (0, 512)) for nw in (1, 3) for tm in (0, 1)] + [(512, 2, 1, (128, 256))] + \
              [(128, nw, tm, (0, 128)) for nw in (1, 5) for tm in (0, 1)] + [(128, 6, 1, (off, 64)) for off in (0, 32, 64)] + \
              [(128, 3, 0, (32, 64))]


@pytest.mark.parametrize("ties", [None, "pair", "all"])
@pytest.mark.parametrize("F,nw,time_major,keep", HEADS_CASES)
def test_heads_epilogue_vs_fp64(engines, sd, F, nw, time_major, keep, ties):
    """EPI_HEADS against fp64 logits of the same bf16 x / W.  Logit bound per element: 256 2^-23 (|x| |W|^T + |b|) (tensor
    core over K = 256, then the fp32 bias add).  Sigmoid bound: s (1 - s) d_logit + 2^-21 (expf and the IEEE division).  The
    velocity argmax must equal the fp64 argmax wherever the top two fp64 logits are further apart than their two bounds, and
    must equal torch.argmax (first maximum) of the kernel's own logits everywhere -- exact ties from duplicated W rows
    included, where it must hold the lower index.  Only rows out_row[w] + f - keep0 for kept frames f may change; the
    sentinel (NaN / -1) of every other row must survive.  With and without the logits output the rolls are identical."""
    eng = engines[F]
    g = torch.Generator(device="cuda").manual_seed(F + 7 * nw + 3 * time_major + keep[0])
    M = nw * F * 88
    x = bf(torch.randn(M, 256, generator=g, device="cuda"))
    w, b = _heads_weights(sd, "time" if time_major else "freq", ties)
    # window slots in a shuffled, far-apart order with gaps between them
    slot = keep[1] + 37
    order = torch.randperm(nw, generator=torch.Generator().manual_seed(nw)).tolist()
    out_row = [1000 + 3 * slot * order[i] for i in range(nw)]
    n_rows = max(out_row) + slot + 50
    rolls, logits = _run_heads(eng, x, w, b, nw, time_major, out_row, keep, n_rows, True)
    rolls_nl, _ = _run_heads(eng, x, w, b, nw, time_major, out_row, keep, n_rows, False)
    for a, c in zip(rolls, rolls_nl):
        assert torch.equal(a.view(torch.uint8) if a.dtype != torch.int8 else a, c.view(torch.uint8) if c.dtype != torch.int8 else c)
    # fp64 reference over the input rows, mapped to (w, f, n)
    ref = x.double() @ w.double().T + b.double()
    eb = gamma_mma(256) * (x.double().abs() @ w.double().abs().T + b.double().abs())
    r = torch.arange(M, device="cuda")
    if time_major:
        f, n, wi = r % F, (r // F) % 88, r // (F * 88)
    else:
        n, f, wi = r % 88, (r // 88) % F, r // (88 * F)
    logit_row = (wi * F + f) * 88 + n
    # velocity logits: every frame, (window, frame, note) order
    got_l = torch.empty(M, 128, dtype=torch.float64, device="cuda")
    got_l[r] = logits[logit_row].double()
    worst_l = ((got_l - ref[:, 3:131]).abs() / eb[:, 3:131]).max().item()
    assert not torch.isnan(logits).any()
    # rolls
    kept = (f >= keep[0]) & (f < keep[0] + keep[1])
    rows = torch.tensor(out_row, device="cuda")[wi] + f - keep[0]
    idx = (rows * 88 + n)[kept]
    touched = torch.zeros(n_rows * 88, dtype=torch.bool, device="cuda")
    touched[idx] = True
    assert int(touched.sum()) == int(kept.sum()), "two kept rows map to one roll element"
    worst_s = 0.0
    for i in range(3):
        flat = rolls[i].view(-1)
        assert torch.isnan(flat[~touched]).all(), f"roll {i}: a row outside the kept frames was written"
        sig = torch.sigmoid(ref[kept, i])
        bound = sig * (1 - sig) * eb[kept, i] + 2.0 ** -21
        es = (flat[idx].double() - sig).abs()
        es = torch.where(torch.isnan(es), torch.full_like(es, float("inf")), es)   # a kept element left at its NaN sentinel
        worst_s = max(worst_s, (es / bound).max().item())
    vel = rolls[3].view(-1)
    assert (vel[~touched] == -1).all(), "velocity roll: a row outside the kept frames was written"
    got_v = vel[idx].long()
    own = got_l.argmax(1)[kept]                        # first maximum of the kernel's own logits
    n_own = int((got_v != own).sum())
    top2 = ref[kept, 3:131].topk(2, dim=1)
    decided = (top2.values[:, 0] - top2.values[:, 1]) > (eb[kept, 3:131].gather(1, top2.indices).sum(1))
    n_ref = int((got_v[decided] != top2.indices[decided, 0]).sum())
    if ties == "pair":
        assert (got_v == 5).all()
    elif ties == "all":
        assert (got_v == 0).all()
    report(f"heads_epilogue_vs_fp64 F={F} nw={nw} time_major={time_major} keep={keep} ties={ties}", logit_err_over_bound=worst_l,
           sigmoid_err_over_bound=worst_s, argmax_vs_own_logits_mismatch=n_own, argmax_vs_fp64_mismatch=n_ref,
           decided_rows=int(decided.sum()), kept_rows=int(kept.sum()))
    assert worst_l <= 1.0 and worst_s <= 1.0
    assert n_own == 0 and n_ref == 0


# ============================================================================================================ transpose
@pytest.mark.parametrize("F,nw", [(512, 1), (512, 3), (512, 64), (128, 1), (128, 5), (128, 256)])
def test_transpose_time_bit_exact(engines, sd, F, nw):
    """(window, frame, note) -> (window, note, frame), x 16 + pos_embedding_time[frame]: one bf16 rounding of an exact fp32
    value (x 16 is exact), so the result must equal torch's bit for bit -- which also pins the handle's pos_time table."""
    eng = engines[F]
    g = torch.Generator(device="cuda").manual_seed(F + nw)
    x = bf(torch.randn(nw * F * 88, 256, generator=g, device="cuda") * 3)
    out = torch.full_like(x, float("nan"))
    _lib.check(eng.lib.etude_k_transpose_time(eng._h, P(x), nw, P(out), stream()), "etude_k_transpose_time")
    torch.cuda.synchronize()
    pos = sd["decoder.pos_embedding_time.weight"][:F].cuda()
    ref = (x.view(nw, F, 88, 256).float() * 16 + pos[None, :, None]).to(torch.bfloat16).permute(0, 2, 1, 3).reshape(-1, 256)
    n_bad = int((out.view(torch.int16) != ref.view(torch.int16)).any(1).sum())
    report(f"transpose_time F={F} nw={nw}", wrong_rows=n_bad)
    assert n_bad == 0


# ============================================================================================================ projections
@pytest.mark.parametrize("M", [2 * 512 * 256, 2 * 512 * 88, 2 * 512 * 88 - 37])
@pytest.mark.parametrize("N", [1536, 768, 256])
def test_projection_gemm_vs_fp64(N, M):
    """The B-stationary K = 256 projection (kv_all N = 1536, Q|K|V N = 768, fc_q N = 256) at the token counts of two windows
    (encoder 2 * 512 * 256, decoder 2 * 512 * 88) and a ragged M.  Bound per element: E = 256 2^-23 (|a| |W|^T + |b|), then
    the bf16 output rounding: err <= E + 2^-8 (|ref| + E)."""
    g = torch.Generator(device="cuda").manual_seed(N + M)
    a = bf(torch.randn(M, 256, generator=g, device="cuda"))
    w = bf(torch.randn(N, 256, generator=g, device="cuda") / 16)
    b = 0.2 * torch.randn(N, generator=g, device="cuda")
    out, _ = _gemm0(a, w, b)
    worst = 0.0
    for r0 in range(0, M, 16384):
        r1 = min(M, r0 + 16384)
        ad = a[r0:r1].double()
        ref = ad @ w.double().T + b.double()
        E = gamma_mma(256) * (ad.abs() @ w.double().abs().T + b.double().abs())
        err = (out[r0:r1].double() - ref).abs()
        err = torch.where(torch.isnan(err), torch.full_like(err, float("inf")), err)
        worst = max(worst, (err / (E + U_BF16 * (ref.abs() + E))).max().item())
    report(f"projection_gemm_vs_fp64 M={M} N={N}", err_over_bound=worst)
    assert worst <= 1.0, worst


def _gemm0(a, w, b):
    lib = _lib.load()
    out = torch.full((a.shape[0], w.shape[0]), float("nan"), dtype=torch.bfloat16, device="cuda")
    _lib.check(lib.etude_k_gemm(P(a), P(w), P(b), a.shape[0], w.shape[0], 256, 0, P(out), None, 0, None, None, None, stream()),
               "etude_k_gemm")
    torch.cuda.synchronize()
    return out, None


# ============================================================================================================ chain3 LayerNorm edges
def _ln64(x, gamma, beta):
    mu = x.mean(-1, keepdim=True)
    var = ((x - mu) ** 2).mean(-1, keepdim=True)
    rstd = 1.0 / torch.sqrt(var + 1e-5)
    return (x - mu) * rstd * gamma + beta, rstd, mu


def _ln_bound(x, dx, gamma, rstd, mu):
    """Elementwise bound of fp32 LayerNorm(x + dx) - LayerNorm64(x) for an input error |dx|: the propagated input error
    |g| rstd (|dx_i| + mean|dx| + |xhat_i| max|dx| rstd), the fp32 statistics (256 2^-23 relative on rstd, the variance
    taken about a pivot inside the row), and the folded x * rstd + (-mean * rstd) whose two terms are each rounded at the
    magnitude |x| rstd (or |mean| rstd: 316 |mean| for a constant row): |g| 2^-22 (|x_i| + |mean|) rstd, plus 2^-22 |y|."""
    xhat = (x - mu) * rstd
    g = gamma.abs()
    prop = g * rstd * (dx + dx.mean(-1, keepdim=True) + xhat.abs() * dx.amax(-1, keepdim=True) * rstd)
    stat = g * xhat.abs() * gamma_mma(256)
    fold = g * 2.0 ** -22 * (x.abs() + mu.abs()) * rstd
    return prop + stat + fold


def _ffn_reference(yk, y, by, w1, b1, w2, b2, gamma, beta):
    """fp64 reference and elementwise bound of the FFN half of chain3, LN(y + relu(bf16(y) W1^T + b1) W2^T + b2), given the
    kernel's own bf16(y) `yk` (the FFN's input: the y-only launch writes the same values) and the fp64 first-LN output `y`
    with its bound `by` (the kernel adds its fp32 y, not bf16(y), to the FFN output).
    ReLU's input carries 256 2^-23 (|yk| |W1|^T + |b1|); ReLU and the rounding to bf16 are monotone, so the kernel's bf16(h)
    lies in [lo, hi] = [bf16(relu(pre - e)), bf16(relu(pre + e))] -- an interval of width 0 wherever both ends round alike.
    With the midpoint c and half-width r the second LN's input is y + b2 + c W2^T up to
        dx2 = by + r |W2|^T + 512 2^-23 (|hi| |W2|^T + |y| + |b2|) + 2^-23 (|y| + |b2|)
    (P V-style accumulation onto the y + b2 initial value, and its own add), and _ln_bound takes it through the LN."""
    d = lambda t: t.double()
    yk, w1, b1, w2, b2 = d(yk), d(w1), d(b1), d(w2), d(b2)
    pre = yk @ w1.T + b1
    e = gamma_mma(256) * (yk.abs() @ w1.abs().T + b1.abs())
    lo = d(bf(torch.relu(pre - e).float()))
    hi = d(bf(torch.relu(pre + e).float()))
    c, r = (lo + hi) / 2, (hi - lo) / 2
    z = c @ w2.T
    x2 = y + b2 + z
    dx2 = by + r @ w2.abs().T + gamma_mma(512) * (hi.abs() @ w2.abs().T + y.abs() + b2.abs()) + 2.0 ** -23 * (y.abs() + b2.abs())
    ref, rstd, mu = _ln64(x2, gamma, beta)
    bound = _ln_bound(x2, dx2, gamma, rstd, mu)
    # what a kernel that skipped the FFN, or dropped b2, would return: the bound must reject both
    wrong = {"skipped_ffn": _ln64(y, gamma, beta)[0], "dropped_b2": _ln64(y + z, gamma, beta)[0]}
    return ref, bound, wrong


@pytest.mark.parametrize("resid_mod", [0, 88])
@pytest.mark.parametrize("ffn", [False, True])
def test_chain_layernorm_edge_rows_vs_fp64(ffn, resid_mod):
    """chain3 (fc_o + residual + LN [+ FFN + residual + LN]) on rows built to stress the LayerNorm statistics, mixed with
    ordinary rows: (a) a constant first-LN input (ctx row 0, constant residual row): the fp64 answer of the first LN is beta,
    the kernel's eps and clamps must give it up to the folded -mean * rstd term (rstd = 316); (b) rows offset by 4096 relative
    to a spread of ~1 (pivot-shifted one-sweep statistics: a naive E[x^2] - mean^2 loses everything); (c) rows with three
    channels at x100 (outlier channels).  fp64 references on the same bf16 operands.  First LN (the y-only launch, run in both
    variants): the input error is the GEMM's 256 2^-23 sum|ctx Wo| plus 2^-23 (|acc| + |bo| + |resid|) for the two adds, then
    _ln_bound and the bf16 output.  FFN variant: _ffn_reference, fed the y-only launch's bf16(y), and the test asserts that
    its bound rejects a skipped FFN and a dropped b2 on these inputs (so it pins the FFN half, not just the LN)."""
    torch.manual_seed(31 + resid_mod + ffn)
    M = 88 * 64 if resid_mod else 128 * 45 + 17
    dev = "cuda"
    ctx = bf(torch.randn(M, 256, device=dev) * 0.7)
    wo = bf(torch.randn(256, 256, device=dev) / 16)
    w1 = bf(torch.randn(512, 256, device=dev) / 16)
    w2 = bf(torch.randn(256, 512, device=dev) / 22)
    bo, b1, b2 = (0.1 * torch.randn(n, device=dev) for n in (256, 512, 256))
    bo[:] = 0.375                               # a constant vector, so ctx row 0 + a constant residual row is constant
    gamma = 1 + 0.1 * torch.randn(256, device=dev)
    beta = 0.1 * torch.randn(256, device=dev)
    n_res = resid_mod if resid_mod else M
    resid = torch.randn(n_res, 256, device=dev)
    kinds = torch.arange(n_res, device=dev) % 8    # 0: constant, 1: offset, 2: outliers, else ordinary
    resid[kinds == 0] = 1.5
    resid[kinds == 1] = 4096.0
    out_ch = torch.tensor([3, 77, 200], device=dev)
    resid[(kinds == 2).nonzero()[:, :1], out_ch] = 100.0 * torch.tensor([1.0, -1.0, 0.5], device=dev)
    resid = bf(resid)
    rkind = kinds if not resid_mod else kinds[torch.arange(M, device=dev) % resid_mod]
    ctx[rkind == 0] = 0
    if resid_mod:
        resid_dev = resid.repeat(3, 1)[: resid_mod + 127].contiguous()
        r_full = resid[torch.arange(M, device=dev) % resid_mod]
    else:
        resid_dev = resid
        r_full = resid
    lib = _lib.load()

    def chain(with_ffn):
        out = torch.full((M, 256), float("nan"), dtype=torch.bfloat16, device=dev)
        f = (lambda t: P(t)) if with_ffn else (lambda t: None)
        _lib.check(lib.etude_k_chain(P(ctx), P(wo), P(bo), f(w1), f(b1), f(w2), f(b2), P(gamma), P(beta), P(resid_dev), resid_mod,
                                     resid_dev.shape[0], P(out), M, stream()), "etude_k_chain")
        torch.cuda.synchronize()
        return out

    yk = chain(False)
    d = lambda t: t.double()
    nan_inf = lambda t: torch.where(torch.isnan(t), torch.full_like(t, float("inf")), t)
    G, B = d(gamma), d(beta)
    acc = d(ctx) @ d(wo).T
    x1 = acc + d(bo) + d(r_full)
    dx1 = gamma_mma(256) * (d(ctx).abs() @ d(wo).abs().T) + 2.0 ** -23 * (acc.abs() + d(bo).abs() + d(r_full).abs())
    y, rstd1, mu1 = _ln64(x1, G, B)
    by = _ln_bound(x1, dx1, G, rstd1, mu1)
    if ffn:   # the FFN bound takes the first LN's bound `by` as given: hold the y-only launch to it here too
        assert (nan_inf((d(yk) - y).abs()) / (by + U_BF16 * (y.abs() + by))).max().item() <= 1.0
        out = chain(True)
        ref, bound, wrong = _ffn_reference(yk, y, by, w1, b1, w2, b2, G, B)
    else:
        out, ref, bound, wrong = yk, y, by, {}
    bound = bound + U_BF16 * (ref.abs() + bound)      # bf16 output
    ratio = nan_inf((d(out) - ref).abs()) / bound
    per_kind = {name: ratio[rkind == k].max().item() for k, name in ((0, "constant"), (1, "offset4096"), (2, "outliers"))}
    per_kind["ordinary"] = ratio[rkind >= 3].max().item()
    rejected = {f"{k}_err_over_bound": ((d(bf(v.float())) - ref).abs() / bound).max().item() for k, v in wrong.items()}
    const_err = (d(out[rkind == 0]) - B).abs().max().item() if not ffn else float("nan")   # the y-only answer there is beta
    report(f"chain3_layernorm_edges ffn={ffn} resid_mod={resid_mod} M={M}", **{f"err_over_bound_{k}": v for k, v in per_kind.items()},
           constant_rows_vs_beta_maxabs=const_err, **rejected)
    assert max(per_kind.values()) <= 1.0, per_kind
    assert all(v > 1.0 for v in rejected.values()), rejected


# ============================================================================================================ full batch
def _window_inputs(b, F, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    return torch.rand(b, 256, F + 64, generator=g, device="cuda") * 20 - 18


def test_full_batch_windows_match_single_runs():
    """The library's largest batch (64 windows: the decoder's Q|K|V buffer passes 2^31 elements, the encoder's x / ctx reach
    exactly 2^31 and the attention output passes 2^31 fp32 values) through Model_SPEC2MIDI.forward with every output
    requested: windows 0, 31 and 63 must equal the same windows run alone bit for bit, rolls A / B, velocity logits and
    attention alike."""
    ex, _ = D.make_extractor(max_windows=64)
    try:
        x = _window_inputs(64, 512, 77)
        outs = ex.model(x)
        keep = {w: [t[w].clone() for t in outs] for w in (0, 31, 63)}
        del outs
        torch.cuda.synchronize()
        for w, full in keep.items():
            one = ex.model(x[w:w + 1])
            for i in range(9):
                assert torch.equal(full[i], one[i][0]), (w, i)
            del one
        report("full_batch_64_windows_vs_single", windows_checked="0/31/63", outputs=9, identical=True)
    finally:
        ex.engine.close()
        del ex
        torch.cuda.empty_cache()


def test_full_batch_hft_windows_match_single_runs(sd):
    """A 128-frame handle at its largest batch (256 windows) through etude_forward_windows: windows 0, 31 and 255 must equal
    the same windows run alone bit for bit (rolls A / B and both velocity logits)."""
    eng = _engine(sd, 128, max_windows=256)
    try:
        nw, F = 256, 128
        feat = (torch.rand(nw * (F + 64), 256, device="cuda") * 20 - 18)

        def run(ws):
            ra, rb = eng.alloc_rolls(len(ws) * F, eng.device), eng.alloc_rolls(len(ws) * F, eng.device)
            va = torch.empty(len(ws) * F * 88 * 128, device="cuda")
            vb = torch.empty_like(va)
            sub = feat.view(nw, F + 64, 256)[ws].reshape(-1, 256) if len(ws) < nw else feat
            eng.forward_windows(sub, [i * (F + 64) for i in range(len(ws))], [i * F for i in range(len(ws))], rb, ra, va, vb)
            torch.cuda.synchronize()
            return ra, rb, va.view(len(ws), -1), vb.view(len(ws), -1)

        ra, rb, va, vb = run(list(range(nw)))
        for w in (0, 31, nw - 1):
            sa, sb, sva, svb = run([w])
            for full, one in zip(ra + rb, sa + sb):
                assert torch.equal(full[w * F:(w + 1) * F], one), w
            assert torch.equal(va[w], sva[0]) and torch.equal(vb[w], svb[0]), w
        del ra, rb, va, vb
        report("full_batch_hft_256_windows_vs_single", windows_checked=f"0/31/{nw - 1}", identical=True)
    finally:
        eng.close()
        del eng
        torch.cuda.empty_cache()
