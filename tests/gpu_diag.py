"""Stage-by-stage GPU diagnostics (run each stage in its own process so a trapping kernel cannot poison the rest):

    python tests/gpu_diag.py gemm|attn|logmel|notes|model|e2e
"""
import ctypes
import os
import sys
import tempfile
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from etude_b200 import _lib  # noqa: E402

try:
    from conftest import report  # noqa: E402
except Exception:  # noqa: BLE001  (stand-alone use)
    def report(name, **values):
        print("PARITY", name, values)

GOLD = os.path.join(ROOT, "tests", "golden")


def P(t):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else None


def stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def gemm(a, w, bias, epi, resid=None, resid_mod=0, gamma=None, beta=None):
    lib = _lib.load_dev()   # the generic tile GEMM epilogues live in the test-only build
    M, K = a.shape
    N = w.shape[0]
    out_bf16 = torch.empty((M, N), dtype=torch.bfloat16, device="cuda")
    out_f32 = torch.empty((M, N), dtype=torch.float32, device="cuda") if epi == 2 else None
    _lib.check(lib.etude_k_gemm(P(a), P(w), P(bias), M, N, K, epi, P(out_bf16), P(resid), resid_mod, P(gamma), P(beta), P(out_f32),
                                stream()), "etude_k_gemm", lib)
    torch.cuda.synchronize()
    return out_bf16, out_f32


def diag_gemm():
    torch.manual_seed(0)
    ok = True
    for (M, N, K, epi) in [(128, 256, 64, 0), (256, 256, 256, 0), (1000, 768, 256, 0), (128 * 150 + 5, 512, 512, 1),
                           (128 * 300, 256, 256, 2), (88 * 7, 256, 512, 2), (128 * 149 + 77, 256, 512, 2), (88 * 512 * 2, 256, 256, 2)]:
        a = (torch.randn(M, K, device="cuda") * 0.5).to(torch.bfloat16)
        w = (torch.randn(N, K, device="cuda") / K ** 0.5).to(torch.bfloat16)
        bias = torch.randn(N, device="cuda")
        ref = a.float() @ w.float().T + bias
        if epi == 1:
            ref = torch.relu(ref)
        resid = gamma = beta = None
        rmod = 0
        if epi == 2:
            rmod = 88 if M % 88 == 0 else 0
            resid = torch.randn(rmod if rmod else M, N, device="cuda")
            gamma = 1 + 0.1 * torch.randn(N, device="cuda")
            beta = 0.1 * torch.randn(N, device="cuda")
            r = resid.repeat(M // rmod, 1) if rmod else resid
            if rmod:   # wrapped table: the first 32 rows repeated after the end (see include/etude_b200_kernels.h)
                resid = torch.cat([resid, resid[:32]]).contiguous()
            ref = torch.nn.functional.layer_norm(ref + r, (N,), gamma, beta, 1e-5)
        t0 = time.time()
        try:
            ob, of = gemm(a, w, bias, epi, resid, rmod, gamma, beta)
        except Exception as e:  # noqa: BLE001
            print(f"GEMM M={M} N={N} K={K} epi={epi}: EXC {e}")
            ok = False
            break
        err_b = (ob.float() - ref).abs().max().item()
        err_f = (of - ref).abs().max().item() if of is not None else float("nan")
        scale = ref.abs().max().item()
        good = err_b <= 2e-2 * max(scale, 1.0) and (of is None or err_f <= 2e-3)
        ok &= good
        print(f"GEMM M={M} N={N} K={K} epi={epi}: bf16 err {err_b:.3e} f32 err {err_f:.3e} (|ref| max {scale:.2f}) "
              f"{'OK' if good else 'FAIL'} [{time.time() - t0:.2f}s]")
        if not good:
            d = (ob.float() - ref).abs()
            bad = (d > 2e-2 * max(scale, 1.0)).nonzero()
            print("   first bad idx:", bad[:5].tolist(), "rows bad:", torch.unique(bad[:, 0])[:10].tolist(),
                  "cols bad:", torch.unique(bad[:, 1])[:10].tolist(), "n_bad", bad.shape[0])
            print("   out[0,:8]", ob[0, :8].float().tolist(), "\n   ref[0,:8]", ref[0, :8].tolist())
    return ok


def diag_chain():
    """chain kernel (fc_o + LN [+ FFN + LN]) vs a torch fp32 reference fed the same bf16 operands."""
    lib = _lib.load()
    torch.manual_seed(2)
    ok = True
    bf = lambda t: t.to(torch.bfloat16)
    for (M, ffn, rmod) in [(128, True, 0), (128, False, 0), (300, True, 0), (88 * 5, True, 88), (128 * 149 + 77, True, 0),
                           (128 * 300, False, 0), (88 * 512 * 2, True, 88), (128 * 600, True, 0)] + ([(1441792, True, 0), (1441792, False, 0), (4194304, True, 0)] if os.environ.get('CHAIN_BIG') else []):
        ctx = bf(torch.randn(M, 256, device="cuda") * 0.7)
        wo = bf(torch.randn(256, 256, device="cuda") / 16)
        w1 = bf(torch.randn(512, 256, device="cuda") / 16)
        w2 = bf(torch.randn(256, 512, device="cuda") / 22)
        bo, b1, b2 = (0.1 * torch.randn(n, device="cuda") for n in (256, 512, 256))
        gamma = 1 + 0.1 * torch.randn(256, device="cuda")
        beta = 0.1 * torch.randn(256, device="cuda")
        if rmod:
            table = bf(torch.randn(rmod, 256, device="cuda"))
            resid_dev = table.repeat(3, 1).contiguous()
            resid = table.repeat(M // rmod, 1)
        else:
            resid_dev = bf(torch.randn(M, 256, device="cuda"))
            resid = resid_dev
        ln = lambda t: torch.nn.functional.layer_norm(t, (256,), gamma, beta, 1e-5)
        y = ln(ctx.float() @ wo.float().T + bo + resid.float())
        if ffn:
            hdn = torch.relu(bf(y).float() @ w1.float().T + b1)
            ref = ln(y + bf(hdn).float() @ w2.float().T + b2)
        else:
            ref = y
        out = resid_dev.clone() if not rmod else torch.empty((M, 256), dtype=torch.bfloat16, device="cuda")
        rsrc = out if not rmod else resid_dev      # in place, as the model uses it
        try:
            _lib.check(lib.etude_k_chain(P(ctx), P(wo), P(bo), P(w1) if ffn else None, P(b1) if ffn else None, P(w2) if ffn else None,
                                         P(b2) if ffn else None, P(gamma), P(beta), P(rsrc), rmod, rsrc.shape[0], P(out), M, stream()),
                       "etude_k_chain")
            torch.cuda.synchronize()
        except Exception as e:  # noqa: BLE001
            print(f"CHAIN M={M} ffn={ffn} rmod={rmod}: EXC {e}")
            return False
        err = (out.float() - ref).abs().max().item()
        good = err <= 4e-2
        ok &= good
        print(f"CHAIN M={M} ffn={ffn} rmod={rmod}: max-abs {err:.3e} (|ref| max {ref.abs().max().item():.2f}) {'OK' if good else 'FAIL'}")
        report(f"chain_vs_torch_fp32 M={M} ffn={ffn} rmod={rmod}", maxabs=err, scale=ref.abs().max().item())
        if not good:
            d = (out.float() - ref).abs()
            bad = (d > 4e-2).nonzero()
            print("   n_bad", bad.shape[0], "rows:", torch.unique(bad[:, 0])[:12].tolist(), "cols:", torch.unique(bad[:, 1])[:12].tolist())
            print("   out[0,:6]", out[0, :6].float().tolist(), "ref[0,:6]", ref[0, :6].tolist())
    return ok


def diag_chain_trace():
    """clock64 timeline of CTA 0 of the FFN chain kernel (MMA thread / one epilogue thread / ring producer)."""
    lib = _lib.load_dev()
    torch.manual_seed(2)
    bf = lambda t: t.to(torch.bfloat16)
    M = 128 * 148 * 12
    ctx = bf(torch.randn(M, 256, device="cuda") * 0.7)
    wo = bf(torch.randn(256, 256, device="cuda") / 16)
    w1 = bf(torch.randn(512, 256, device="cuda") / 16)
    w2 = bf(torch.randn(256, 512, device="cuda") / 22)
    bo, b1, b2 = (0.1 * torch.randn(n, device="cuda") for n in (256, 512, 256))
    gamma = 1 + 0.1 * torch.randn(256, device="cuda")
    beta = 0.1 * torch.randn(256, device="cuda")
    x = bf(torch.randn(M, 256, device="cuda"))
    def run():
        _lib.check(lib.etude_k_chain(P(ctx), P(wo), P(bo), P(w1), P(b1), P(w2), P(b2), P(gamma), P(beta), P(x), 0, M, P(x), M, stream()),
                   "etude_k_chain")
    for _ in range(3):
        run()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(); run(); e1.record(); torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    print(f"CHAIN_TRACE M={M}: {ms:.3f} ms untraced, {2 * M * (256 * 256 + 2 * 512 * 256) / ms / 1e9:.0f} TFLOP/s")
    _lib.check(lib.etude_debug_chain_trace(1, None, 0), "trace on")
    run()
    n = 3 * 512 * 2
    buf = (ctypes.c_int64 * n)()
    _lib.check(lib.etude_debug_chain_trace(0, buf, n), "trace read")
    a = np.array(buf, dtype=np.int64).reshape(3, 512, 2)
    names = {0: "MMA", 1: "EPI", 2: "TMA"}
    ev = []
    for r in range(3):
        for i in range(512):
            if a[r, i, 1] != 0:
                ev.append((int(a[r, i, 1]), r, int(a[r, i, 0])))
    ev.sort()
    t0 = min(t for t, r, i in ev if i // 100 == 5)
    print("events of tiles 5..7 of CTA 0 (clk relative to the first event of tile 5):")
    for t, r, i in ev:
        if 5 <= i // 100 <= 7:
            print(f"  {t - t0:8d}  {names[r]}  tile {i // 100} ev {i % 100}")
    return True


def diag_attn_trace():
    """clock64 timeline of CTA 0 of attention4 at the encoder shape: S issue, P V issue, softmax begin/end, drain begin/end."""
    lib = _lib.load_dev()
    torch.manual_seed(3)
    S, L = 148 * 16 // 4, 256
    qkv = torch.randn(S * L, 768, device="cuda").to(torch.bfloat16)
    out = torch.zeros((S * L, 256), dtype=torch.bfloat16, device="cuda")
    args = (P(qkv), S * L, 768, 0, L, P(qkv), 768, 256, 512)
    def run():
        _lib.check(lib.etude_k_attention(*args, S, L, L, P(out), None, stream()), "etude_k_attention")
    for _ in range(3):
        run()
    torch.cuda.synchronize()
    _lib.check(lib.etude_debug_chain_trace(1, None, 0), "trace on")
    run()
    n = 8 * 192 * 2
    buf = (ctypes.c_int64 * n)()
    _lib.check(lib.etude_debug_chain_trace(0, buf, n), "trace read")
    a = np.array(buf, dtype=np.int64).reshape(8, 192, 2)
    names = ["S-issue", "PV-issued", "drain-top", "(unused)", "drain-ready", "drain-freed", "drain-stored", "PV-o_full"]
    t0 = a[0, 0, 1]
    print("tile: " + " ".join(f"{n:>11s}" for n in names) + "   (clk since the first S issue; tile = 128 x 128 scores)")
    for g in range(24, 48):
        if a[0, g, 1] == 0:
            break
        print(f"{g:4d}: " + " ".join(f"{int(a[r, g, 1] - t0):11d}" for r in range(8)))
    return True


def diag_mma_bench():
    """tcgen05.mma execution rate per shape / operand source (clk per MMA, one CTA per SM)."""
    lib = _lib.load_dev()
    out = (ctypes.c_int64 * 2)()
    for grid in (148,):
        for mode, n in [(0, 128), (2, 64), (2, 128), (2, 256), (3, 64), (3, 128), (3, 256), (4, 64), (5, 64)]:
            iters = 2048
            _lib.check(lib.etude_debug_mma_bench(mode, n, iters, 4, grid, out), "mma_bench")
            _lib.check(lib.etude_debug_mma_bench(mode, n, iters, 4, grid, out), "mma_bench")
            fl = 2 * 128 * n * 16
            print(f"MMA grid={grid:3d} {['SS', 'TS', 'SS-uniform', 'TS-uniform', 'TS-uniform-Bmn', 'SS-uniform-Bmn'][mode]} M128 N{n:<3d} K16: issue {out[0] / iters:6.1f} clk/MMA, "
                  f"complete {out[1] / iters:6.1f} clk/MMA = {fl * iters / out[1]:6.0f} flop/clk/SM (floor {128 * n / 256:.0f} clk)")
    return True


def diag_mma_mix():
    """tcgen05.mma rate while other warps of the CTA load / store TMEM."""
    lib = _lib.load_dev()
    out = (ctypes.c_int64 * 2)()
    for ts in (1, 0):
        for st_too in (0, 1):
            for n_ld in (0, 4, 8, 16):
                iters = 4096
                _lib.check(lib.etude_debug_mma_mix(ts, iters, n_ld, st_too, 148, out), "mma_mix")
                _lib.check(lib.etude_debug_mma_mix(ts, iters, n_ld, st_too, 148, out), "mma_mix")
                print(f"MMAMIX {'TS M128 N64 ' if ts else 'SS M128 N128'} K16 with {n_ld:2d} warps doing tcgen05.ld{'+st' if st_too else '   '}: "
                      f"{out[0] / iters:7.1f} clk per MMA; {out[1]} ld iterations by one warp ({out[0] / max(out[1], 1):.0f} clk each)")
    return True


def diag_pairmma():
    """cta_group::2 self-test (pairmma.cuh): SS pair MMA with B split over the two CTAs, TS pair MMA with A in TMEM."""
    lib = _lib.load_dev()
    torch.manual_seed(3)
    a = torch.randn(256, 64, device="cuda").to(torch.bfloat16)
    b = torch.randn(128, 64, device="cuda").to(torch.bfloat16)
    vt = torch.randn(64, 128, device="cuda").to(torch.bfloat16)
    d = torch.full((256, 128), float("nan"), device="cuda")
    o = torch.full((256, 64), float("nan"), device="cuda")
    _lib.check(lib.etude_debug_pairmma(P(a), P(b), P(vt), P(d), P(o)), "etude_debug_pairmma", lib)
    d_ref = a.float() @ b.float().t()
    p_ref = d_ref.to(torch.bfloat16).float()
    o_ref = p_ref @ vt.float().t()
    e_d = (d - d_ref).abs().max().item()
    e_o = (o - o_ref).abs().max().item()
    ok = e_d < 1e-3 and e_o < 0.05 * o_ref.abs().max().item() / 10
    print(f"PAIRMMA D err {e_d:.3e} (|ref| max {d_ref.abs().max().item():.2f}), O err {e_o:.3e} (|ref| max {o_ref.abs().max().item():.2f}) {'OK' if ok else 'FAIL'}")
    if not ok:   # which quadrants are wrong: rows by CTA, columns by the CTA that supplied the B half
        for name, got, ref, h in (("D", d, d_ref, 64), ("O", o, o_ref, 32)):
            for r in range(2):
                for c in range(2):
                    q = (got[128 * r:128 * r + 128, h * c:h * c + h] - ref[128 * r:128 * r + 128, h * c:h * c + h]).abs().max().item()
                    print(f"   {name} rows of CTA {r}, B half of CTA {c}: err {q:.3e}")
    return ok


def diag_pairmma_bench():
    """tcgen05.mma rates: cta_group::2 (M = 256 over a CTA pair) next to cta_group::1 (M = 128), uniform issue loops."""
    lib = _lib.load_dev()
    out = (ctypes.c_int64 * 2)()
    iters = 4096
    for ts in (0, 1):
        for n in (64, 128, 192, 256):
            _lib.check(lib.etude_debug_pairmma_bench(ts, n, iters, 0, 148, out), "pairmma_bench", lib)
            _lib.check(lib.etude_debug_pairmma_bench(ts, n, iters, 0, 148, out), "pairmma_bench", lib)
            clk2 = out[1] / iters
            mode1 = 3 if ts else 2
            _lib.check(lib.etude_debug_mma_bench(mode1, n, iters, 4, 148, out), "mma_bench", lib)
            _lib.check(lib.etude_debug_mma_bench(mode1, n, iters, 4, 148, out), "mma_bench", lib)
            clk1 = out[1] / iters
            floor = 128 * n * 16 * 2 / 8192
            print(f"MMARATE {'TS' if ts else 'SS'} N{n:3d} K16: cta_group::1 (M128) {clk1:6.1f} clk/MMA = {100 * floor / clk1:5.1f} % of the tensor floor ({floor:.0f} clk); "
                  f"cta_group::2 (M256 over the pair) {clk2:6.1f} clk/MMA = {100 * floor / clk2:5.1f} %")
    for alt in (1, 2):
        for n in (64, 128):
            _lib.check(lib.etude_debug_pairmma_bench(0, n, iters, alt, 148, out), "pairmma_bench", lib)
            _lib.check(lib.etude_debug_pairmma_bench(0, n, iters, alt, 148, out), "pairmma_bench", lib)
            print(f"MMARATE SS N{n:3d} K16 cta_group::2, consecutive MMAs alternating two accumulators{' and sharing the A slice' if alt == 2 else ''}: "
                  f"{out[1] / iters:6.1f} clk/MMA")
    return True


def diag_embed():
    """Tensor-core embedding (hi/lo bf16 split) against a torch fp32 reference of the same op (conv -> linear -> scale + pos)."""
    ex, sd = make_extractor(max_windows=8)
    eng = ex.engine
    lib = eng.lib
    from oracle import model as omodel
    torch.manual_seed(5)
    nw = 8
    rows = 512 * 3 + 64
    feat = (torch.rand(rows, 256, device="cuda") * 23 - 18).contiguous()
    win_rows = [0, 512, 1024, 7, 300, 1000, 512, 64]
    out = torch.zeros((nw * 512 * 256, 256), dtype=torch.bfloat16, device="cuda")
    _lib.check(lib.etude_k_embed(eng._h, P(feat), _lib.i64_array(win_rows), nw, P(out), 0, stream()), "etude_k_embed")
    torch.cuda.synchronize()
    got = out.float().view(nw, 512, 256, 256)
    # torch fp32 reference: conv(1x5, 4 ch) along the 65-frame context -> linear(244, 256) -> * 16 + pos[bin]
    w = {k: v.cuda().float() for k, v in sd.items() if k.startswith("encoder.")}
    ok = True
    for wi in (0, 3, 7):
        x = feat[win_rows[wi]: win_rows[wi] + 576]                      # [576, 256]
        u = x.unfold(0, 65, 1)                                            # [512, 256, 65]
        c = torch.nn.functional.conv2d(u.reshape(512 * 256, 1, 1, 65), w["encoder.conv.weight"], w["encoder.conv.bias"])  # [N,4,1,61]
        t = torch.nn.functional.linear(c.reshape(512 * 256, 244), w["encoder.tok_embedding_freq.weight"], w["encoder.tok_embedding_freq.bias"])
        ref = (t * 16.0).view(512, 256, 256) + w["encoder.pos_embedding_freq.weight"][None]
        e2 = (got[wi] - ref).abs().max().item()
        scale = ref.abs().max().item()
        good = e2 <= 0.01 * scale     # bf16 output rounding (2^-9 relative) + bf16 weights over 65 taps
        ok &= good
        print(f"EMBED window {wi}: tensor-core err {e2:.3e} (|ref| max {scale:.2f}, tolerance {0.01 * scale:.3e}) {'OK' if good else 'FAIL'}")
    e0, e1_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for variant in (0, 17, 18, 20, 22):   # 16 + mask: 1 no stores, 2 no epilogue arithmetic, 4 no A-tile build (diagnostics)
        out = torch.zeros((nw * 512 * 256, 256), dtype=torch.bfloat16, device="cuda")
        for it in range(4):
            if it == 1:
                e0.record()
            _lib.check(lib.etude_k_embed(eng._h, P(feat), _lib.i64_array(win_rows), nw, P(out), variant, stream()), "etude_k_embed")
        e1_.record()
        torch.cuda.synchronize()
        print(f"EMBED variant {variant}: {e0.elapsed_time(e1_) / 3:.3f} ms per {nw} windows")
    return ok


def diag_tmem_bench():
    """TMEM read bandwidth, MUFU and pack rates per SM as a function of the number of warps (clk per loop body per warp)."""
    lib = _lib.load_dev()
    out = (ctypes.c_int64 * 1)()
    names = ["tcgen05.ld x32 (4 KB)", "32 ex2 / lane", "16 bf16x2 packs / lane", "softmax pass-2 body (32 cols)", "16 fmax3 / lane",
             "tcgen05.st x16 (2 KB)", "2 x tcgen05.ld x32 (8 KB)"]
    for mode in (0, 6, 5, 3):
        for nw in (1, 4, 8, 16):
            iters = 4096
            _lib.check(lib.etude_debug_tmem_bench(mode, nw, iters, 148, out), "tmem_bench")
            _lib.check(lib.etude_debug_tmem_bench(mode, nw, iters, 148, out), "tmem_bench")
            per = out[0] / iters
            print(f"TMEMBENCH {names[mode]:32s} warps={nw:2d}: {per:7.1f} clk per body per warp -> {nw / per:6.3f} bodies/clk/SM")
    return True


def attention_ref(q, k, v):
    # q [S, Lq, 4, 64], k/v [S, Lk, 4, 64]
    e = torch.einsum("sqhd,skhd->shqk", q.float(), k.float()) / 8.0
    p = torch.softmax(e, dim=-1)
    o = torch.einsum("shqk,skhd->sqhd", p, v.float())
    return o, p


def diag_attn():
    lib = _lib.load()
    torch.manual_seed(1)
    ok = True
    for (S, Lq, Lk, cross) in [(3, 256, 256, False), (5, 88, 88, False), (4, 88, 256, True), (2, 512, 512, False), (300, 256, 256, False),
                               (75, 512, 512, False), (700, 88, 256, True), (900, 88, 88, False)]:
        if cross:
            qsrc = (torch.randn(S * Lq, 256, device="cuda")).to(torch.bfloat16)
            kvsrc = (torch.randn(S * Lk, 1536, device="cuda")).to(torch.bfloat16)
            q = qsrc.view(S, Lq, 4, 64)
            k = kvsrc[:, 512:768].reshape(S, Lk, 4, 64)
            v = kvsrc[:, 768:1024].reshape(S, Lk, 4, 64)
            args = (P(qsrc), S * Lq, 256, 0, Lq, P(kvsrc), 1536, 512, 768)
        else:
            qkv = (torch.randn(S * Lq, 768, device="cuda")).to(torch.bfloat16)
            q = qkv[:, :256].reshape(S, Lq, 4, 64)
            k = qkv[:, 256:512].reshape(S, Lk, 4, 64)
            v = qkv[:, 512:].reshape(S, Lk, 4, 64)
            args = (P(qkv), S * Lq, 768, 0, Lq, P(qkv), 768, 256, 512)
        out = torch.zeros((S * Lq, 256), dtype=torch.bfloat16, device="cuda")
        probs = torch.zeros((S, 4, Lq, Lk), dtype=torch.float32, device="cuda") if Lk <= 256 else None
        try:
            _lib.check(lib.etude_k_attention(*args, S, Lq, Lk, P(out), P(probs), stream()), "etude_k_attention")
            torch.cuda.synchronize()
        except Exception as e:  # noqa: BLE001
            print(f"ATTN S={S} Lq={Lq} Lk={Lk}: EXC {e}")
            return False
        tf = float("nan")
        if S >= 75:  # timing of the big shapes (no probabilities output), CUDA events on the launching stream
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            for it in range(6):
                if it == 1:
                    e0.record()
                _lib.check(lib.etude_k_attention(*args, S, Lq, Lk, P(out), None, stream()), "etude_k_attention")
            e1.record()
            torch.cuda.synchronize()
            tf = 4.0 * S * 4 * Lq * Lk * 64 * 5 / (e0.elapsed_time(e1) * 1e-3) / 1e12
        ref, pref = attention_ref(q, k, v)
        err = (out.view(S, Lq, 4, 64).float() - ref).abs().max().item()
        perr = (probs - pref).abs().max().item() if probs is not None else float("nan")
        good = err <= 3e-2 and (probs is None or perr <= 2e-3)
        ok &= good
        print(f"ATTN S={S} Lq={Lq} Lk={Lk} cross={cross}: out err {err:.3e} probs err {perr:.3e} {'OK' if good else 'FAIL'}  {tf:.0f} TFLOP/s")
        report(f"attention_vs_torch_fp32 S={S} Lq={Lq} Lk={Lk}", out_maxabs=err, probs_maxabs=perr, tflops=tf)
        if not good:
            d = (out.view(S, Lq, 4, 64).float() - ref).abs()
            print("   err by head:", d.amax(dim=(0, 1, 3)).tolist(), " by d-chunk:", d.view(S, Lq, 4, 8, 8).amax(dim=(0, 1, 2, 4)).tolist())
            print("   err by q-row block(32):", d.amax(dim=(0, 2, 3)).view(-1, 8 if Lq % 8 == 0 else 1).amax(1)[:16].tolist())
            if probs is not None:
                dp = (probs - pref).abs()
                print("   probs err by key block(32):", dp.amax(dim=(0, 1, 2)).view(-1, 8).amax(1).tolist()[:16])
    return ok


def diag_attn_qkv():
    """Fused Q|K|V projection + attention (attn_qkv.cuh) against a torch fp32 reference fed the same bf16 x / W (reference
    amt_apc.py:342-368); the reference rounds Q, K, V to bf16 like the kernel's MMA operands."""
    lib = _lib.load_dev() if os.environ.get("ETUDE_DIAG_DEV") else _lib.load()
    torch.manual_seed(7)
    ok = True
    for S in ((1, 75, 16384) if os.environ.get("ETUDE_DIAG_DEV") else (1, 2, 3, 75, 148, 512, 1000, 2048, 16384)):
        xs_scale = 1.5
        x = (torch.randn(S * 256, 256, device="cuda") * xs_scale).to(torch.bfloat16)
        w = (torch.randn(768, 256, device="cuda") / 16).to(torch.bfloat16)       # fc_q | fc_k | fc_v rows (nn.Linear layout)
        b = 0.2 * torch.randn(768, device="cuda")
        # head-major packing: row h * 192 + {Q_h | K_h | V_h}
        idx = torch.cat([torch.cat([torch.arange(64) + part * 256 + h * 64 for part in range(3)]) for h in range(4)]).cuda()
        w_hm, b_hm = w[idx].contiguous(), b[idx].contiguous()
        out = torch.zeros((S * 256, 256), dtype=torch.bfloat16, device="cuda")
        try:
            _lib.check(lib.etude_k_attn_qkv(P(x), P(w_hm), P(b_hm), S, P(out), stream()), "etude_k_attn_qkv", lib)
            torch.cuda.synchronize()
        except Exception as e:  # noqa: BLE001
            print(f"ATTNQKV S={S}: EXC {e}")
            return False
        tf = float("nan")
        if S >= 1000:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            for it in range(6):
                if it == 1:
                    e0.record()
                _lib.check(lib.etude_k_attn_qkv(P(x), P(w_hm), P(b_hm), S, P(out), stream()), "etude_k_attn_qkv")
            e1.record()
            torch.cuda.synchronize()
            fl = 2.0 * S * 256 * 768 * 256 + 4.0 * S * 4 * 256 * 256 * 64
            tf = fl * 5 / (e0.elapsed_time(e1) * 1e-3) / 1e12
        # EVERY sequence is checked (in slabs of 64: a sampled check of the first / last sequences once let a bug through that
        # only hit iterations in the middle of a cluster's work list)
        err, ref_max, per_seq = 0.0, 0.0, []
        for s0 in range(0, S, 64):
            s1 = min(S, s0 + 64)
            xs = x.view(S, 256, 256)[s0:s1].float()
            qkv = (xs @ w.float().T + b).to(torch.bfloat16)
            q, k, v = (qkv[..., i * 256:(i + 1) * 256].reshape(s1 - s0, 256, 4, 64) for i in range(3))
            ref, _ = attention_ref(q, k, v)
            got = out.view(S, 256, 4, 64)[s0:s1].float()
            d = (got - ref).abs()
            d = torch.where(torch.isnan(d), torch.full_like(d, float("inf")), d)
            per_seq.append(d.amax(dim=(1, 2, 3)))
            err = max(err, d.max().item())
            ref_max = max(ref_max, ref.abs().max().item())
        per_seq = torch.cat(per_seq)
        good = err <= 0.01 * max(1.0, ref_max)   # bf16 P / Q / K / V operands: 2^-8 relative on |out| ~ 6
        ok &= good
        print(f"ATTNQKV S={S}: out err {err:.3e} (|ref| max {ref_max:.2f}) {'OK' if good else 'FAIL'}  {tf:.0f} TFLOP/s")
        report(f"attn_qkv_fused_vs_torch_fp32 S={S}", out_maxabs=err, tflops=tf)
        if not good:
            bad = torch.nonzero(per_seq > 0.01 * max(1.0, ref_max)).flatten().tolist()
            print(f"   {len(bad)} bad sequences of {S}; first: {bad[:24]}")
            print(f"   bad sequence index mod 74 (cluster): {sorted(set(i % 74 for i in bad))[:40]}")
            print(f"   bad sequence index // 74 (iteration of its cluster): {sorted(set(i // 74 for i in bad))[:40]}")
            got = out.view(S, 256, 4, 64)[bad[0]].float()
            xs = x.view(S, 256, 256)[bad[0]:bad[0] + 1].float()
            qkv = (xs @ w.float().T + b).to(torch.bfloat16)
            q, k, v = (qkv[..., i * 256:(i + 1) * 256].reshape(1, 256, 4, 64) for i in range(3))
            d = (got - attention_ref(q, k, v)[0][0]).abs()
            print("   first bad sequence: err by head:", [round(t, 4) for t in d.amax(dim=(0, 2)).tolist()])
            print("   err by token block(32):", [round(t, 4) for t in d.amax(dim=(1, 2)).view(8, 32).amax(1).tolist()])
            print("   err by dim block(16):", [round(t, 4) for t in d.amax(dim=(0, 1)).view(4, 16).amax(1).tolist()])
    return ok


def diag_attn_qkv_cross():
    """The product's CTA-pair kernel (attn_pair.cuh) against the independent cta_group::1 implementation (attn_qkv.cuh, test-only
    library) on identical inputs, including activations of the first encoder layer's size: the x16-scaled embedding is not
    normalised before the first attention, so scores run into the hundreds / thousands (log2 domain), softmax rows are one-hot
    and the maxima of the two key blocks lie far apart -- the regime of attn_pair's asymmetric reference and of its clamped
    polynomial ex2.  (Against torch such inputs only measure bf16 rounding flips of Q / K between almost-tied keys; the two
    kernels share the projection bit for bit, so here any difference beyond bf16 rounding of P is a softmax / P V bug.)"""
    lib = _lib.load_dev()
    torch.manual_seed(11)
    ok = True
    for S, sc, shift in ((148, 1.5, 0.0), (148, 24.0, 0.0), (512, 60.0, 0.0), (300, 200.0, 0.0), (300, 24.0, 40.0)):
        x = (torch.randn(S * 256, 256, device="cuda") * sc)
        if shift:   # half of every sequence's tokens far away from the other half: block maxima > 2^100 apart in both directions
            x.view(S, 256, 256)[:, 128:] += shift * torch.sign(torch.randn(S, 1, 256, device="cuda"))
        x = x.to(torch.bfloat16)
        w = (torch.randn(768, 256, device="cuda") / 16).to(torch.bfloat16)
        b = 0.2 * torch.randn(768, device="cuda")
        idx = torch.cat([torch.cat([torch.arange(64) + part * 256 + h * 64 for part in range(3)]) for h in range(4)]).cuda()
        w_hm, b_hm = w[idx].contiguous(), b[idx].contiguous()
        o_pair = torch.zeros((S * 256, 256), dtype=torch.bfloat16, device="cuda")
        o_ref = torch.zeros_like(o_pair)
        _lib.check(lib.etude_k_attn_qkv(P(x), P(w_hm), P(b_hm), S, P(o_pair), stream()), "etude_k_attn_qkv", lib)
        _lib.check(lib.etude_debug_attn_qkv_cta1(P(x), P(w_hm), P(b_hm), S, P(o_ref), stream()), "etude_debug_attn_qkv_cta1", lib)
        torch.cuda.synchronize()
        a, r = o_pair.float().view(S, 256, 4, 64), o_ref.float().view(S, 256, 4, 64)
        d = (a - r).abs()
        d = torch.where(torch.isnan(d), torch.full_like(d, float("inf")), d)
        tol = 2.0 ** -6 * max(1.0, r.abs().max().item())     # a few bf16 ulps of the largest output
        bad = torch.nonzero(d.amax(dim=(1, 2, 3)) > tol).flatten().tolist()
        good = not bad and bool(torch.isfinite(a).all())
        ok &= good
        print(f"ATTNQKV_CROSS S={S} x*{sc} shift {shift}: max diff {d.max().item():.3e} (|out| max {r.abs().max().item():.1f}, tol {tol:.2f}) "
              f"{'OK' if good else 'FAIL: %d sequences, first %s' % (len(bad), bad[:12])}")
        report(f"attn_pair_vs_cta1_kernel S={S} x_scale={sc} shift={shift}", maxdiff=d.max().item(), out_scale=r.abs().max().item())
    return ok


def diag_attn_qkv_trace():
    """clock64 timeline of cluster 0 / rank 0 of the fused projection + attention kernel (dev build)."""
    lib = _lib.load_dev()
    torch.manual_seed(7)
    S = 74 * 24
    x = (torch.randn(S * 256, 256, device="cuda") * 1.5).to(torch.bfloat16)
    w_hm = (torch.randn(768, 256, device="cuda") / 16).to(torch.bfloat16)
    b_hm = 0.2 * torch.randn(768, device="cuda")
    out = torch.zeros((S * 256, 256), dtype=torch.bfloat16, device="cuda")
    def run():
        _lib.check(lib.etude_k_attn_qkv(P(x), P(w_hm), P(b_hm), S, P(out), stream()), "etude_k_attn_qkv", lib)
    for _ in range(3):
        run()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(); run(); e1.record(); torch.cuda.synchronize()
    print(f"ATTNQKV_TRACE S={S}: {e0.elapsed_time(e1) * 1e3:.0f} us untraced = {e0.elapsed_time(e1) * 1e3 / 24 / 4:.2f} us per (sequence, head)")
    _lib.check(lib.etude_debug_chain_trace(1, None, 0), "trace on", lib)
    run()
    n = 16 * 64 * 8
    buf = (ctypes.c_int64 * n)()
    _lib.check(lib.etude_debug_chain_trace(0, buf, n), "trace read", lib)
    a = np.array(buf, dtype=np.int64)
    names = {0: ("TMA", ["x issue", "W0", "W1", "W2", "W3"]), 1: ("PROJ", ["acc_free", "w0", "w1", "w2", "w3"]),
             2: ("S", ["qk_ready", "buf0", "buf1"]), 3: ("PV", ["v_ready+o_free", "p0", "p1"]),
             4: ("EPI", ["acc_full", "acc released", "qk pub", "v_free", "v pub"]), 5: ("DRAIN", ["o_full", "o_free", "stored"]),
             6: ("SM0", ["s_full", "max", "p_full"]), 7: ("SM1", ["s_full", "max", "p_full"])}
    both = bool(np.any(a[8 * 64 * 8:]))        # attn_pair.cuh traces both ranks of cluster 0 on a common time axis
    a = a.reshape(16, 64, 8) if both else a[:8 * 64 * 8].reshape(8, 64, 8)
    t0 = a[1, 8, 0]
    rel = lambda v: int(v - t0) if v else -1
    print("clk relative to PROJ acc_free of iteration 8 (iteration = (sequence, head); 4 per sequence)"
          + ("; rank 1 rows: same axis to within the start-up cluster barrier's release skew" if both else ""))
    for it in range(8, 17):
        print(f"--- iteration {it}")
        for r in range(16 if both else 8):
            if r >= 8 and not np.any(a[r, it]):
                continue
            nm, evs = names[r & 7]
            print(f"   {nm + ('.1' if r >= 8 else ''):8s} " + "  ".join(f"{e}={rel(a[r, it, k])}" for k, e in enumerate(evs)))
    return True


def make_extractor(max_windows=4):
    from etude_b200 import AMTAPC_Extractor, ExtractorConfig
    from oracle import model as omodel
    sd = omodel.init_state_dict(0)
    with tempfile.TemporaryDirectory() as tmp:     # the extractor reads the checkpoint in its constructor
        path = os.path.join(tmp, "sd.pth")
        torch.save(sd, path)
        return AMTAPC_Extractor(ExtractorConfig(), path, device="cuda:0", max_windows=max_windows), sd


def diag_logmel():
    ex, _ = make_extractor()
    z = np.load(os.path.join(GOLD, "logmel.npz"))
    ok = True
    for case in ["noise_1s", "tones_2s", "noise_ragged", "noise_short", "silence"]:
        feat = ex.wave_to_feature(z[case + "_wave"]).cpu().numpy()
        ref = z[case + "_feat"]
        err = np.abs(feat - ref).max() if feat.shape == ref.shape else float("inf")
        good = err <= 1e-3
        ok &= good
        print(f"LOGMEL {case}: shape {feat.shape} vs {ref.shape} max-abs {err:.3e} {'OK' if good else 'FAIL'}")
        report("logmel_vs_reference_" + case, maxabs=float(err), tolerance=1e-3)
        if not good and feat.shape == ref.shape:
            d = np.abs(feat - ref)
            print("   worst frame/bin:", np.unravel_index(d.argmax(), d.shape), "per-frame max:", d.max(1)[:8], "got", feat[0, :4], "ref", ref[0, :4])
    return ok


def diag_notes():
    from conftest import NOTE_CASES, note_variants
    ex, _ = make_extractor()
    z = np.load(os.path.join(GOLD, "notes.npz"))
    ok = True
    for case in NOTE_CASES:
        t_on, t_off, t_mpe = z[case + "__thr"]
        for mo, mv, ref in note_variants(z, case):
            got = ex._mpe2note(z[case + "__onset"], z[case + "__offset"], z[case + "__mpe"], z[case + "__velocity"],
                               thred_onset=t_on, thred_offset=t_off, thred_mpe=t_mpe, mode_velocity=mv, mode_offset=mo)
            good = got == ref
            ok &= good
            msg = ""
            if not good:
                nd = sum(1 for a, b in zip(got, ref) if a != b)
                first = next(((a, b) for a, b in zip(got, ref) if a != b), None)
                msg = f" len {len(got)} vs {len(ref)}; {nd} differ; first {first}"
            print(f"NOTES {case} {mo} {mv}: {'OK' if good else 'FAIL'}{msg}")
    return ok


def diag_model():
    ex, sd = make_extractor(max_windows=2)
    z = np.load(os.path.join(GOLD, "model_window.npz"))
    x = torch.from_numpy(z["input_spec"]).cuda()
    t0 = time.time()
    o = ex.model(x)
    torch.cuda.synchronize()
    print(f"MODEL forward 1 window {time.time() - t0:.3f}s")
    ok = True
    for i, k in [(0, "onset_f"), (1, "offset_f"), (2, "mpe_f"), (5, "onset_t"), (6, "offset_t"), (7, "mpe_t")]:
        err = np.abs(o[i].cpu().numpy() - z[k]).max()
        good = err <= 2e-2
        ok &= good
        print(f"MODEL {k}: max-abs {err:.3e} {'OK' if good else 'FAIL'}")
    fr = z["frames"]
    for i, k in [(3, "velocity_f_sample"), (8, "velocity_t_sample")]:
        err = np.abs(o[i][0, fr].cpu().numpy() - z[k]).max()
        print(f"MODEL {k}: logits max-abs {err:.3e} (|ref| max {np.abs(z[k]).max():.2f})")
    err = np.abs(o[4][0, fr].cpu().numpy() - z["attention_sample"]).max()
    print(f"MODEL attention: max-abs {err:.3e}")
    for i, k in [(3, "velocity_f_argmax"), (8, "velocity_t_argmax")]:
        agree = (o[i].argmax(3).cpu().numpy() == z[k]).mean()
        print(f"MODEL {k}: agreement {agree:.4f}")
    return ok


def diag_e2e():
    import __graft_entry__ as g
    g.smoke()
    return True


if __name__ == "__main__":
    stage = sys.argv[1]
    fn = {"pairmma": diag_pairmma, "pairmma_bench": diag_pairmma_bench, "gemm": diag_gemm, "chain": diag_chain, "chain_trace": diag_chain_trace, "mma_bench": diag_mma_bench, "embed": diag_embed, "mma_mix": diag_mma_mix, "attn_trace": diag_attn_trace, "tmem_bench": diag_tmem_bench, "attn": diag_attn, "attn_qkv": diag_attn_qkv, "attn_qkv_cross": diag_attn_qkv_cross, "attn_qkv_trace": diag_attn_qkv_trace, "logmel": diag_logmel, "notes": diag_notes, "model": diag_model, "e2e": diag_e2e}[stage]
    print(f"== {stage} ==", flush=True)
    ok = fn()
    print(f"== {stage}: {'PASS' if ok else 'FAIL'} ==", flush=True)
    sys.exit(0 if ok else 1)
