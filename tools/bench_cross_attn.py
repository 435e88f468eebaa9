"""Decoder cross-attention at the forward pass's shapes: the fused kernel (etude_k_cross_attn: K|V projected per frame inside
the attention kernel) against the two-kernel path it replaces (gemm_bstat writing the layer's K|V [tokens, 512] to HBM, then
attention4 reading it back), for the three layers (layer 0: the shared q0-style table; layers 1-2: 88 query rows per frame).

32 windows x 512 frames = 16 384 frames by default: x is 2.1 GB and the K|V 4.3 GB per layer, far larger than the 126 MB L2.
Each layer's two variants are warmed up, then timed with CUDA events in alternation (fused, pair, fused, pair, ...).
Prints one JSON line (and writes it to --out FILE when given)."""
import argparse
import json
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=16384)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    from oracle import model as omodel
    from test_cross_attn_gpu import LAYERS, fused, head_major, layer_inputs, two_kernel  # noqa: F401
    from etude_b200 import _lib
    import gpu_diag as D

    sd = omodel.init_state_dict(0)
    F = a.frames
    lib = _lib.load()
    out = torch.empty((F * 88, 256), dtype=torch.bfloat16, device="cuda")
    kv = torch.empty((F * 256, 512), dtype=torch.bfloat16, device="cuda")
    res = {"frames": F, "gpu": torch.cuda.get_device_name(), "layers": []}
    try:
        import subprocess
        res["power_limit"] = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                                            capture_output=True, text=True).stdout.strip()
    except OSError:
        pass
    for layer in range(3):
        x, wkv, bkv, q, stride = layer_inputs(sd, layer, F, seed=11 + layer)
        w_hm, b_hm = head_major(wkv[:256], wkv[256:], bkv[:256], bkv[256:])

        def run_fused():
            _lib.check(lib.etude_k_cross_attn(D.P(x), D.P(w_hm), D.P(b_hm), D.P(q), q.shape[0], stride, F, D.P(out), D.stream()), "cross")

        def run_pair():
            _lib.check(lib.etude_k_gemm(D.P(x), D.P(wkv), D.P(bkv), F * 256, 512, 256, 0, D.P(kv), None, 0, None, None, None, D.stream()),
                       "gemm")
            _lib.check(lib.etude_k_attention(D.P(q), q.shape[0], 256, 0, stride, D.P(kv), 512, 0, 256, F, 88, 256, D.P(out), None,
                                             D.stream()), "attention")

        for fn in (run_fused, run_pair, run_fused, run_pair):
            fn()
        torch.cuda.synchronize()
        t = {"fused": [], "pair": []}
        for _ in range(a.reps):
            for name, fn in (("fused", run_fused), ("pair", run_pair)):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                fn()
                e1.record()
                torch.cuda.synchronize()
                t[name].append(e0.elapsed_time(e1))
        fm, pm = min(t["fused"]), min(t["pair"])
        flop = 2.0 * F * 256 * 512 * 256 + 4.0 * F * 4 * 88 * 256 * 64
        res["layers"].append({"layer": layer, "fused_ms": t["fused"], "pair_ms": t["pair"], "ratio_min": fm / pm,
                              "fused_tflops": flop / fm / 1e9})
    res["ratio_worst_layer"] = max(l["ratio_min"] for l in res["layers"])
    line = json.dumps(res)
    print(line)
    if a.out:
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
