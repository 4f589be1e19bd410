"""Micro-benchmarks of the individual kernels on the shapes of the MapAnything hot path (run under gpurun)."""
import json
import sys
from pathlib import Path

import torch

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT / "map-anything_b200"))
from mapanything_b200 import ops  # noqa: E402


def timeit(fn, iters=20, warm=3):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    for _ in range(iters):
        fn()
    e.record()
    torch.cuda.synchronize()
    return s.elapsed_time(e) / iters


def main():
    V = int(sys.argv[1]) if len(sys.argv) > 1 else 8
    only = sys.argv[2] if len(sys.argv) > 2 else "all"   # "all" | "attn" | "gemm" | "conv"
    res = []
    M = 1370 * V
    for name, (m, n, k) in {} if only not in ("all", "gemm") else {
        "enc_qkv": (M, 3072, 1024), "enc_proj": (M, 1024, 1024), "enc_fc1": (M, 4096, 1024), "enc_fc2": (M, 1024, 4096),
        "is_qkv": (1369 * V + 1, 2304, 768), "is_proj": (1369 * V + 1, 768, 768), "is_fc1": (1369 * V + 1, 3072, 768),
        "is_fc2": (1369 * V + 1, 768, 3072),
    }.items():
        x = torch.randn(m, k, device="cuda").bfloat16()
        w = torch.randn(n, k, device="cuda").bfloat16()
        o = torch.empty(m, n, device="cuda", dtype=torch.bfloat16)
        for bn in (0, 64, 128, 256, 2128, 2256):
            t = timeit(lambda: ops.gemm(x, w, o, block_n=bn))
            res.append({"kernel": "gemm", "name": name, "bn": bn, "M": m, "N": n, "K": k, "ms": t, "tflops": 2 * m * n * k / t / 1e9})
        t = timeit(lambda: torch.matmul(x, w.t()))
        res.append({"kernel": "cublas", "name": name, "M": m, "N": n, "K": k, "ms": t, "tflops": 2 * m * n * k / t / 1e9})
    for name, (n, H, W, Cc, Co) in {} if only not in ("all", "conv") else {"rn1_148": (4, 148, 148, 96, 256), "rcu_148": (4, 148, 148, 256, 256), "rcu_74": (4, 74, 74, 256, 256),
                                    "reg1_296": (4, 296, 296, 256, 128), "reg2_518": (2, 518, 518, 128, 128)}.items():
        x = torch.randn(n, H, W, Cc, device="cuda").bfloat16()
        w = torch.randn(Co, 9 * Cc, device="cuda").bfloat16()
        o = torch.empty(n * H * W, Co, device="cuda", dtype=torch.bfloat16)
        for bn in (0, 64, 128, 256, 2128, 2256):
            if bn % 1000 > Co and bn:
                continue
            t = timeit(lambda: ops.conv3x3(x, w, o, block_n=bn))
            res.append({"kernel": "conv3x3", "name": name, "bn": bn, "ms": t, "tflops": 2 * n * H * W * Co * 9 * Cc / t / 1e9})
    for name, (nseq, L, H) in {} if only not in ("all", "attn") else {"enc_attn": (V, 1370, 16), "frame_attn": (V, 1369, 12), "global_attn": (1, 1369 * V + 1, 12)}.items():
        D = H * 64
        qkv = torch.randn(nseq * L, 3 * D, device="cuda").bfloat16()
        o = torch.empty(nseq * L, D, device="cuda", dtype=torch.bfloat16)
        t = timeit(lambda: ops.attention(qkv[:, :D], qkv[:, D:2 * D], qkv[:, 2 * D:], o, num_heads=H, num_seqs=nseq, q_len=L, kv_len=L))
        fl = 4 * nseq * H * L * L * 64
        res.append({"kernel": "attn", "name": name, "nseq": nseq, "L": L, "H": H, "ms": t, "tflops": fl / t / 1e9})
        if len(sys.argv) > 3 and sys.argv[3] == "nosdpa":
            continue
        q4 = qkv.view(nseq, L, 3, H, 64).permute(2, 0, 3, 1, 4)
        t = timeit(lambda: torch.nn.functional.scaled_dot_product_attention(q4[0], q4[1], q4[2]))
        res.append({"kernel": "sdpa", "name": name, "ms": t, "tflops": fl / t / 1e9})
    for r in res:
        print(json.dumps(r))


if __name__ == "__main__":
    main()
