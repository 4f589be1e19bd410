"""Short-sequence attention: correctness against F.scaled_dot_product_attention and TFLOP/s.  Each shape runs on v5 when its
(query tile x head x sequence) items number at least 6 per SM, on v3 otherwise (ma_attention_fwd_ex); the kernel is printed.
python tools/check_attn_v5.py"""
import json
import sys

import torch
import torch.nn.functional as F

sys.path.insert(0, "map-anything_b200")
from mapanything_b200 import ops  # noqa: E402

sms = torch.cuda.get_device_properties(0).multi_processor_count
for nseq, L, H in ((8, 1370, 16), (8, 1369, 12), (3, 1369, 12), (24, 1370, 16), (5, 700, 12), (40, 257, 8), (2, 4096, 16)):
    D = H * 64
    g = torch.Generator(device="cuda").manual_seed(nseq * 1000 + L + H)
    qkv = (torch.randn(nseq * L, 3 * D, device="cuda", generator=g) * 1.5).bfloat16()
    out = torch.full((nseq * L, D), float("nan"), device="cuda", dtype=torch.bfloat16)

    def run():
        ops.attention(qkv[:, :D], qkv[:, D:2 * D], qkv[:, 2 * D:], out, num_heads=H, num_seqs=nseq, q_len=L, kv_len=L)

    run()
    torch.cuda.synchronize()
    q, k, v = (qkv[:, i * D:(i + 1) * D].view(nseq, L, H, 64).transpose(1, 2) for i in range(3))
    ref = F.scaled_dot_product_attention(q.float(), k.float(), v.float()).transpose(1, 2).reshape(nseq * L, D)
    err = (out.float() - ref).abs().max().item()
    finite = bool(torch.isfinite(out.float()).all())
    for _ in range(3):
        run()
    ts = []
    for _ in range(5):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(10):
            run()
        b.record()
        torch.cuda.synchronize()
        ts.append(a.elapsed_time(b) / 10)
    ms = sorted(ts)[2]
    kernel = "v5" if -(-L // 128) * H * nseq >= 6 * sms else "v3"
    print(json.dumps({"nseq": nseq, "L": L, "H": H, "kernel": kernel, "finite": finite, "max_abs_err": round(err, 5), "us": round(ms * 1e3, 1),
                      "tflops": round(4.0 * nseq * H * L * L * 64 / ms / 1e9, 1)}), flush=True)
