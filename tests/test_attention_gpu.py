"""GPU parity tests for the tcgen05 flash attention (ma_attention_fwd) against fp32 PyTorch softmax attention."""
import pytest
import torch

pytestmark = pytest.mark.gpu


def _ref(qkv, nseq, L, H, q_stride=None):
    D = H * 64
    q_stride = q_stride or L
    outs = []
    for s in range(nseq):
        blk = qkv[s * q_stride : s * q_stride + L].float()
        q, k, v = blk[:, :D], blk[:, D : 2 * D], blk[:, 2 * D :]
        q = q.view(L, H, 64).transpose(0, 1)
        k = k.view(L, H, 64).transpose(0, 1)
        v = v.view(L, H, 64).transpose(0, 1)
        a = torch.softmax(q @ k.transpose(1, 2) / 8.0, dim=-1)
        outs.append((a @ v).transpose(0, 1).reshape(L, D))
    return outs


# the last four shapes have >= 6 x 148 (query tile, head, sequence) items: the persistent two-stream kernel (v5) with 11, 3, 2
# and 1 key steps per item; the others run on v3 / v2
@pytest.mark.parametrize("nseq,L,H", [(1, 128, 1), (1, 256, 2), (2, 1370, 16), (3, 1369, 12), (1, 2739, 12), (1, 100, 4),
                                      (8, 1370, 16), (40, 257, 8), (40, 200, 12), (60, 100, 16)])
def test_attention_self(nseq, L, H):
    from mapanything_b200 import ops

    D = H * 64
    g = torch.Generator(device="cuda").manual_seed(nseq * 1000 + L + H)
    qkv = (torch.randn(nseq * L, 3 * D, device="cuda", generator=g) * 1.5).bfloat16()
    out = torch.full((nseq * L, D), float("nan"), device="cuda", dtype=torch.bfloat16)
    ops.attention(qkv[:, :D], qkv[:, D : 2 * D], qkv[:, 2 * D :], out, num_heads=H, num_seqs=nseq, q_len=L, kv_len=L)
    torch.cuda.synchronize()
    refs = _ref(qkv, nseq, L, H)
    for s in range(nseq):
        got = out[s * L : (s + 1) * L].float()
        assert torch.isfinite(got).all(), f"non-finite output in seq {s}"
        err = (got - refs[s]).abs().max().item()
        # |out| reaches ~6 here (values are randn * 1.5): one bf16 ulp of the output alone is 1.6e-2 .. 3.1e-2
        assert err < 3e-2, f"seq {s}: max abs err {err}"


def test_attention_frame_inside_global_buffer():
    """Frame attention over V views stored inside a (V*N+1)-row buffer: strided sequences, trailing extra token untouched."""
    from mapanything_b200 import ops

    V, N, H = 3, 1369, 12
    D = H * 64
    g = torch.Generator(device="cuda").manual_seed(5)
    qkv = torch.randn(V * N + 1, 3 * D, device="cuda", generator=g).bfloat16()
    out = torch.zeros(V * N + 1, D, device="cuda", dtype=torch.bfloat16)
    ops.attention(qkv[:, :D], qkv[:, D : 2 * D], qkv[:, 2 * D :], out, num_heads=H, num_seqs=V, q_len=N, kv_len=N)
    refs = _ref(qkv, V, N, H)
    for s in range(V):
        err = (out[s * N : (s + 1) * N].float() - refs[s]).abs().max().item()
        assert err < 2e-2, f"view {s}: {err}"
    assert out[-1].abs().max().item() == 0.0


def test_attention_cross_lengths():
    """q_len != kv_len with separate q / kv buffers (the sequence-parallel global-attention shape)."""
    from mapanything_b200 import ops

    H, Lq, Lk = 12, 700, 2739
    D = H * 64
    g = torch.Generator(device="cuda").manual_seed(6)
    q = torch.randn(Lq, D, device="cuda", generator=g).bfloat16()
    kv = torch.randn(Lk, 2 * D, device="cuda", generator=g).bfloat16()
    out = torch.empty(Lq, D, device="cuda", dtype=torch.bfloat16)
    ops.attention(q, kv[:, :D], kv[:, D:], out, num_heads=H, num_seqs=1, q_len=Lq, kv_len=Lk)
    qf = q.float().view(Lq, H, 64).transpose(0, 1)
    kf = kv[:, :D].float().view(Lk, H, 64).transpose(0, 1)
    vf = kv[:, D:].float().view(Lk, H, 64).transpose(0, 1)
    ref = (torch.softmax(qf @ kf.transpose(1, 2) / 8.0, -1) @ vf).transpose(0, 1).reshape(Lq, D)
    err = (out.float() - ref).abs().max().item()
    assert err < 2e-2, err


def _ref_cross(q, k, v, H):
    Lq, Lk = q.shape[0], k.shape[0]
    qf = q.float().view(Lq, H, 64).transpose(0, 1)
    kf = k.float().view(Lk, H, 64).transpose(0, 1)
    vf = v.float().view(Lk, H, 64).transpose(0, 1)
    return (torch.softmax(qf @ kf.transpose(1, 2) / 8.0, -1) @ vf).transpose(0, 1).reshape(Lq, H * 64)


def test_attention_kv_segments_padded_slots():
    """Keys spread over per-rank slots of a padded all-gather buffer (ragged slot lengths; NaN-free zero padding between)."""
    from mapanything_b200 import ops

    H, Lq, slot = 12, 1000, 1500
    lens = [1370, 1369, 77, 1500]
    D = H * 64
    g = torch.Generator(device="cuda").manual_seed(7)
    q = torch.randn(Lq, D, device="cuda", generator=g).bfloat16()
    kv = torch.zeros(len(lens) * slot, 2 * D, device="cuda", dtype=torch.bfloat16)
    parts = []
    for r, ln in enumerate(lens):
        blk = torch.randn(ln, 2 * D, device="cuda", generator=g).bfloat16()
        kv[r * slot:r * slot + ln] = blk
        parts.append(blk)
    dense = torch.cat(parts, 0)
    out = torch.empty(Lq, D, device="cuda", dtype=torch.bfloat16)
    ops.attention(q, kv[:, :D], kv[:, D:], out, num_heads=H, num_seqs=1, q_len=Lq, kv_len=sum(lens),
                  kv_seq_stride=kv.shape[0], kv_segments=[(r * slot, ln) for r, ln in enumerate(lens)])
    ref = _ref_cross(q, dense[:, :D], dense[:, D:], H)
    err = (out.float() - ref).abs().max().item()
    assert err < 2e-2, err


@pytest.mark.parametrize("order", [(0, 1, 2), (2, 0, 1), (2, 1)])
def test_attention_state_carry_equals_single_pass(order):
    """Local keys first (state out), remote keys later (state in): same result as one pass over the keys of `order`, in any
    order.  The resumed launch has more than 4096 keys (v2 kernel) for the three-slot orders, 2738 (v3 kernel) for (2, 1)."""
    from mapanything_b200 import ops

    H, Lq, slot = 12, 1369 * 2 + 1, 2800
    lens = [2739, 2738, 1369]
    D = H * 64
    g = torch.Generator(device="cuda").manual_seed(8)
    q = (torch.randn(Lq, D, device="cuda", generator=g) * 1.5).bfloat16()
    kv = torch.zeros(len(lens) * slot, 2 * D, device="cuda", dtype=torch.bfloat16)
    for r, ln in enumerate(lens):
        kv[r * slot:r * slot + ln] = (torch.randn(ln, 2 * D, device="cuda", generator=g) * 1.5).bfloat16()
    segs = [(r * slot, ln) for r, ln in enumerate(lens)]
    dense = torch.cat([kv[r0:r0 + ln] for r0, ln in (segs[i] for i in sorted(order))], 0)
    ref = _ref_cross(q, dense[:, :D], dense[:, D:], H)
    state = (torch.full((Lq, D), float("nan"), device="cuda"), torch.full((Lq, H), float("nan"), device="cuda"))
    first, rest = [segs[order[0]]], [segs[i] for i in order[1:]]
    ops.attention(q, kv[:, :D], kv[:, D:], None, num_heads=H, num_seqs=1, q_len=Lq, kv_len=first[0][1],
                  kv_seq_stride=kv.shape[0], kv_segments=first, state=state, state_out=True)
    out = torch.empty(Lq, D, device="cuda", dtype=torch.bfloat16)
    ops.attention(q, kv[:, :D], kv[:, D:], out, num_heads=H, num_seqs=1, q_len=Lq, kv_len=sum(l for _, l in rest),
                  kv_seq_stride=kv.shape[0], kv_segments=rest, state=state, state_in=True)
    err = (out.float() - ref).abs().max().item()
    assert torch.isfinite(out.float()).all()
    assert err < 2e-2, err


@pytest.mark.parametrize("split", [2, 3])
def test_attention_kv_split_and_merge(split):
    """kv range cut into parts (one CTA each, partial states) + ma_attention_merge == one pass."""
    from mapanything_b200 import ops

    H, Lq, Lk = 12, 1369 * 2 + 1, 1369 * 3 + 1
    D = H * 64
    g = torch.Generator(device="cuda").manual_seed(9 + split)
    q = (torch.randn(Lq, D, device="cuda", generator=g) * 1.2).bfloat16()
    kv = (torch.randn(Lk, 2 * D, device="cuda", generator=g) * 1.2).bfloat16()
    ref = _ref_cross(q, kv[:, :D], kv[:, D:], H)
    state = (torch.full((split, Lq, D), float("nan"), device="cuda"), torch.full((split, Lq, H), float("-inf"), device="cuda"))
    ops.attention(q, kv[:, :D], kv[:, D:], None, num_heads=H, num_seqs=1, q_len=Lq, kv_len=Lk, state=state, state_out=True,
                  kv_split=split)
    out = torch.empty(Lq, D, device="cuda", dtype=torch.bfloat16)
    ops.attention_merge(state, out, num_heads=H)
    assert torch.isfinite(out.float()).all()
    err = (out.float() - ref).abs().max().item()
    assert err < 2.5e-2, err

    # tail-only: slots below `first` write the final output themselves, the others leave partial states
    n_slots = -(-Lq // 256) * H
    first = n_slots - 17
    state = (torch.full((split, Lq, D), float("nan"), device="cuda"), torch.full((split, Lq, H), float("-inf"), device="cuda"))
    out2 = torch.full((Lq, D), float("nan"), device="cuda", dtype=torch.bfloat16)
    ops.attention(q, kv[:, :D], kv[:, D:], out2, num_heads=H, num_seqs=1, q_len=Lq, kv_len=Lk, state=state, kv_split=split,
                  kv_split_from=first)
    assert torch.isnan(out2.float()).any(), "split slots must not have written the output yet"
    ops.attention_merge(state, out2, num_heads=H, first_slot=first)
    assert torch.isfinite(out2.float()).all()
    err = (out2.float() - ref).abs().max().item()
    assert err < 2.5e-2, err


def _ref_rows_fp64(q_rows, k, v, H):
    """fp64 softmax attention for a few query rows: q_rows [R, H*64] bf16, k / v [L, H*64] bf16 -> [R, H*64] fp64."""
    R, L = q_rows.shape[0], k.shape[0]
    qf = q_rows.double().view(R, H, 64).transpose(0, 1)
    kf = k.double().view(L, H, 64).transpose(0, 1)
    vf = v.double().view(L, H, 64).transpose(0, 1)
    return (torch.softmax(qf @ kf.transpose(1, 2) / 8.0, -1) @ vf).transpose(0, 1).reshape(R, H * 64)


def test_attention_long_sequence_64_views():
    """One global-attention sequence of 64 * 1369 + 1 = 87617 tokens (the 8-GPU bench scene; 685 kv tiles): 256 sampled query
    rows against an fp64 softmax.  Exercises the lazy rescale and the bf16 probabilities over ~10^3 tiles."""
    from mapanything_b200 import ops

    H, L = 12, 64 * 1369 + 1
    D = H * 64
    g = torch.Generator(device="cuda").manual_seed(21)
    qkv = (torch.randn(L, 3 * D, device="cuda", generator=g) * 1.3).bfloat16()
    # a drifting score level: later keys score higher on average, so the running maximum keeps moving (forces rescales)
    qkv[:, D:2 * D] += (torch.linspace(0, 1.5, L, device="cuda")[:, None] * torch.sign(qkv[:1, :D].float())).bfloat16()
    out = torch.full((L, D), float("nan"), device="cuda", dtype=torch.bfloat16)
    ops.attention(qkv[:, :D], qkv[:, D:2 * D], qkv[:, 2 * D:], out, num_heads=H, num_seqs=1, q_len=L, kv_len=L)
    torch.cuda.synchronize()
    assert torch.isfinite(out.float()).all()
    rows = torch.randint(0, L, (256,), generator=torch.Generator().manual_seed(3)).cuda()
    rows[0], rows[1] = 0, L - 1
    ref = _ref_rows_fp64(qkv[rows, :D], qkv[:, D:2 * D], qkv[:, 2 * D:], H)
    err = (out[rows].double() - ref).abs().max().item()
    scale = ref.abs().max().item()
    print(f"\n[attention, 87617 keys] max abs err {err:.3e} (|out| max {scale:.3f})")
    assert err < 2e-2 * max(1.0, scale), err


def test_attention_sharded_protocol_100_views():
    """The sequence-parallel global attention of BASELINE config[3] as rank 0 of 8 executes it: 100 views = 136901 key rows
    in 8 padded slots, 13 * 1369 + 1 local query rows; local keys first (partial state), the 7 remote slots in a second
    launch (second partial state), ma_attention_merge.  256 sampled rows against an fp64 softmax over all 136901 keys."""
    from mapanything_b200 import ops
    from mapanything_b200.sharding import ViewShardPlan, partition_views

    H, N = 12, 1369
    D = H * 64
    plan = ViewShardPlan(partition_views(100, 8), 0, N)
    rows, slot = plan.rows(), plan.slot_rows
    g = torch.Generator(device="cuda").manual_seed(22)
    kv = torch.zeros(plan.world * slot, 2 * D, device="cuda", dtype=torch.bfloat16)
    dense = []
    for r in range(plan.world):
        blk = (torch.randn(plan.rows(r), 2 * D, device="cuda", generator=g) * 1.3).bfloat16()
        kv[r * slot:r * slot + plan.rows(r)] = blk
        dense.append(blk)
    q = (torch.randn(rows, D, device="cuda", generator=g) * 1.3).bfloat16()
    K, V = kv[:, :D], kv[:, D:]
    so = torch.empty(2, rows, D, device="cuda")
    sm = torch.full((2, rows, H), float("-inf"), device="cuda")
    common = dict(num_heads=H, num_seqs=1, q_len=rows, kv_seq_stride=kv.shape[0])
    remote = plan.remote_segments()
    ops.attention(q, K, V, None, kv_len=rows, kv_segments=plan.local_segment(), state=(so[:1], sm[:1]), state_out=True, **common)
    ops.attention(q, K, V, None, kv_len=sum(l for _, l in remote), kv_segments=remote, state=(so[1:], sm[1:]), state_out=True,
                  **common)
    out = torch.full((rows, D), float("nan"), device="cuda", dtype=torch.bfloat16)
    ops.attention_merge((so, sm), out, num_heads=H)
    torch.cuda.synchronize()
    assert torch.isfinite(out.float()).all()
    # the order of the dense keys must follow the segment order the kernel walked: local slot, then ranks 1..7
    order = [0] + [(0 + i) % plan.world for i in range(1, plan.world)]
    alld = torch.cat([dense[r] for r in order], 0)
    assert alld.shape[0] == plan.total_rows == 100 * N + 1
    pick = torch.randint(0, rows, (256,), generator=torch.Generator().manual_seed(4)).cuda()
    ref = _ref_rows_fp64(q[pick], alld[:, :D], alld[:, D:], H)
    err = (out[pick].double() - ref).abs().max().item()
    print(f"\n[sharded attention protocol, 136901 keys in 8 slots] max abs err {err:.3e}")
    assert err < 2e-2, err


@pytest.mark.parametrize("views", [3, 5, 8, 9, 12])
def test_engine_global_attention_tail_split_matches_sdpa(views):
    """Engine._attention_one_sequence (what every global block of a single-GPU scene calls): the two-tile ping-pong kernel with
    the last partial wave of CTAs split over the key range (2-4 parts, Engine._pick_tail_split) + ma_attention_merge, against
    F.scaled_dot_product_attention.  The view counts cover 2 parts (3, 8), 4 parts (5), 3 parts (12) and no split (9) on 148 SMs."""
    import torch.nn.functional as F

    from mapanything_b200 import MapAnything, tiny_config

    eng = MapAnything(**tiny_config()).to("cuda").eval().engine()
    H, D, L = 12, 768, 1369 * views + 1
    pick = eng._pick_tail_split(L, L, H)
    g = torch.Generator(device="cuda").manual_seed(100 + views)
    qkv = (torch.randn(L, 3 * D, device="cuda", generator=g) * 1.5).bfloat16()
    out = torch.full((L, D), float("nan"), device="cuda", dtype=torch.bfloat16)
    eng._attention_one_sequence(qkv[:, :D], qkv[:, D:2 * D], qkv[:, 2 * D:], out, H, L, L)
    q, k, v = (qkv[:, i * D:(i + 1) * D].view(L, H, 64).transpose(0, 1)[None] for i in range(3))
    ref = F.scaled_dot_product_attention(q.float(), k.float(), v.float())[0].transpose(0, 1).reshape(L, D)
    got = out.float()
    assert torch.isfinite(got).all(), f"non-finite output (split {pick})"
    err = (got - ref).abs().max().item()
    print(f"\n[global attention, {views} views, {L} tokens] tail split {pick}: max abs err {err:.2e}")
    assert err < 3e-2, (pick, err)
