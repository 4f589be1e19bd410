"""Host-side argument checks of ma_attention_fwd_ex / ma_attention_merge and of their ops wrappers, run before any CUDA call.

The forward kernels write a partial softmax state as float4 rows of state_o (head h at column 64 h) and one float per (row,
head) of state_m whenever the call carries a state: STATE_IN, STATE_OUT, or a kv split (which writes partial states also
without STATE_OUT).  The merge loads state_o as float2 and stores out as bf16 pairs.  A call whose buffers break that must
be refused with MA_ERR_INVALID naming the operand instead of being launched.  The C side cannot see tensor widths, so
ops.attention / ops.attention_merge refuse views narrower than heads*64 columns, or with fewer rows than the call writes.

The C calls pass fake, never dereferenced device addresses.  They are made only where no CUDA device is visible: if a check
were missing, the call would go on to the launch, and on a GPU box that would run a kernel on those addresses."""
import ctypes

import pytest
import torch

pytestmark = pytest.mark.skipif(torch.cuda.is_available(), reason="passes fake device addresses; host-only check")

BASE = 1 << 32  # fake device addresses, 16-byte aligned
Q, K, V, OUT, SO, SM = (BASE + i * (1 << 26) for i in range(6))
H, D = 2, 128               # heads, heads * 64
LQ, LK = 300, 5000          # 40 kv tiles of 128 keys: kv_split up to 40
MA_ERR_INVALID = -1
MA_ATTN_STATE_IN, MA_ATTN_STATE_OUT = 1, 2


def _lib():
    from mapanything_b200 import _lib

    if not _lib.LIB_PATH.exists():
        pytest.skip("library not built (python map-anything_b200/build.py)")
    return _lib


def _fwd(*, flags=0, kv_split=2, state_o=SO, ld_state_o=D, state_m=SM, out=OUT):
    lib = _lib()
    ext = lib.AttnExt()
    ext.flags, ext.kv_split, ext.kv_split_from = flags, kv_split, 0
    ext.state_o, ext.ld_state_o, ext.state_m = state_o, ld_state_o, state_m
    ext.split_stride_o, ext.split_stride_m = LQ * D, LQ * H
    rc = lib.load().ma_attention_fwd_ex(Q, D, LQ, 0, K, D, LK, 0, V, D, 0, out, D, 0, 1, H, LQ, LK, LQ, LK, 0.125,
                                        ctypes.byref(ext), None)
    return rc, lib.load().ma_last_error().decode()


def _merge(*, state_o=SO, ld_state_o=D, state_m=SM, out=OUT, ldo=D):
    lib = _lib().load()
    rc = lib.ma_attention_merge(state_o, ld_state_o, LQ * D, state_m, LQ * H, 2, LQ, H, 0.125, out, ldo, -1, None)
    return rc, lib.ma_last_error().decode()


# (call, arguments, text the error must contain).  Each case is legal except for the one bad operand.
REFUSED = {
    "split_ld_state_o_plus2": (_fwd, dict(ld_state_o=D + 2), "ld_state_o"),
    "split_state_o_off8": (_fwd, dict(state_o=SO + 8), "state_o not 16-byte aligned"),
    "split_ld_state_o_short": (_fwd, dict(ld_state_o=D - 64), "ld_state_o"),
    "split_state_m_off2": (_fwd, dict(state_m=SM + 2), "state_m not 4-byte aligned"),
    "state_out_state_m_off2": (_fwd, dict(flags=MA_ATTN_STATE_OUT, kv_split=1, state_m=SM + 2), "state_m not 4-byte aligned"),
    "merge_state_o_off4": (_merge, dict(state_o=SO + 4), "state_o not 8-byte aligned"),
    "merge_state_m_off2": (_merge, dict(state_m=SM + 2), "state_m not 4-byte aligned"),
    "merge_out_off2": (_merge, dict(out=OUT + 2), "out not 4-byte aligned"),
    "merge_ld_state_o_short": (_merge, dict(ld_state_o=D - 64), "ld_state_o"),
    "merge_ldo_short": (_merge, dict(ldo=D - 64), "ldo"),
}


@pytest.mark.parametrize("case", sorted(REFUSED))
def test_refuses_bad_state_or_output_buffer(case):
    call, kw, text = REFUSED[case]
    rc, msg = call(**kw)
    assert rc == MA_ERR_INVALID, f"{case}: accepted ({rc}: {msg})"
    assert text in msg, msg


@pytest.mark.parametrize("call,kw", [
    (_fwd, dict()),                                                    # kv split, partial states only
    (_fwd, dict(flags=MA_ATTN_STATE_OUT, kv_split=1, out=None)),
    (_fwd, dict(flags=MA_ATTN_STATE_IN, kv_split=1, ld_state_o=D + 4)),
    (_merge, dict()),
    (_merge, dict(state_o=SO + 8, out=OUT + 4, ld_state_o=D + 2, ldo=D + 2)),
])
def test_legal_buffers_pass_the_checks(call, kw):
    """Control: legal buffers get past the checks, and the call then fails only for want of a device."""
    rc, msg = call(**kw)
    assert rc != 0
    for text in ("state_o", "state_m", "ld_state_o", "ldo", "aligned", "heads*64"):
        assert text not in msg, msg


# ---- ops wrappers: CPU tensors, refused before the library is called -----------------------------------------------


def _qkvo(rows=LQ, cols=D):
    return [torch.zeros(rows, cols, dtype=torch.bfloat16) for _ in range(4)]


def _attention(**kw):
    from mapanything_b200 import ops

    q, k, v, out = _qkvo()
    args = dict(q=q, k=k, v=v, out=out, num_heads=H, num_seqs=1, q_len=LQ, kv_len=LQ)
    args.update(kw)
    q, k, v, out = args.pop("q"), args.pop("k"), args.pop("v"), args.pop("out")
    return ops.attention(q, k, v, out, **args)


@pytest.mark.parametrize("operand", ["q", "k", "v", "out"])
def test_ops_attention_refuses_narrow_operand(operand):
    wide = torch.zeros(LQ, 2 * D, dtype=torch.bfloat16)
    with pytest.raises(ValueError, match=f"{operand} has {D - 64} columns"):
        _attention(**{operand: wide[:, :D - 64]})


def test_ops_attention_refuses_short_out():
    """Two sequences 200 rows apart: the second one's query rows end at row 200 + 150 = 350."""
    q, k, v, _ = _qkvo(rows=400)
    out = torch.zeros(349, D, dtype=torch.bfloat16)
    with pytest.raises(ValueError, match="out has 349 rows, the call writes 350"):
        _attention(q=q, k=k, v=v, out=out, num_seqs=2, q_len=150, kv_len=150, q_seq_stride=200, kv_seq_stride=200)


def test_ops_attention_refuses_narrow_state():
    so = torch.zeros(2, LQ, 2 * D)[:, :, :D - 64]
    sm = torch.full((2, LQ, H), float("-inf"))
    with pytest.raises(ValueError, match=f"state_o has {D - 64} columns"):
        _attention(state=(so, sm), kv_split=2, kv_len=LQ)


def _merge_ops(so, sm, out):
    from mapanything_b200 import ops

    return ops.attention_merge((so, sm), out, num_heads=H)


def test_ops_attention_merge_refuses_narrow_out():
    out = torch.zeros(LQ, 2 * D, dtype=torch.bfloat16)[:, :D - 64]
    with pytest.raises(ValueError, match=f"out has {D - 64} columns"):
        _merge_ops(torch.zeros(2, LQ, D), torch.zeros(2, LQ, H), out)


def test_ops_attention_merge_refuses_narrow_state():
    so = torch.zeros(2, LQ, 2 * D)[:, :, :D - 64]
    with pytest.raises(ValueError, match="state_o is"):
        _merge_ops(so, torch.zeros(2, LQ, H), torch.zeros(LQ, D, dtype=torch.bfloat16))


@pytest.mark.parametrize("short", ["state_o", "state_m"])
def test_ops_attention_merge_refuses_short_state(short):
    """out has LQ rows; a state with LQ - 1 rows would be read past its end."""
    so = torch.zeros(2, LQ - (short == "state_o"), D)
    sm = torch.zeros(2, LQ - (short == "state_m"), H)
    with pytest.raises(ValueError, match=short):
        _merge_ops(so, sm, torch.zeros(LQ, D, dtype=torch.bfloat16))
