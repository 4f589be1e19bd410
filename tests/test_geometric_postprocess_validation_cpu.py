"""Host-side argument checks of the geometric-input and post-processing kernels (csrc/geometric_inputs.cu,
csrc/postprocess.cu) that run before any CUDA call.

fuse_add loads and stores float4 through feat, dense_a, dense_b and g0..g3, so each of them that is present must be 16-byte
aligned.  apply_mask reads in[px * in_stride + in_offset + c] for c < width: a negative in_offset, or in_offset + width past
in_stride, reads the neighbouring pixel or past the buffer.  unshuffle_split divides H and W by patch, so patch = 0 must be
refused before the division.  A call that breaks one of these rules must be refused with MA_ERR_INVALID naming the operand
instead of being launched.

The calls pass fake, never dereferenced device addresses.  They are made only where no CUDA device is visible: if a check
were missing, the call would go on to the launch, and on a GPU box that would run a kernel on those addresses."""
import subprocess
import sys
from pathlib import Path

import pytest
import torch

pytestmark = pytest.mark.skipif(torch.cuda.is_available(), reason="passes fake device addresses; host-only check")

BASE = 1 << 32  # fake device addresses, 16-byte aligned
FEAT, DA, AS, DB, BS, G0, G1, G2, G3, GW, IN, MASK, OUT, FAC = (BASE + i * (1 << 28) for i in range(14))
MA_ERR_INVALID = -1
ROOT = Path(__file__).resolve().parents[1]


def _lib():
    from mapanything_b200 import _lib

    if not _lib.LIB_PATH.exists():
        pytest.skip("library not built (python map-anything_b200/build.py)")
    return _lib.load()


def _call(fn, *args):
    lib = _lib()
    rc = getattr(lib, fn)(*args)
    return rc, lib.ma_last_error().decode()


def fuse_add(*, feat=FEAT, dense_a=DA, dense_b=DB, g0=G0, g1=G1, g2=G2, g3=G3, C=1024):
    a_slot = AS if dense_a else None
    b_slot = BS if dense_b else None
    gw = GW if (g0 or g1 or g2 or g3) else None
    return _call("ma_fuse_add", feat, 4, 1369, C, dense_a, a_slot, dense_b, b_slot, g0, g1, g2, g3, gw, None)


def apply_mask(*, in_stride=3, in_offset=0, width=3):
    return _call("ma_apply_mask", IN, in_stride, in_offset, MASK, OUT, 518 * 518, width, None)


def unshuffle(*, patch=14, H=518, W=518, cpad=592):
    return _call("ma_unshuffle_split", IN, OUT, 2, H, W, 3, patch, cpad, 0, None, None)


# (call, arguments, start of the error message).  Each case is legal except for the one bad operand.
REFUSED = {
    "fuse_add_feat_off4": (fuse_add, dict(feat=FEAT + 4), "ma_fuse_add: feat not 16-byte aligned"),
    "fuse_add_dense_a_off8": (fuse_add, dict(dense_a=DA + 8), "ma_fuse_add: dense_a not 16-byte aligned"),
    "fuse_add_dense_b_off4": (fuse_add, dict(dense_b=DB + 4), "ma_fuse_add: dense_b not 16-byte aligned"),
    "fuse_add_g0_off4": (fuse_add, dict(g0=G0 + 4), "ma_fuse_add: g0 not 16-byte aligned"),
    "fuse_add_g1_off12": (fuse_add, dict(g1=G1 + 12), "ma_fuse_add: g1 not 16-byte aligned"),
    "fuse_add_g2_off8": (fuse_add, dict(g2=G2 + 8), "ma_fuse_add: g2 not 16-byte aligned"),
    "fuse_add_g3_off4": (fuse_add, dict(g3=G3 + 4), "ma_fuse_add: g3 not 16-byte aligned"),
    "fuse_add_g3_off4_alone": (fuse_add, dict(dense_a=None, g0=None, g1=None, g2=None, g3=G3 + 4),
                               "ma_fuse_add: g3 not 16-byte aligned"),
    "apply_mask_offset_past_stride": (apply_mask, dict(in_stride=3, in_offset=1, width=3), "ma_apply_mask: in_offset"),
    "apply_mask_offset_width_past_stride": (apply_mask, dict(in_stride=3, in_offset=2, width=2), "ma_apply_mask: in_offset"),
    "apply_mask_negative_offset": (apply_mask, dict(in_stride=3, in_offset=-1, width=1), "ma_apply_mask: in_offset"),
}


@pytest.mark.parametrize("case", sorted(REFUSED))
def test_refuses_misaligned_or_out_of_pixel_operand(case):
    call, kw, want = REFUSED[case]
    rc, msg = call(**kw)
    assert rc == MA_ERR_INVALID, f"{case}: accepted ({msg})"
    assert msg.startswith(want), msg


def test_unshuffle_split_refuses_patch_zero():
    """patch = 0 must come back as MA_ERR_INVALID, not as an integer division by zero in H % patch.  Run in a child
    process, so that a library that divides first fails this test instead of killing the test session."""
    code = (
        "import sys\n"
        f"sys.path[:0] = [{str(ROOT)!r}, {str(ROOT / 'map-anything_b200')!r}]\n"
        "from mapanything_b200 import _lib\n"
        "lib = _lib.load()\n"
        f"rc = lib.ma_unshuffle_split({IN}, {OUT}, 2, 518, 518, 3, 0, 592, 0, None, None)\n"
        "print(rc, lib.ma_last_error().decode())\n"
    )
    _lib()
    res = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=300)
    assert res.returncode == 0, f"the call killed the process (exit code {res.returncode}): {res.stderr[-500:]}"
    rc, _, msg = res.stdout.strip().partition(" ")
    assert int(rc) == MA_ERR_INVALID, res.stdout
    assert msg.startswith("ma_unshuffle_split: patch"), msg


# Legal edge operands: each gets past the checks and then fails for want of a device, not of alignment or range.
ACCEPTED = {
    "apply_mask_depth_z_from_pts3d_cam": (apply_mask, dict(in_stride=3, in_offset=2, width=1)),
    "apply_mask_full_pixel": (apply_mask, dict(in_stride=3, in_offset=0, width=3)),
    "fuse_add_dense_a_only": (fuse_add, dict(dense_b=None, g0=None, g1=None, g2=None, g3=None)),
    "fuse_add_view_pe": (fuse_add, dict(dense_a=None, dense_b=None, g1=None, g2=None, g3=None, C=768)),
    "fuse_add_feat_only": (fuse_add, dict(dense_a=None, dense_b=None, g0=None, g1=None, g2=None, g3=None, C=4)),
    "fuse_add_depth_without_pose": (fuse_add, dict(dense_a=None, g0=None, g1=None, g2=None)),
    "unshuffle_patch1": (unshuffle, dict(patch=1, H=37, W=21, cpad=8)),
}


@pytest.mark.parametrize("case", sorted(ACCEPTED))
def test_legal_edge_operands_pass_the_checks(case):
    call, kw = ACCEPTED[case]
    rc, msg = call(**kw)
    assert rc != 0, f"{case}: launched without a device"
    assert "aligned" not in msg and "in_offset" not in msg and "bad" not in msg and "patch" not in msg, msg
