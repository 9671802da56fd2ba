"""CPU: the decode kernel's anchor limits and head alignment are checked with the parameters, before any CUDA call, by
btpost_workspace_bytes and by every entry point -- and the GPU shape cases are named after the decode variant the
launcher selects for them."""
import ctypes as C

import pytest

from btpost import _lib
from btpost.api import num_anchors

OK, BAD_ARG, UNSUPPORTED, MISALIGNED = 0, -1, -2, -4


def _params(S, layout=_lib.LAYOUT_L2, N=None):
    p = _lib.BtParams()
    p.batch, p.nc, p.nm, p.reg_max, p.max_det, p.max_gt = 1, 3, 32, 16, 300, 32
    p.num_anchors = num_anchors(S) if N is None else N
    p.img_h = p.img_w = S
    p.proto_h = p.proto_w = S // 4
    p.layout = layout
    p.num_iou_thrs = 10
    return p


def _io(**extra):
    """Fake, 16-byte aligned device pointers for the inputs and outputs of the decode stage except `cm_pos`.  check_stage1
    looks at the head (or the raw maps) before the outputs, so a call that passes the parameter checks returns
    BT_ERR_MISALIGNED for a misaligned head and BT_ERR_BAD_ARG otherwise, from btpost_run and btpost_decode_filter
    alike: no kernel is launched on these pointers, with or without a GPU."""
    io = _lib.BtIO()
    for f in ("head", "maps0", "maps1", "maps2", "coeffs", "n_cand", "gt_count", "gt_boxes", "gt_boxes_raw", "gt_labels", "cm"):
        setattr(io, f, 4096)
    for k, v in extra.items():
        setattr(io, k, v)
    return io


def _calls(p, io):
    L = _lib.load()
    n = C.c_size_t()
    ws_rc = L.btpost_workspace_bytes(C.byref(p), C.byref(n))
    ws = n.value if ws_rc == OK else 1 << 40
    args = (C.byref(p), C.byref(io), C.c_void_p(256), C.c_size_t(ws), None)
    return ws_rc, L.btpost_run(*args), L.btpost_decode_filter(*args)


@pytest.mark.parametrize("layout,S,N", [
    (_lib.LAYOUT_L2, 672, None),        # 9261 anchors, N % 4 != 0: above the 8192 of the one-anchor-per-thread decoder
    (_lib.LAYOUT_L2, 640, 32772),       # N % 4 == 0, above 8 x 1024 x 4
    (_lib.LAYOUT_L1, 1280, None),       # 33600 anchors
])
def test_anchor_counts_above_the_limit_are_rejected_before_any_cuda_call(layout, S, N):
    p = _params(S, layout, N)
    ws_rc, run_rc, decode_rc = _calls(p, _io())
    assert (ws_rc, run_rc, decode_rc) == (UNSUPPORTED, UNSUPPORTED, UNSUPPORTED)


@pytest.mark.parametrize("layout,S,N", [
    (_lib.LAYOUT_L2, 640, 8191),
    (_lib.LAYOUT_L2, 640, 32768),
    (_lib.LAYOUT_L1, 1248, None),       # 31941 anchors, N % 4 != 0: the raw-map decoder takes four per thread anyway
])
def test_anchor_counts_at_the_limit_are_accepted(layout, S, N):
    p = _params(S, layout, N)
    # past the parameter checks, stopped by the missing cm_pos (a launch attempt would return BT_ERR_CUDA)
    assert _calls(p, _io()) == (OK, BAD_ARG, BAD_ARG)


def test_misaligned_head_is_reported_as_misaligned():
    p = _params(640)
    io = _io(head=4096 + 4)
    assert _calls(p, io) == (OK, MISALIGNED, MISALIGNED)
    q = _params(640, _lib.LAYOUT_L1)               # the raw-map layout has no head: its pointer is not looked at
    assert _calls(q, io) == (OK, BAD_ARG, BAD_ARG)


def test_unsupported_error_text_names_the_anchor_limit():
    msg = _lib.load().btpost_error_string(UNSUPPORTED).decode()
    assert "32768" in msg and "8192" in msg and "anchors" in msg
    assert "head" in _lib.load().btpost_error_string(MISALIGNED).decode()


def decode_variant(layout, bf16, S):
    """launch_decode_filter's choice (csrc/decode_filter.cu): the block covers one eighth of the anchors in one pass,
    in groups of VEC anchors, rounded up to whole warps."""
    N = num_anchors(S)
    block = lambda v: ((-(-N // v) + 7) // 8 + 31) // 32 * 32
    if layout == "l1":
        if block(4) <= 320:
            return (4, 320)
        return (2, 1024) if block(2) <= 1024 else (4, 1024)
    vec = 4 if N % 4 == 0 else 1
    if not bf16 and vec == 4 and block(4) <= 288:
        return (4, 288)
    return (vec, 320 if block(vec) <= 320 else 1024)


def test_gpu_shape_cases_select_the_variant_they_name():
    from test_gpu_shapes import CASES
    seen = set()
    for name, layout, bf16, S, _, _ in CASES:
        vec, maxt = decode_variant(layout, bf16, S)
        assert name.startswith(f"{layout}-{'bf16' if bf16 else 'f32'}-vec{vec}-{maxt}"), name
        seen.add((layout, bf16, vec, maxt))
        pw = S // 4
        if "pw16" in name or "pw24" in name:
            assert pw % 32 == int(name.split("-pw")[1]), name
        if "tinytile" in name:
            assert pw < 32 and num_anchors(S) < 8 * 8
    # every instantiation the launcher can select, except the ones the suite already runs at 160^2 / 640^2 / 1024^2
    assert seen >= {("l2", False, 1, 320), ("l2", False, 4, 288), ("l2", False, 1, 1024), ("l2", False, 4, 320),
                    ("l2", True, 1, 320), ("l2", True, 1, 1024), ("l2", True, 4, 1024),
                    ("l1", False, 2, 1024), ("l1", False, 4, 1024), ("l1", True, 2, 1024), ("l1", True, 4, 1024)}
