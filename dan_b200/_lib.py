"""ctypes binding of libdan_b200.so (include/dan_b200.h).

PyTorch is used for tensor hand-off only: every call passes ``tensor.data_ptr()``
and the current CUDA stream.  There is NO fallback: if the shared library is
missing, or a tensor is not a contiguous CUDA tensor, the call raises."""
from __future__ import annotations

import ctypes
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
# DAN_B200_LIB: an alternative build of the same library (tuning experiments, tools/variant.sh)
LIB_PATH = os.environ.get("DAN_B200_LIB") or os.path.join(_HERE, "libdan_b200.so")

DAN_MAX_LAYERS = 16
DAN_MAX_DEPTH_TOTAL = 128
DAN_MATCH_DUAL = 0
DAN_MATCH_MINING = 1
# element types of the predictions of the *_typed entry points (results bit-identical to fp32 on the widened values)
DAN_DTYPE_F32 = 0
DAN_DTYPE_F16 = 1
DAN_DTYPE_BF16 = 2
PRED_DTYPES = {torch.float32: DAN_DTYPE_F32, torch.float16: DAN_DTYPE_F16, torch.bfloat16: DAN_DTYPE_BF16}

c_i32 = ctypes.c_int32
c_i64 = ctypes.c_int64
c_f32 = ctypes.c_float
c_vp = ctypes.c_void_p
c_sz = ctypes.c_size_t


class DanError(RuntimeError):
    """A libdan_b200 call returned a negative status (mirrors the TF op's InvalidArgument)."""

    def __init__(self, code, msg):
        super().__init__("libdan_b200 error %d: %s" % (code, msg))
        self.code = code


class Pyramid(ctypes.Structure):
    _fields_ = [
        ("num_layers", c_i32), ("image_h", c_i32), ("image_w", c_i32),
        ("layer_h", c_i32 * DAN_MAX_LAYERS), ("layer_w", c_i32 * DAN_MAX_LAYERS),
        ("depth", c_i32 * DAN_MAX_LAYERS), ("clip", c_i32 * DAN_MAX_LAYERS),
        ("stride", c_f32 * DAN_MAX_LAYERS),
        ("offset_h", c_f32 * DAN_MAX_LAYERS), ("offset_w", c_f32 * DAN_MAX_LAYERS),
        ("border", c_f32 * DAN_MAX_LAYERS),
        ("anchor_h", c_f32 * DAN_MAX_DEPTH_TOTAL), ("anchor_w", c_f32 * DAN_MAX_DEPTH_TOTAL),
    ]


DAN_MAX_GRIDS = 8


class EncodeParams(ctypes.Structure):
    _fields_ = [
        ("matcher", c_i32), ("ignore_threshold", c_f32), ("positive_threshold", c_f32),
        ("prior_scaling", c_f32 * 4), ("pa_scale", c_f32), ("debug", c_i32),
        ("negative_low_thres", c_f32), ("min_match", c_i32), ("stop_positive_thres", c_f32),
        ("ignore_between", c_i32), ("gt_max_first", c_i32),
        ("num_grids", c_i32), ("grid_start", c_i32 * DAN_MAX_GRIDS), ("grid_w", c_i32 * DAN_MAX_GRIDS),
        ("grid_h", c_i32 * DAN_MAX_GRIDS),
    ]


class PostprocessParams(ctypes.Structure):
    _fields_ = [
        ("num_classes", c_i32), ("image_h", c_i32), ("image_w", c_i32),
        ("select_threshold", c_f32), ("min_size", c_f32), ("keep_topk", c_i32),
        ("nms_topk", c_i32), ("nms_threshold", c_f32), ("prior_scaling", c_f32 * 4),
    ]


DAN_MAX_PEERS = 16


class PeerExchangeArgs(ctypes.Structure):
    """dan_peer_exchange of include/dan_b200.h."""
    _fields_ = [("num_destinations", c_i32), ("delta_bytes", c_i64 * DAN_MAX_PEERS), ("flag", c_vp * DAN_MAX_PEERS), ("state", c_vp)]


class RoutingLayers(ctypes.Structure):
    """dan_routing_layers of include/dan_b200.h."""
    _fields_ = [("num_layers", c_i32), ("feat_height", c_i32 * 16), ("feat_width", c_i32 * 16), ("anchor_depth", c_i32 * 16),
                ("feat_strides", c_i32 * 16)]


_SIGNATURES = {
    "dan_version": (ctypes.c_int, []),
    "dan_last_error": (ctypes.c_char_p, []),
    "dan_device_ok": (ctypes.c_int, []),
    "dan_anchor_count": (c_i64, [ctypes.POINTER(Pyramid)]),
    "dan_generate_anchors": (ctypes.c_int, [ctypes.POINTER(Pyramid), c_vp, c_vp, c_vp, c_vp, c_vp, c_vp]),
    "dan_iou_matrix": (ctypes.c_int, [c_vp, c_vp, c_vp, c_vp, c_vp, c_i32, c_vp, c_i32, c_vp, c_vp]),
    "dan_intersection_matrix": (ctypes.c_int, [c_vp, c_vp, c_vp, c_vp, c_i32, c_vp, c_i32, c_vp, c_vp]),
    "dan_match_workspace_bytes": (c_sz, [c_i32, c_i32]),
    "dan_small_mining_match": (ctypes.c_int, [c_vp, c_i32, c_i32, c_f32, c_f32, c_f32, c_i32, c_f32, c_vp, c_vp,
                                              c_vp, c_sz, c_vp]),
    "dan_dual_max_match": (ctypes.c_int, [c_vp, c_i32, c_i32, c_f32, c_f32, c_i32, c_i32, c_vp, c_vp, c_vp, c_sz, c_vp]),
    "dan_encode_workspace_bytes": (c_sz, [c_i32, c_i32, c_i32]),
    "dan_encode_batch": (ctypes.c_int, [ctypes.POINTER(EncodeParams), c_vp, c_vp, c_vp, c_vp, c_vp, c_i32, c_vp, c_vp,
                                        c_i32, c_i32, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_sz, c_vp]),
    "dan_encode_batch_profile": (ctypes.c_int, [ctypes.POINTER(EncodeParams), c_vp, c_vp, c_vp, c_vp, c_vp, c_i32, c_vp, c_vp,
                                                c_i32, c_i32, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_sz, c_vp,
                                                ctypes.POINTER(c_f32)]),
    "dan_decode_batch": (ctypes.c_int, [c_vp, c_vp, c_vp, c_vp, c_vp, c_i32, c_i32, ctypes.POINTER(c_f32), c_vp, c_vp]),
    "dan_decode_batch_typed": (ctypes.c_int, [c_i32, c_vp, c_vp, c_vp, c_vp, c_vp, c_i32, c_i32, ctypes.POINTER(c_f32), c_vp,
                                              c_vp]),
    "dan_softmax": (ctypes.c_int, [c_vp, c_i64, c_i32, c_vp, c_vp]),
    "dan_select_bboxes": (ctypes.c_int, [c_vp, c_i32, c_i32, c_vp, c_i64, c_f32, c_vp, c_vp, c_vp]),
    "dan_clip_bboxes": (ctypes.c_int, [c_vp, c_i64, c_f32, c_f32, c_vp, c_vp]),
    "dan_filter_bboxes": (ctypes.c_int, [c_vp, c_vp, c_i64, c_f32, c_vp, c_vp, c_vp]),
    "dan_bbox_convert": (ctypes.c_int, [c_vp, c_i64, c_i32, c_vp, c_vp]),
    "dan_sort_workspace_bytes": (c_sz, [c_i64, c_i32]),
    "dan_sort_bboxes": (ctypes.c_int, [c_vp, c_vp, c_i64, c_i32, c_vp, c_vp, c_vp, c_vp, c_sz, c_vp]),
    "dan_nms_workspace_bytes": (c_sz, [c_i64, c_i32]),
    "dan_nms_bboxes": (ctypes.c_int, [c_vp, c_vp, c_i64, c_i32, c_f32, c_vp, c_vp, c_vp, c_vp, c_vp, c_sz, c_vp]),
    "dan_postprocess_workspace_bytes": (c_sz, [c_i32, c_i32, c_i32, c_i32]),
    "dan_postprocess_batch": (ctypes.c_int, [ctypes.POINTER(PostprocessParams), c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp,
                                             c_i32, c_i32, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_sz, c_vp]),
    "dan_postprocess_batch_profile": (ctypes.c_int, [ctypes.POINTER(PostprocessParams), c_vp, c_vp, c_vp, c_vp, c_vp, c_vp,
                                                     c_vp, c_i32, c_i32, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_sz, c_vp,
                                                     ctypes.POINTER(c_f32)]),
    "dan_hard_negative_workspace_bytes": (c_sz, [c_i32, c_i64]),
    "dan_hard_negative_mining": (ctypes.c_int, [c_vp, c_i32, c_vp, c_vp, c_vp, c_i32, c_i64, c_f32, c_i32, c_i32, c_i32,
                                                c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_sz, c_vp]),
    "dan_routing_workspace_bytes": (c_sz, [c_i64, c_i32]),
    "dan_dynamic_anchor_routing_eval": (ctypes.c_int, [ctypes.POINTER(RoutingLayers), c_vp, c_vp, c_vp, c_vp, c_i64, c_i32,
                                                       c_vp, c_vp, c_vp, c_sz, c_vp]),
    "dan_detect_face_workspace_bytes": (c_sz, [c_i64]),
    "dan_detect_face_select": (ctypes.c_int, [c_vp, c_vp, c_i64, c_f32, c_i32, c_vp, c_vp, c_vp, c_vp, c_sz, c_vp]),
    "dan_detect_face_batch_workspace_bytes": (c_sz, [c_i64, c_i32]),
    "dan_detect_face_batch": (ctypes.c_int, [c_i32, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_i64, c_i32, ctypes.POINTER(c_f32), c_f32,
                                             c_i32, c_vp, c_vp, c_vp, c_sz, c_vp]),
    "dan_bbox_vote": (ctypes.c_int, [c_vp, c_vp, c_i32, c_i32, c_f32, c_i32, c_vp, c_vp, c_vp, c_vp, c_vp]),
    "dan_bbox_vote_workspace_bytes": (c_sz, [c_i32, c_i32]),
    "dan_bbox_vote_ws": (ctypes.c_int, [c_vp, c_vp, c_i32, c_i32, c_f32, c_i32, c_vp, c_vp, c_vp, c_vp, c_vp, c_sz, c_vp]),
    "dan_gt_handoff": (ctypes.c_int, [c_vp, c_vp, c_vp, c_vp, c_i32, c_i32, c_f32, c_f32, c_f32, c_f32, c_vp, c_vp, c_vp, c_vp,
                                      c_vp]),
    "dan_peer_alloc": (ctypes.c_int, [c_sz, ctypes.POINTER(c_vp), c_vp]),
    "dan_peer_open": (ctypes.c_int, [c_vp, ctypes.POINTER(c_vp)]),
    "dan_peer_close": (ctypes.c_int, [c_vp]),
    "dan_peer_free": (ctypes.c_int, [c_vp]),
    "dan_postprocess_batch_peers": (ctypes.c_int, [ctypes.POINTER(PostprocessParams), c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp,
                                                   c_i32, c_i32, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_sz,
                                                   ctypes.POINTER(PeerExchangeArgs), c_vp]),
    "dan_postprocess_batch_typed": (ctypes.c_int, [ctypes.POINTER(PostprocessParams), c_i32, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp,
                                                   c_vp, c_i32, c_i32, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_sz,
                                                   ctypes.POINTER(PeerExchangeArgs), c_vp, ctypes.POINTER(c_f32)]),
    "dan_wait_detections": (ctypes.c_int, [c_vp, c_vp, c_i32, c_vp]),
    "dan_nccl_load": (ctypes.c_int, [ctypes.c_char_p]),
    "dan_nccl_version": (ctypes.c_int, []),
    "dan_comm_unique_id": (ctypes.c_int, [c_vp]),
    "dan_comm_init": (ctypes.c_int, [c_vp, c_i32, c_i32, ctypes.POINTER(c_vp)]),
    "dan_comm_init_ctas": (ctypes.c_int, [c_vp, c_i32, c_i32, c_i32, ctypes.POINTER(c_vp)]),
    "dan_comm_destroy": (ctypes.c_int, [c_vp]),
    "dan_gather_detections": (ctypes.c_int, [c_vp, c_vp, c_vp, c_sz, c_vp]),
}

EXPORTED_SYMBOLS = tuple(_SIGNATURES)

_lib = None


def lib():
    """Load libdan_b200.so (fails loudly when it has not been built)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                "dan_b200: %s is missing. Build it with `python -m dan_b200.build` "
                "(nvcc, sm_100a). There is no CPU / PyTorch fallback." % LIB_PATH)
        handle = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in _SIGNATURES.items():
            fn = getattr(handle, name)
            fn.restype = res
            fn.argtypes = args
        _lib = handle
    return _lib


def check(rc):
    if rc != 0:
        raise DanError(rc, lib().dan_last_error().decode("utf-8", "replace"))


def stream_ptr():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def require_device():
    """The product path is CUDA only: refuse to run without an sm_100 device."""
    if not torch.cuda.is_available():
        raise RuntimeError("dan_b200 needs a CUDA device (sm_100a); there is no CPU fallback")


def dev_ptr(t, dtype=None, name="tensor", allow_pinned=False):
    """data_ptr() of a contiguous CUDA tensor (None -> NULL).  allow_pinned: a page-locked HOST tensor is accepted too
    (arguments the kernels may read in place over PCIe, see dan_postprocess_batch in include/dan_b200.h)."""
    if t is None:
        return ctypes.c_void_p(0)
    if not isinstance(t, torch.Tensor) or not (t.is_cuda or (allow_pinned and t.is_pinned())):
        raise TypeError("%s must be a CUDA torch.Tensor%s (no CPU fallback)" % (name, " or a pinned host tensor" if allow_pinned else ""))
    if dtype is not None and t.dtype != dtype:
        raise TypeError("%s must be %s, got %s" % (name, dtype, t.dtype))
    if not t.is_contiguous():
        raise ValueError("%s must be contiguous" % name)
    return ctypes.c_void_p(t.data_ptr())


def pred_dtype(t, name="pred"):
    """DAN_DTYPE_* code of a prediction tensor (fp32, fp16 or bf16); TypeError for any other dtype."""
    code = PRED_DTYPES.get(getattr(t, "dtype", None))
    if code is None:
        raise TypeError("%s must be float32, float16 or bfloat16, got %s" % (name, getattr(t, "dtype", type(t).__name__)))
    return code


def is_half_cuda(t):
    """A CUDA tensor of fp16 / bf16 predictions, which the typed entry points take as they are."""
    return isinstance(t, torch.Tensor) and t.is_cuda and t.dtype in (torch.float16, torch.bfloat16)


def as_f32(t, device=None):
    """Hand-off helper: move python lists / numpy arrays / tensors to a contiguous fp32 CUDA tensor."""
    if not isinstance(t, torch.Tensor):
        t = torch.as_tensor(t, dtype=torch.float32)
    if device is None:
        device = torch.device("cuda", torch.cuda.current_device())
    return t.to(device=device, dtype=torch.float32).contiguous()


class Workspace(object):
    """Grow-only device scratch buffer owned by the caller side (the library never allocates).  One buffer per
    (device, stream): a workspace is only ever used by kernels of the stream it was requested on."""

    def __init__(self):
        self._buf = None

    def get(self, nbytes, device):
        nbytes = int(nbytes)
        if self._buf is None or self._buf.numel() < nbytes or self._buf.device != device:
            self._buf = torch.empty(max(nbytes, 256), dtype=torch.uint8, device=device)
        return self._buf


class StreamWorkspaces(object):
    """Default scratch of the standalone entry points: one grow-only Workspace per (device, current stream), so that
    calls issued on different streams or devices never share scratch memory.  Inside a CUDA-graph capture the key is
    the capturing stream.  (Explicit Workspace objects, as pipeline.HotPath uses, bypass this.)"""

    def __init__(self):
        self._by_stream = {}

    def get(self, nbytes, device):
        key = (device.index if device.index is not None else torch.cuda.current_device(),
               int(torch.cuda.current_stream(device).cuda_stream))
        ws = self._by_stream.get(key)
        if ws is None:
            ws = self._by_stream[key] = Workspace()
        return ws.get(nbytes, device)
