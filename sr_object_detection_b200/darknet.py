"""Python mirror of the drop-in C API (include/darknet_b200.h), via ctypes.

Same names, argument meaning and by-value struct passing as the C header, so the parity tests
read like calls into the reference's own API:

    net = dn.parse_network_cfg("yolo-voc.cfg"); dn.load_weights(net, "yolo-voc.weights")
    out = dn.network_predict(net, images)           # numpy fp32 [B][outputs]
    boxes, probs = dn.get_region_boxes(net, b, thresh)
    dn.do_nms_sort(boxes, probs, nms)

Everything executes in libyolo2_b200.so on the GPU; nothing here computes.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

from . import _lib

_fp = C.POINTER(C.c_float)
_ip = C.POINTER(C.c_int)


class Tree(C.Structure):
    _fields_ = [("leaf", _ip), ("n", C.c_int), ("parent", _ip), ("group", _ip),
                ("name", C.POINTER(C.c_char_p)), ("groups", C.c_int), ("group_size", _ip),
                ("group_offset", _ip)]


class Box(C.Structure):
    _fields_ = [("x", C.c_float), ("y", C.c_float), ("w", C.c_float), ("h", C.c_float)]


class Layer(C.Structure):
    pass


class NetworkState(C.Structure):
    pass


_FWD = C.c_void_p  # function pointers are opaque on the Python side

Layer._fields_ = [
    ("type", C.c_int), ("activation", C.c_int), ("cost_type", C.c_int),
    ("forward", _FWD), ("forward_gpu", _FWD),
    ("batch_normalize", C.c_int), ("batch", C.c_int), ("flipped", C.c_int),
    ("inputs", C.c_int), ("outputs", C.c_int),
    ("h", C.c_int), ("w", C.c_int), ("c", C.c_int),
    ("out_h", C.c_int), ("out_w", C.c_int), ("out_c", C.c_int),
    ("n", C.c_int), ("groups", C.c_int),
    ("size", C.c_int), ("stride", C.c_int), ("pad", C.c_int), ("reverse", C.c_int),
    ("index", C.c_int), ("binary", C.c_int), ("xnor", C.c_int),
    ("softmax", C.c_int), ("classes", C.c_int), ("coords", C.c_int),
    ("max_boxes", C.c_int), ("log", C.c_int), ("sqrt", C.c_int), ("rescore", C.c_int),
    ("bias_match", C.c_int), ("random", C.c_int), ("absolute", C.c_int), ("classfix", C.c_int),
    ("jitter", C.c_float), ("thresh", C.c_float),
    ("coord_scale", C.c_float), ("object_scale", C.c_float), ("noobject_scale", C.c_float),
    ("class_scale", C.c_float), ("temperature", C.c_float), ("dot", C.c_float),
    ("dontload", C.c_int), ("dontloadscales", C.c_int), ("adam", C.c_int),
    ("softmax_tree", C.POINTER(Tree)), ("map", _ip), ("cost", _fp),
    ("biases", _fp), ("scales", _fp), ("weights", _fp), ("rolling_mean", _fp),
    ("rolling_variance", _fp), ("m", _fp), ("v", _fp), ("input_layers", _ip), ("input_sizes", _ip),
    ("output", _fp), ("workspace_size", C.c_size_t),
    ("output_gpu", _fp), ("weights_gpu", _fp), ("biases_gpu", _fp), ("scales_gpu", _fp),
    ("b200", C.c_void_p),
]


class Network(C.Structure):
    _fields_ = [
        ("workspace", _fp), ("n", C.c_int), ("batch", C.c_int), ("seen", _ip), ("epoch", C.c_float),
        ("subdivisions", C.c_int), ("momentum", C.c_float), ("decay", C.c_float),
        ("layers", C.POINTER(Layer)), ("outputs", C.c_int), ("output", _fp), ("policy", C.c_int),
        ("learning_rate", C.c_float), ("gamma", C.c_float), ("scale", C.c_float), ("power", C.c_float),
        ("time_steps", C.c_int), ("step", C.c_int), ("max_batches", C.c_int),
        ("scales", _fp), ("steps", _ip), ("num_steps", C.c_int), ("burn_in", C.c_int),
        ("adam", C.c_int), ("B1", C.c_float), ("B2", C.c_float), ("eps", C.c_float),
        ("inputs", C.c_int), ("h", C.c_int), ("w", C.c_int), ("c", C.c_int),
        ("max_crop", C.c_int), ("min_crop", C.c_int),
        ("angle", C.c_float), ("aspect", C.c_float), ("exposure", C.c_float),
        ("saturation", C.c_float), ("hue", C.c_float),
        ("gpu_index", C.c_int), ("hierarchy", C.POINTER(Tree)),
        ("input_gpu", C.POINTER(_fp)), ("truth_gpu", C.POINTER(_fp)),
        ("b200", C.c_void_p),
    ]


NetworkState._fields_ = [("truth", _fp), ("input", _fp), ("delta", _fp), ("workspace", _fp),
                         ("train", C.c_int), ("index", C.c_int), ("net", Network)]


class Detection(C.Structure):
    _fields_ = [("x", C.c_float), ("y", C.c_float), ("w", C.c_float), ("h", C.c_float),
                ("prob", C.c_float), ("obj_id", C.c_int), ("box_index", C.c_int)]


class ClassHit(C.Structure):
    """Mirror of `y2_class_hit`: one (index, probability) pair of a classify result."""
    _fields_ = [("index", C.c_int), ("prob", C.c_float)]


class BBox(C.Structure):
    """Mirror of `y2_bbox` (bbox_t): a tracked box in frame pixels."""
    _fields_ = [("x", C.c_uint), ("y", C.c_uint), ("w", C.c_uint), ("h", C.c_uint), ("prob", C.c_float),
                ("obj_id", C.c_uint), ("track_id", C.c_uint)]


FrameDesc = _lib.FrameDesc
FRAME_RGB24, FRAME_BGR24, FRAME_NV12 = 0, 1, 2  # y2_frame_desc.format
Tiling = _lib.Tiling
TILE_MAX = 16  # Y2_TILE_MAX: most columns or rows of a tiling


class Image(C.Structure):
    _fields_ = [("h", C.c_int), ("w", C.c_int), ("c", C.c_int), ("data", _fp)]


# LAYER_TYPE values (layer.h:13-38)
CONVOLUTIONAL, DECONVOLUTIONAL, CONNECTED, MAXPOOL, SOFTMAX, DETECTION, DROPOUT, CROP, ROUTE, COST, \
    NORMALIZATION, AVGPOOL, LOCAL, SHORTCUT, ACTIVE, RNN, GRU, CRNN, BATCHNORM, NETWORK, XNOR, REGION, \
    REORG, BLANK = range(24)

# ACTIVATION (activations.h:6-8)
LOGISTIC, RELU, RELIE, LINEAR, RAMP, TANH, PLSE, LEAKY, ELU, LOGGY, STAIR, HARDTAN, LHTAN = range(13)


class Dim3(C.Structure):
    """dim3 as returned by cuda_gridsize (cuda.c:51-62)."""
    _fields_ = [("x", C.c_uint), ("y", C.c_uint), ("z", C.c_uint)]


_declared = False


def lib() -> C.CDLL:
    global _declared
    l = _lib.load()
    if _declared:
        return l
    fp, i, f = _fp, C.c_int, C.c_float
    sig = {
        "parse_network_cfg": (Network, [C.c_char_p]),
        "load_weights": (None, [C.POINTER(Network), C.c_char_p]),
        "load_weights_upto": (None, [C.POINTER(Network), C.c_char_p, i]),
        "save_weights": (None, [Network, C.c_char_p]),
        "free_network": (None, [Network]),
        "network_predict": (fp, [Network, fp]),
        "get_network_output": (fp, [Network]),
        "get_network_output_layer": (fp, [Network, i]),
        "get_network_output_size": (i, [Network]),
        "get_network_input_size": (i, [Network]),
        "set_batch_network": (None, [C.POINTER(Network), i]),
        "resize_network": (i, [C.POINTER(Network), i, i]),
        "get_region_boxes": (None, [Layer, i, i, f, C.POINTER(fp), C.POINTER(Box), i, _ip]),
        "do_nms_sort": (None, [C.POINTER(Box), C.POINTER(fp), i, i, f]),
        "box_iou": (f, [Box, Box]),
        "cuda_set_device": (None, [i]),
        "network_upload_input": (None, [Network, fp]),
        "network_forward_device": (None, [Network]),
        "network_detect_device": (None, [Network, f, f, C.POINTER(Detection), _ip, i]),
        "network_detect_batch": (None, [Network, fp, f, f, C.POINTER(Detection), _ip, i]),
        "network_pipeline_staging": (fp, [Network, i]),
        "network_pipeline_next_slot": (i, [Network]),
        "network_detect_submit": (i, [Network, fp, f, f, i]),
        "network_detect_wait": (i, [Network, C.POINTER(Detection), _ip, i]),
        "network_detect_submit_resident": (i, [Network, f, f, i]),
        "network_pipeline_input_device": (C.c_void_p, [Network, i]),
        "network_pipeline_staging_u8": (C.POINTER(C.c_ubyte), [Network, i]),
        "network_detect_submit_u8": (i, [Network, C.POINTER(C.c_ubyte), f, f, i]),
        "network_detect_batch_u8": (None, [Network, C.POINTER(C.c_ubyte), f, f, C.POINTER(Detection), _ip, i]),
        "network_pipeline_staging_frames": (C.POINTER(C.c_ubyte), [Network, i, i, i]),
        "network_detect_submit_frames": (i, [Network, C.POINTER(C.c_ubyte), i, i, f, f, i]),
        "network_detect_batch_frames": (None, [Network, C.POINTER(C.c_ubyte), i, i, f, f, C.POINTER(Detection), _ip, i]),
        "network_pipeline_staging_frame_list": (C.POINTER(C.c_ubyte), [Network, i, i, _ip, _ip,
                                                                        C.POINTER(C.c_size_t)]),
        "network_detect_submit_frame_list": (i, [Network, i, C.POINTER(C.POINTER(C.c_ubyte)), _ip, _ip, f, f, i]),
        "network_detect_batch_frame_list": (None, [Network, i, C.POINTER(C.POINTER(C.c_ubyte)), _ip, _ip, f, f,
                                                   C.POINTER(Detection), _ip, i]),
        "network_streams_open": (None, [Network, i]),
        "network_stream_reset": (None, [Network, i]),
        "network_detect_submit_streams": (i, [Network, i, _ip, C.POINTER(C.POINTER(C.c_ubyte)), _ip, _ip, f, f, i]),
        "network_detect_submit_streams_resident": (i, [Network, i, _ip, f, f, i]),
        "network_detect_batch_streams": (None, [Network, i, _ip, C.POINTER(C.POINTER(C.c_ubyte)), _ip, _ip, f, f,
                                                C.POINTER(Detection), _ip, i]),
        "network_streams_track": (None, [Network, i]),
        "network_detect_submit_streams_tracked": (i, [Network, i, _ip, C.POINTER(C.POINTER(C.c_ubyte)), _ip, _ip, f, f,
                                                       i, i]),
        "network_detect_submit_streams_tracked_resident": (i, [Network, i, _ip, _ip, _ip, f, f, i, i]),
        "network_detect_batch_streams_tracked": (None, [Network, i, _ip, C.POINTER(C.POINTER(C.c_ubyte)), _ip, _ip, f,
                                                        f, i, C.POINTER(BBox), _ip, i]),
        "network_detect_wait_tracked": (i, [Network, C.POINTER(BBox), _ip, i]),
        "network_classify_submit_frame_list": (i, [Network, i, C.POINTER(C.POINTER(C.c_ubyte)), _ip, _ip, i]),
        "network_classify_batch_frame_list": (None, [Network, i, C.POINTER(C.POINTER(C.c_ubyte)), _ip, _ip, i,
                                                     C.POINTER(ClassHit)]),
        "network_pipeline_staging_frame_descs": (C.POINTER(C.c_ubyte), [Network, i, i, C.POINTER(FrameDesc),
                                                                         C.POINTER(C.c_size_t)]),
        "network_detect_submit_frame_descs": (i, [Network, i, C.POINTER(FrameDesc), C.c_void_p, f, f, i]),
        "network_detect_batch_frame_descs": (None, [Network, i, C.POINTER(FrameDesc), C.c_void_p, f, f,
                                                    C.POINTER(Detection), _ip, i]),
        "network_detect_submit_streams_descs": (i, [Network, i, _ip, C.POINTER(FrameDesc), C.c_void_p, f, f, i]),
        "network_detect_batch_streams_descs": (None, [Network, i, _ip, C.POINTER(FrameDesc), C.c_void_p, f, f,
                                                      C.POINTER(Detection), _ip, i]),
        "network_detect_submit_streams_tracked_descs": (i, [Network, i, _ip, C.POINTER(FrameDesc), C.c_void_p, f, f,
                                                             i, i]),
        "network_detect_batch_streams_tracked_descs": (None, [Network, i, _ip, C.POINTER(FrameDesc), C.c_void_p, f,
                                                              f, i, C.POINTER(BBox), _ip, i]),
        "network_detect_submit_tiled_descs": (i, [Network, i, C.POINTER(FrameDesc), C.POINTER(Tiling), C.c_void_p, f,
                                                   f, i]),
        "network_detect_batch_tiled_descs": (None, [Network, i, C.POINTER(FrameDesc), C.POINTER(Tiling), C.c_void_p,
                                                    f, f, C.POINTER(Detection), _ip, i]),
        "network_classify_submit_frame_descs": (i, [Network, i, C.POINTER(FrameDesc), C.c_void_p, i]),
        "network_classify_batch_frame_descs": (None, [Network, i, C.POINTER(FrameDesc), C.c_void_p, i,
                                                      C.POINTER(ClassHit)]),
        "network_classify_device": (None, [Network, i, C.POINTER(ClassHit)]),
        "network_classify_batch": (None, [Network, fp, i, C.POINTER(ClassHit)]),
        "network_classify_batch_frames": (None, [Network, C.POINTER(C.c_ubyte), i, i, i, C.POINTER(ClassHit)]),
        "network_classify_submit": (i, [Network, fp, i]),
        "network_classify_submit_u8": (i, [Network, C.POINTER(C.c_ubyte), i]),
        "network_classify_submit_frames": (i, [Network, C.POINTER(C.c_ubyte), i, i, i]),
        "network_classify_submit_resident": (i, [Network, i]),
        "network_classify_wait": (i, [Network, C.POINTER(ClassHit), i]),
        "parse_network_cfg_multi": (C.POINTER(Network), [C.c_char_p, C.c_char_p, _ip, i, i]),
        "free_network_multi": (None, [C.POINTER(Network), i]),
        "network_multi_batch": (i, [C.POINTER(Network), i]),
        "network_detect_batch_multi": (None, [C.POINTER(Network), i, fp, f, f, C.POINTER(Detection), _ip, i]),
        "network_detect_batch_u8_multi": (None, [C.POINTER(Network), i, C.POINTER(C.c_ubyte), f, f, C.POINTER(Detection), _ip, i]),
        "network_detect_submit_multi": (None, [C.POINTER(Network), i, fp, f, f, i]),
        "network_detect_submit_u8_multi": (None, [C.POINTER(Network), i, C.POINTER(C.c_ubyte), f, f, i]),
        "network_detect_wait_multi": (None, [C.POINTER(Network), i, C.POINTER(Detection), _ip, i]),
        "network_sync": (None, [Network]),
        "network_stream": (C.c_void_p, [Network]),
        "network_conv_flops": (C.c_double, [Network]),
        "network_launch_count": (i, [Network]),
        "network_conv_kernel": (i, [Network, i]),
        "network_profile_layers": (i, [Network, fp, i]),
        "network_set_eager": (None, [Network, i]),
        "network_input_staging": (fp, [Network]),
        "network_input_device": (C.c_void_p, [Network]),
        "y2_bind_thread_to_device": (i, [i]),
        "resize_image": (Image, [Image, i, i]),
        "free_image": (None, [Image]),
        "letterbox_image": (Image, [Image, i, i]),
        "embed_image": (None, [Image, Image, i, i]),
        "fill_image": (None, [Image, f]),
        "top_k": (None, [fp, i, i, _ip]),
        "read_tree": (C.POINTER(Tree), [C.c_char_p]),
        "max_index": (i, [fp, i]),
        "fill_cpu": (None, [i, f, fp, i]),
        "copy_cpu": (None, [i, fp, i, fp, i]),
        "axpy_cpu": (None, [i, f, fp, i, fp, i]),
        "scal_cpu": (None, [i, f, fp, i]),
        "fill_ongpu": (None, [i, f, C.c_void_p, i]),
        "copy_ongpu": (None, [i, C.c_void_p, i, C.c_void_p, i]),
        "axpy_ongpu": (None, [i, f, C.c_void_p, i, C.c_void_p, i]),
        "scal_ongpu": (None, [i, f, C.c_void_p, i]),
        "activate": (f, [f, i]),
        "activate_array": (None, [fp, i, i]),
        "activate_array_ongpu": (None, [C.c_void_p, i, i]),
        "cuda_gridsize": (Dim3, [C.c_size_t]),
        "cuda_make_array": (C.c_void_p, [fp, C.c_size_t]),
        "cuda_push_array": (None, [C.c_void_p, fp, C.c_size_t]),
        "cuda_pull_array": (None, [C.c_void_p, fp, C.c_size_t]),
        "cuda_free": (None, [C.c_void_p]),
        "y2_abi_sizeof": (C.c_size_t, [i]),
    }
    for name, (res, args) in sig.items():
        fn = getattr(l, name)
        fn.restype = res
        fn.argtypes = args
    # the ctypes mirrors above must match the C structs exactly (by-value passing)
    assert l.y2_abi_sizeof(0) == C.sizeof(Layer), (l.y2_abi_sizeof(0), C.sizeof(Layer))
    assert l.y2_abi_sizeof(1) == C.sizeof(Network), (l.y2_abi_sizeof(1), C.sizeof(Network))
    assert l.y2_abi_sizeof(2) == C.sizeof(NetworkState)
    assert l.y2_abi_sizeof(3) == C.sizeof(Detection)
    assert l.y2_abi_sizeof(5) == C.sizeof(ClassHit)
    assert l.y2_abi_sizeof(6) == C.sizeof(BBox)
    assert l.y2_abi_sizeof(7) == C.sizeof(FrameDesc), (l.y2_abi_sizeof(7), C.sizeof(FrameDesc))
    assert l.y2_abi_sizeof(8) == C.sizeof(Tiling), (l.y2_abi_sizeof(8), C.sizeof(Tiling))
    _declared = True
    return l


def _quiet_stderr():
    """The parser prints the layer table on stderr like the reference; tests silence it."""
    class _Ctx:
        def __enter__(self):
            if os.environ.get("Y2_VERBOSE"):
                self.saved = None
                return
            import sys
            sys.stderr.flush()
            self.saved = os.dup(2)
            self.null = os.open(os.devnull, os.O_WRONLY)
            os.dup2(self.null, 2)

        def __exit__(self, *a):
            if self.saved is not None:
                os.dup2(self.saved, 2)
                os.close(self.saved)
                os.close(self.null)
    return _Ctx()


def gpu_index() -> int:
    return C.c_int.in_dll(lib(), "gpu_index").value


def set_gpu_index(v: int) -> None:
    C.c_int.in_dll(lib(), "gpu_index").value = v


def parse_network_cfg(path: str) -> Network:
    with _quiet_stderr():
        return lib().parse_network_cfg(str(path).encode())


def load_weights(net: Network, path: str) -> None:
    with _quiet_stderr():
        lib().load_weights(C.byref(net), str(path).encode())


def free_network(net: Network) -> None:
    lib().free_network(net)


def set_batch_network(net: Network, b: int) -> None:
    lib().set_batch_network(C.byref(net), b)


def resize_network(net: Network, w: int, h: int) -> int:
    with _quiet_stderr():
        return lib().resize_network(C.byref(net), w, h)


def _as_fp(a: np.ndarray):
    assert a.dtype == np.float32 and a.flags["C_CONTIGUOUS"]
    return a.ctypes.data_as(_fp)


def network_predict(net: Network, images: np.ndarray) -> np.ndarray:
    """images: fp32 [B][C][H][W]; returns a copy of the borrowed output, [B][outputs]."""
    assert images.size == net.batch * net.inputs, (images.shape, net.batch, net.inputs)
    out = lib().network_predict(net, _as_fp(images))
    n = lib().get_network_output_size(net)
    return np.ctypeslib.as_array(out, shape=(net.batch, n)).copy()


def get_network_output_layer(net: Network, i: int) -> np.ndarray:
    out = lib().get_network_output_layer(net, i)
    return np.ctypeslib.as_array(out, shape=(net.batch, net.layers[i].outputs)).copy()


def region_layer(net: Network) -> Layer:
    return net.layers[net.n - 1]


def get_region_boxes(net: Network, b: int, thresh: float, only_objectness: int = 0, use_map: bool = False,
                     w: int = 1, h: int = 1):
    """get_region_boxes on batch element b (the reference reads element 0 of l.output; callers
    advance the pointer per image, which is what this does)."""
    l = Layer.from_buffer_copy(region_layer(net))
    total = l.w * l.h * l.n
    classes = 200 if use_map else l.classes
    base = C.cast(l.output, C.c_void_p).value
    l.output = C.cast(base + b * l.outputs * 4, _fp)
    probs = np.zeros((total, classes), np.float32)
    boxes = np.zeros((total, 4), np.float32)
    rows = (_fp * total)(*[C.cast(probs.ctypes.data + j * classes * 4, _fp) for j in range(total)])
    lib().get_region_boxes(l, w, h, thresh, rows, boxes.ctypes.data_as(C.POINTER(Box)), only_objectness,
                           l.map if use_map else None)
    return boxes, probs


def do_nms_sort(boxes: np.ndarray, probs: np.ndarray, thresh: float) -> None:
    total, classes = probs.shape
    rows = (_fp * total)(*[C.cast(probs.ctypes.data + j * classes * 4, _fp) for j in range(total)])
    lib().do_nms_sort(boxes.ctypes.data_as(C.POINTER(Box)), rows, total, classes, thresh)


def network_detect_batch(net: Network, images: np.ndarray | None, thresh: float, nms: float,
                         max_det: int = 256):
    """Extension: batched forward + decode + NMS + pick; returns a list (per image) of
    structured arrays with fields x,y,w,h,prob,obj_id,box_index."""
    dets = (Detection * (net.batch * max_det))()
    counts = (C.c_int * net.batch)()
    if images is None:
        lib().network_detect_device(net, thresh, nms, dets, counts, max_det)
    else:
        lib().network_detect_batch(net, _as_fp(images), thresh, nms, dets, counts, max_det)
    arr = np.ctypeslib.as_array(dets)
    out = []
    for b in range(net.batch):
        c = min(counts[b], max_det)
        out.append(arr[b * max_det:b * max_det + c].copy())
    return out, list(counts)


def _hits_arrays(hits, batch: int, top: int):
    arr = np.ctypeslib.as_array(hits)[:batch * top].reshape(batch, top)
    return arr["index"].astype(np.int32), arr["prob"].astype(np.float32)


def _as_u8(a: np.ndarray):
    assert a.dtype == np.uint8 and a.flags["C_CONTIGUOUS"]
    return a.ctypes.data_as(C.POINTER(C.c_ubyte))


def _frame_list_args(frames):
    """(n, frame pointers, widths, heights) of a sequence of uint8 [h][w][3] arrays, for the *_frame_list entries"""
    n = len(frames)
    for a in frames:
        assert a.dtype == np.uint8 and a.ndim == 3 and a.shape[2] == 3 and a.flags["C_CONTIGUOUS"], (a.dtype, a.shape)
    ptrs = (C.POINTER(C.c_ubyte) * max(n, 1))(*[_as_u8(a) for a in frames])
    fw = (C.c_int * max(n, 1))(*[a.shape[1] for a in frames])
    fh = (C.c_int * max(n, 1))(*[a.shape[0] for a in frames])
    return n, ptrs, fw, fh


def network_pipeline_staging_frame_list(net: Network, slot: int, sizes):
    """The slot's pinned staging buffer laid out for frames of sizes [(frame_w, frame_h), ...]: one writable uint8
    [h][w][3] view per frame at its place.  Fill the views and pass them as the frame list to skip the host copy;
    they stay valid until a larger list makes the slot's buffer grow."""
    n = len(sizes)
    fw = (C.c_int * max(n, 1))(*[s[0] for s in sizes])
    fh = (C.c_int * max(n, 1))(*[s[1] for s in sizes])
    offsets = (C.c_size_t * max(n, 1))()
    base = C.cast(lib().network_pipeline_staging_frame_list(net, slot, n, fw, fh, offsets), C.c_void_p).value
    return [np.ctypeslib.as_array(C.cast(base + offsets[i], C.POINTER(C.c_ubyte)), shape=(h, w, 3))
            for i, (w, h) in enumerate(sizes)]


def _det_lists(dets, counts, n: int, max_det: int):
    arr = np.ctypeslib.as_array(dets)
    return [arr[b * max_det:b * max_det + min(counts[b], max_det)].copy() for b in range(n)], list(counts)[:n]


def network_detect_frame_list(net: Network, frames, thresh: float, nms: float, max_det: int = 256):
    """Extension: detection on a list of 1 .. batch decoded frames (uint8 [h][w][3] arrays, each of its own size),
    resized on the device.  Returns (per-image detection arrays, counts) for len(frames) images."""
    n, ptrs, fw, fh = _frame_list_args(frames)
    dets = (Detection * (max(n, 1) * max_det))()
    counts = (C.c_int * max(n, 1))()
    lib().network_detect_batch_frame_list(net, n, ptrs, fw, fh, thresh, nms, dets, counts, max_det)
    return _det_lists(dets, counts, n, max_det)


def network_detect_submit_frame_list(net: Network, frames, thresh: float, nms: float, max_det: int = 256) -> int:
    """Queue a frame list on the submit/wait pipeline; network_detect_wait_n(net, len(frames), ...) collects it."""
    n, ptrs, fw, fh = _frame_list_args(frames)
    return lib().network_detect_submit_frame_list(net, n, ptrs, fw, fh, thresh, nms, max_det)


def network_detect_wait_n(net: Network, n: int, max_det: int = 256):
    """network_detect_wait for the oldest detection batch in flight, which holds n images"""
    dets = (Detection * (net.batch * max_det))()
    counts = (C.c_int * net.batch)()
    lib().network_detect_wait(net, dets, counts, max_det)
    return _det_lists(dets, counts, n, max_det)


def network_streams_open(net: Network, max_streams: int) -> None:
    """Extension: (re)open streams 0 .. max_streams-1 for the 3-frame-mean entries, every one starting over."""
    lib().network_streams_open(net, max_streams)


def network_stream_reset(net: Network, stream: int) -> None:
    lib().network_stream_reset(net, stream)


def _stream_ids(stream_ids, n: int):
    ids = [int(s) for s in stream_ids]
    assert len(ids) == n, (len(ids), n)
    return (C.c_int * max(n, 1))(*ids)


def network_detect_streams(net: Network, stream_ids, frames, thresh: float, nms: float, max_det: int = 256):
    """Extension: detection on a list of decoded frames (uint8 [h][w][3] arrays of their own sizes), frame i from
    video stream stream_ids[i] and decoded on that stream's 3-frame mean, as Detector::detect(img, thresh,
    use_mean = true).  Returns (per-image detection arrays, counts) for len(frames) images."""
    n, ptrs, fw, fh = _frame_list_args(frames)
    dets = (Detection * (max(n, 1) * max_det))()
    counts = (C.c_int * max(n, 1))()
    lib().network_detect_batch_streams(net, n, _stream_ids(stream_ids, n), ptrs, fw, fh, thresh, nms, dets, counts,
                                       max_det)
    return _det_lists(dets, counts, n, max_det)


def network_detect_submit_streams(net: Network, stream_ids, frames, thresh: float, nms: float,
                                  max_det: int = 256) -> int:
    """Queue a streams frame list on the submit/wait pipeline; network_detect_wait_n(net, len(frames), ...) collects
    it."""
    n, ptrs, fw, fh = _frame_list_args(frames)
    return lib().network_detect_submit_streams(net, n, _stream_ids(stream_ids, n), ptrs, fw, fh, thresh, nms, max_det)


def network_detect_submit_streams_resident(net: Network, stream_ids, thresh: float, nms: float,
                                           max_det: int = 256) -> int:
    """The same with the first len(stream_ids) images already in the slot's device input
    (network_pipeline_input_device)."""
    n = len(stream_ids)
    return lib().network_detect_submit_streams_resident(net, n, _stream_ids(stream_ids, n), thresh, nms, max_det)


def network_streams_track(net: Network, frames_story: int = 6) -> None:
    """Extension: turn tracking on for the opened streams (Detector::tracking's frames_story), every track over."""
    lib().network_streams_track(net, frames_story)


def network_detect_streams_tracked(net: Network, stream_ids, frames, thresh: float, nms: float, use_mean: bool = True,
                                   max_det: int = 256):
    """Extension: as network_detect_streams, then tracked per stream as Detector::detect(img, thresh, use_mean) and
    Detector::tracking(boxes, frames_story) would.  Returns (per-image arrays with fields x, y, w, h (pixels), prob,
    obj_id, track_id; full counts) for len(frames) images."""
    n, ptrs, fw, fh = _frame_list_args(frames)
    boxes = (BBox * (max(n, 1) * max_det))()
    counts = (C.c_int * max(n, 1))()
    lib().network_detect_batch_streams_tracked(net, n, _stream_ids(stream_ids, n), ptrs, fw, fh, thresh, nms,
                                               int(use_mean), boxes, counts, max_det)
    return _det_lists(boxes, counts, n, max_det)


def network_detect_submit_streams_tracked(net: Network, stream_ids, frames, thresh: float, nms: float,
                                          use_mean: bool = True, max_det: int = 256) -> int:
    """Queue a tracked streams frame list; network_detect_wait_tracked(net, len(frames), ...) collects it."""
    n, ptrs, fw, fh = _frame_list_args(frames)
    return lib().network_detect_submit_streams_tracked(net, n, _stream_ids(stream_ids, n), ptrs, fw, fh, thresh, nms,
                                                       int(use_mean), max_det)


def network_detect_submit_streams_tracked_resident(net: Network, stream_ids, sizes, thresh: float, nms: float,
                                                   use_mean: bool = True, max_det: int = 256) -> int:
    """The same with the first len(stream_ids) images already in the slot's device input; sizes [(w, h), ...] are
    the frame sizes in pixels the boxes are scaled to."""
    n = len(stream_ids)
    assert len(sizes) == n, (len(sizes), n)
    fw = (C.c_int * max(n, 1))(*[int(s[0]) for s in sizes])
    fh = (C.c_int * max(n, 1))(*[int(s[1]) for s in sizes])
    return lib().network_detect_submit_streams_tracked_resident(net, n, _stream_ids(stream_ids, n), fw, fh, thresh,
                                                                nms, int(use_mean), max_det)


def network_detect_wait_tracked(net: Network, n: int, max_det: int = 256):
    """network_detect_wait_tracked for the oldest batch in flight, a tracked batch of n images"""
    boxes = (BBox * (net.batch * max_det))()
    counts = (C.c_int * net.batch)()
    lib().network_detect_wait_tracked(net, boxes, counts, max_det)
    return _det_lists(boxes, counts, n, max_det)


def _rows(obj, ndim_shapes):
    """(address, shape, byte strides, on_device) of a uint8 array: a numpy array (host) or any object with
    __cuda_array_interface__ (device), e.g. a torch or cupy tensor"""
    cai = getattr(obj, "__cuda_array_interface__", None)
    if cai is not None:
        if cai["typestr"] not in ("|u1", "<u1", ">u1"):
            raise ValueError(f"frame_desc: a uint8 array is needed, got typestr {cai['typestr']}")
        shape = tuple(int(v) for v in cai["shape"])
        strides = cai.get("strides")
        if strides is None:  # C-contiguous
            strides, step = [], 1
            for d in reversed(shape):
                strides.insert(0, step)
                step *= d
        addr, on_device = int(cai["data"][0]), 1
    elif isinstance(obj, np.ndarray):
        if obj.dtype != np.uint8:
            raise ValueError(f"frame_desc: a uint8 array is needed, got {obj.dtype}")
        shape, strides, addr, on_device = obj.shape, obj.strides, obj.ctypes.data, 0
    else:
        raise TypeError("frame_desc: a numpy array or an object with __cuda_array_interface__ is needed")
    shape, strides = tuple(shape), tuple(int(v) for v in strides)
    if len(shape) not in ndim_shapes or any(v <= 0 for v in shape) or any(v < 0 for v in strides):
        raise ValueError(f"frame_desc: an array of {' or '.join(map(str, ndim_shapes))} dimensions with positive "
                         f"extents and strides is needed, got shape {shape} strides {strides}")
    return addr, shape, strides, on_device


def _pitch(shape, strides, row_elems: int, what: str) -> int:
    """the row pitch of rows of row_elems interleaved bytes (the trailing axes must be dense); whether it is wide
    enough is the library's rule (y2_frame_desc_rows)"""
    dense = 1
    for d, st in zip(reversed(shape[1:]), reversed(strides[1:])):
        if d > 1 and st != dense:
            raise ValueError(f"frame_desc: {what} rows are not interleaved bytes (shape {shape}, strides {strides})")
        dense *= d
    return strides[0] if shape[0] > 1 else row_elems


# what y2_frame_desc_rows refuses, by its Y2_FRAME_BAD_* code
_FRAME_RULES = {1: "a size of 0 or less", 2: "an unknown format", 3: "NV12 needs an even width and height",
                4: "a row of more than INT_MAX bytes", 5: "rows overlap (pitch below the row's bytes)",
                6: "UV rows overlap (uv_pitch below the row's bytes)"}


def frame_desc(obj, fmt: int) -> FrameDesc:
    """A y2_frame_desc for a frame held in a numpy array (host memory) or in an object with __cuda_array_interface__
    (memory of the network's GPU, read in place).  fmt FRAME_RGB24 / FRAME_BGR24: a uint8 [h][w][3] array whose rows
    may be pitched; FRAME_NV12: one uint8 [h*3/2][w] array (the Y plane, then the interleaved UV plane) or a pair
    (y [h][w], uv [h/2][w] or [h/2][w/2][2]) on the same side.  The pitch comes from the row stride.  The descriptor
    keeps a reference to the array(s); device frames must stay unchanged until the wait that returns their batch."""
    d = FrameDesc()
    if fmt in (FRAME_RGB24, FRAME_BGR24):
        addr, shape, strides, on_device = _rows(obj, (3,))
        if shape[2] != 3:
            raise ValueError(f"frame_desc: RGB/BGR frames are [h][w][3], got shape {shape}")
        d.data, d.h, d.w = addr, shape[0], shape[1]
        d.pitch = _pitch(shape, strides, 3 * shape[1], "frame")
    elif fmt == FRAME_NV12:
        if isinstance(obj, (tuple, list)):
            y, uv = obj
            addr, shape, strides, on_device = _rows(y, (2,))
            uaddr, ushape, ustrides, uon = _rows(uv, (2, 3))
            h, w = shape
            if uon != on_device:
                raise ValueError("frame_desc: the Y and UV planes must both be host or both be device arrays")
            if ushape[0] != h // 2 or int(np.prod(ushape[1:])) != w or (len(ushape) == 3 and ushape[2] != 2):
                raise ValueError(f"frame_desc: the UV plane of a {w}x{h} NV12 frame is [h/2][w] or [h/2][w/2][2], "
                                 f"got {ushape}")
            d.uv, d.uv_pitch = uaddr, _pitch(ushape, ustrides, w, "UV")
        else:
            addr, shape, strides, on_device = _rows(obj, (2,))
            if shape[0] % 3:
                raise ValueError(f"frame_desc: a one-array NV12 frame is [h*3/2][w], got {shape}")
            h, w = shape[0] * 2 // 3, shape[1]
        d.data, d.h, d.w = addr, h, w
        d.pitch = _pitch(shape, strides, w, "Y")
    else:
        raise ValueError(f"frame_desc: unknown format {fmt}")
    d.format, d.on_device = fmt, on_device
    rc = _lib.load().y2_frame_desc_rows(C.byref(d), C.byref(_lib.FrameRows()))
    if rc:
        raise ValueError(f"frame_desc: {_FRAME_RULES.get(rc, rc)}: {d.w}x{d.h}, pitch {d.pitch}, uv_pitch "
                         f"{d.uv_pitch}, format {fmt}")
    d._keep = obj
    return d


def _descs_arg(descs):
    n = len(descs)
    return n, (FrameDesc * max(n, 1))(*descs)


def network_pipeline_staging_frame_descs(net: Network, slot: int, descs):
    """The slot's pinned staging buffer laid out for a descriptor list (only sizes, formats and on_device are read):
    per frame a writable uint8 view at its place ([h][w][3], or [h*3/2][w] for NV12), None for a device frame.  Fill
    the views and pass frame_desc(view, fmt) to skip the host copy; they stay valid until a larger list makes the
    slot's buffer grow."""
    n, arr = _descs_arg(descs)
    offsets = (C.c_size_t * max(n, 1))()
    base = C.cast(lib().network_pipeline_staging_frame_descs(net, slot, n, arr, offsets), C.c_void_p).value
    views = []
    for i, d in enumerate(descs):
        if d.on_device:
            views.append(None)
            continue
        shape = (d.h * 3 // 2, d.w) if d.format == FRAME_NV12 else (d.h, d.w, 3)
        views.append(np.ctypeslib.as_array(C.cast(base + offsets[i], C.POINTER(C.c_ubyte)), shape=shape))
    return views


def network_detect_frame_descs(net: Network, descs, thresh: float, nms: float, max_det: int = 256, ready=None):
    """Extension: detection on a list of 1 .. batch frame descriptors (frame_desc), converted to RGB and resized on
    the device.  ready: a raw cudaEvent_t (torch.cuda.Event().cuda_event) the network waits for before it reads any
    device frame.  Returns (per-image detection arrays, counts) for len(descs) images."""
    n, arr = _descs_arg(descs)
    dets = (Detection * (max(n, 1) * max_det))()
    counts = (C.c_int * max(n, 1))()
    lib().network_detect_batch_frame_descs(net, n, arr, ready, thresh, nms, dets, counts, max_det)
    return _det_lists(dets, counts, n, max_det)


def network_detect_submit_frame_descs(net: Network, descs, thresh: float, nms: float, max_det: int = 256,
                                      ready=None) -> int:
    """Queue a descriptor list on the submit/wait pipeline; network_detect_wait_n(net, len(descs), ...) collects it."""
    n, arr = _descs_arg(descs)
    return lib().network_detect_submit_frame_descs(net, n, arr, ready, thresh, nms, max_det)


def _tiling_arg(tiling):
    if tiling is None:
        return None
    if not isinstance(tiling, Tiling):
        tiling = Tiling(*tiling)
    return C.byref(tiling)


def network_detect_tiled_descs(net: Network, descs, tiling, thresh: float, nms: float, max_det: int = 256,
                               ready=None):
    """Extension: tiled detection of a list of frame descriptors (frame_desc).  Each frame goes through the network as
    the tiles of `tiling` (a Tiling, or a (cols, rows, overlap, full) tuple), and its detections are merged by
    do_nms_sort over the union of its tiles' boxes.  Returns (per-frame detection arrays relative to the frame,
    counts); box_index is the index in the frame's union (tile * l.w*l.h*l.n + box)."""
    n, arr = _descs_arg(descs)
    dets = (Detection * (max(n, 1) * max_det))()
    counts = (C.c_int * max(n, 1))()
    lib().network_detect_batch_tiled_descs(net, n, arr, _tiling_arg(tiling), ready, thresh, nms, dets, counts, max_det)
    return _det_lists(dets, counts, n, max_det)


def network_detect_submit_tiled_descs(net: Network, descs, tiling, thresh: float, nms: float, max_det: int = 256,
                                      ready=None) -> int:
    """Queue a tiled descriptor list on the submit/wait pipeline; network_detect_wait_n(net, len(descs), ...) collects
    it."""
    n, arr = _descs_arg(descs)
    return lib().network_detect_submit_tiled_descs(net, n, arr, _tiling_arg(tiling), ready, thresh, nms, max_det)


def network_detect_streams_descs(net: Network, stream_ids, descs, thresh: float, nms: float, max_det: int = 256,
                                 ready=None):
    """network_detect_streams on frame descriptors."""
    n, arr = _descs_arg(descs)
    dets = (Detection * (max(n, 1) * max_det))()
    counts = (C.c_int * max(n, 1))()
    lib().network_detect_batch_streams_descs(net, n, _stream_ids(stream_ids, n), arr, ready, thresh, nms, dets, counts,
                                             max_det)
    return _det_lists(dets, counts, n, max_det)


def network_detect_submit_streams_descs(net: Network, stream_ids, descs, thresh: float, nms: float,
                                        max_det: int = 256, ready=None) -> int:
    n, arr = _descs_arg(descs)
    return lib().network_detect_submit_streams_descs(net, n, _stream_ids(stream_ids, n), arr, ready, thresh, nms,
                                                     max_det)


def network_detect_streams_tracked_descs(net: Network, stream_ids, descs, thresh: float, nms: float,
                                         use_mean: bool = True, max_det: int = 256, ready=None):
    """network_detect_streams_tracked on frame descriptors; boxes are scaled to each descriptor's w x h."""
    n, arr = _descs_arg(descs)
    boxes = (BBox * (max(n, 1) * max_det))()
    counts = (C.c_int * max(n, 1))()
    lib().network_detect_batch_streams_tracked_descs(net, n, _stream_ids(stream_ids, n), arr, ready, thresh, nms,
                                                     int(use_mean), boxes, counts, max_det)
    return _det_lists(boxes, counts, n, max_det)


def network_detect_submit_streams_tracked_descs(net: Network, stream_ids, descs, thresh: float, nms: float,
                                                use_mean: bool = True, max_det: int = 256, ready=None) -> int:
    n, arr = _descs_arg(descs)
    return lib().network_detect_submit_streams_tracked_descs(net, n, _stream_ids(stream_ids, n), arr, ready, thresh,
                                                             nms, int(use_mean), max_det)


def network_classify_frame_descs(net: Network, descs, top: int = 5, ready=None):
    """Extension: classification of a list of frame descriptors, each converted to RGB and letterboxed on the device:
    (indices int32 [n][top], probs float32 [n][top])."""
    n, arr = _descs_arg(descs)
    hits = (ClassHit * (max(n, 1) * top))()
    lib().network_classify_batch_frame_descs(net, n, arr, ready, top, hits)
    return _hits_arrays(hits, n, top)


def network_classify_submit_frame_descs(net: Network, descs, top: int = 5, ready=None) -> int:
    """Queue a descriptor list for classification; network_classify_wait(net, top, n=len(descs)) collects it."""
    n, arr = _descs_arg(descs)
    return lib().network_classify_submit_frame_descs(net, n, arr, ready, top)


def network_classify_batch(net: Network, images: np.ndarray | None = None, frames: np.ndarray | None = None,
                           top: int = 5, frame_list=None):
    """Extension: batched forward + WordTree products + top-k on the device.  images: prepared fp32 [B][C][H][W]
    (already letterboxed); frames: uint8 RGB [B][fh][fw][3] of any size, letterboxed on the device; frame_list: a
    sequence of 1 .. B uint8 [h][w][3] arrays of their own sizes, letterboxed on the device; none: the last forward
    pass.  Returns (indices int32 [n][top], probs float32 [n][top]), best first, n = B or len(frame_list)."""
    if frame_list is not None:
        n, ptrs, fw, fh = _frame_list_args(frame_list)
        hits = (ClassHit * (max(n, 1) * top))()
        lib().network_classify_batch_frame_list(net, n, ptrs, fw, fh, top, hits)
        return _hits_arrays(hits, n, top)
    hits = (ClassHit * (net.batch * top))()
    if frames is not None:
        assert frames.ndim == 4 and frames.shape[0] == net.batch and frames.shape[3] == 3, frames.shape
        lib().network_classify_batch_frames(net, _as_u8(frames), frames.shape[2], frames.shape[1], top, hits)
    elif images is not None:
        assert images.size == net.batch * net.inputs, (images.shape, net.batch, net.inputs)
        lib().network_classify_batch(net, _as_fp(images), top, hits)
    else:
        lib().network_classify_device(net, top, hits)
    return _hits_arrays(hits, net.batch, top)


def network_classify_submit(net: Network, images: np.ndarray | None = None, frames: np.ndarray | None = None,
                            u8: np.ndarray | None = None, top: int = 5, frame_list=None) -> int:
    """Queue one batch on the submit/wait pipeline: prepared fp32 images, frames of any size, uint8 images at the
    network size (u8), a list of frames of their own sizes (frame_list; collect it with
    network_classify_wait(net, top, n=len(frame_list))), or none of them (the slot's device input already holds the
    batch).  Returns the slot."""
    if frame_list is not None:
        n, ptrs, fw, fh = _frame_list_args(frame_list)
        return lib().network_classify_submit_frame_list(net, n, ptrs, fw, fh, top)
    if frames is not None:
        return lib().network_classify_submit_frames(net, _as_u8(frames), frames.shape[2], frames.shape[1], top)
    if u8 is not None:
        return lib().network_classify_submit_u8(net, _as_u8(u8), top)
    if images is not None:
        return lib().network_classify_submit(net, _as_fp(images), top)
    return lib().network_classify_submit_resident(net, top)


def network_classify_wait(net: Network, top: int = 5, n: int | None = None):
    """The oldest classify batch in flight, which holds n images (default: the batch): (indices int32 [n][top], probs
    float32 [n][top])."""
    hits = (ClassHit * (net.batch * top))()
    lib().network_classify_wait(net, hits, top)
    return _hits_arrays(hits, net.batch if n is None else n, top)


class _DevBuf:
    """Device allocation through the kernel C-ABI (y2_malloc / y2_memcpy_*), freed on exit."""

    def __init__(self, nbytes: int, host: np.ndarray | None = None):
        self.lib = _lib.load()
        self.ptr = C.c_void_p()
        self.nbytes = int(nbytes)
        _lib.check(self.lib.y2_malloc(C.byref(self.ptr), max(self.nbytes, 16)), "y2_malloc")
        if host is not None:
            host = np.ascontiguousarray(host)
            _lib.check(self.lib.y2_memcpy_h2d(self.ptr, host.ctypes.data, host.nbytes, None), "h2d")
            _lib.check(self.lib.y2_stream_sync(None))

    def get(self, dtype, shape) -> np.ndarray:
        out = np.empty(shape, dtype)
        _lib.check(self.lib.y2_memcpy_d2h(out.ctypes.data, self.ptr, out.nbytes, None), "d2h")
        _lib.check(self.lib.y2_stream_sync(None))
        return out

    def free(self):
        if self.ptr:
            self.lib.y2_free(self.ptr)
            self.ptr = C.c_void_p()


def decode_region_input(net: Network, region_in: np.ndarray, thresh: float, nms: float, use_map: bool = False) -> dict:
    """Run the region layer + get_region_boxes + do_nms_sort kernels on a given region-layer INPUT
    (fp32 [B][n*(5+classes)][h][w], the conv-head layout of the reference) for every image, through
    the kernel C-ABI with the region layer's own parameters (anchors, tree, map).  Returns the
    arrays the oracle drivers dump: region_out, boxes, probs_pre, probs_post, region_after_boxes.
    Used by the parity tests to feed both sides identical region inputs."""
    lib = _lib.load()
    l = region_layer(net)
    assert l.type == REGION
    B = region_in.shape[0]
    hw, n, classes = l.w * l.h, l.n, l.classes
    size = classes + 5
    total = hw * n
    assert region_in.size == B * total * size
    bufs = []

    def dev(nbytes, host=None):
        b = _DevBuf(nbytes, host)
        bufs.append(b)
        return b

    try:
        xin = dev(region_in.nbytes, region_in.astype(np.float32))
        flat = dev(region_in.nbytes)
        out = dev(region_in.nbytes)
        biases = dev(n * 2 * 4, np.ctypeslib.as_array(l.biases, (n * 2,)).astype(np.float32))
        _lib.check(lib.y2_nchw_to_flat_f32(xin.ptr, flat.ptr, B, n * size, hw, None), "nchw_to_flat")
        groups, gs, go, parent, tree_n = 0, None, None, None, 0
        if l.softmax_tree:
            t = l.softmax_tree.contents
            groups, tree_n = t.groups, t.n
            gs = dev(groups * 4, np.ctypeslib.as_array(t.group_size, (groups,)).astype(np.int32)).ptr
            go = dev(groups * 4, np.ctypeslib.as_array(t.group_offset, (groups,)).astype(np.int32)).ptr
            parent = dev(t.n * 4, np.ctypeslib.as_array(t.parent, (t.n,)).astype(np.int32)).ptr
        _lib.check(lib.y2_region_forward(flat.ptr, out.ptr, B, hw, n, classes, int(bool(l.softmax or l.softmax_tree)),
                                         groups, gs, go, None), "region_forward")
        region_out = out.get(np.float32, (B, total, size))
        map_n, map_dev = 0, None
        if use_map:
            assert l.map, "region layer has no map"
            map_n = 200
            map_dev = dev(200 * 4, np.ctypeslib.as_array(l.map, (200,)).astype(np.int32)).ptr
        out_classes = map_n or classes
        boxes = dev(B * total * 4 * 4)
        probs = dev(B * total * out_classes * 4)
        _lib.check(lib.y2_region_boxes(out.ptr, biases.ptr, boxes.ptr, probs.ptr, B, l.w, l.h, n, classes, 1.0, 1.0,
                                       thresh, 0, l.classfix, tree_n, parent, map_dev, map_n, None), "region_boxes")
        pre = probs.get(np.float32, (B, total, out_classes))
        if nms > 0:
            _lib.check(lib.y2_nms_sort(boxes.ptr, probs.ptr, B, total, out_classes, nms, None), "nms_sort")
        post = probs.get(np.float32, (B, total, out_classes))
        res = {"region_out": region_out, "boxes": boxes.get(np.float32, (B, total, 4)),
               "region_after_boxes": out.get(np.float32, (B, total, size))}
        if out_classes != classes:  # the reference's probs rows are `classes` wide, only 200 are written
            full_pre = np.zeros((B, total, classes), np.float32)
            full_post = np.zeros((B, total, classes), np.float32)
            full_pre[:, :, :out_classes] = pre
            full_post[:, :, :out_classes] = post
            pre, post = full_pre, full_post
        res["probs_pre"], res["probs_post"] = pre, post
        return res
    finally:
        for b in bufs:
            b.free()


def tree_detect_region_input(net: Network, region_in: np.ndarray, thresh: float, nms: float, max_det: int | None = None):
    """The sparse softmax-tree detection kernels (y2_region_tree_detect + y2_tree_nms_collect) on a given region-layer
    INPUT (fp32 [B][n*(5+classes)][h][w], the conv-head layout), with the region layer's own anchors and tree.
    Returns a list (per image) of detection record arrays, like network_detect_batch."""
    lib = _lib.load()
    l = region_layer(net)
    assert l.type == REGION and l.softmax_tree
    t = l.softmax_tree.contents
    B = region_in.shape[0]
    hw, n, classes = l.w * l.h, l.n, l.classes
    size, total = classes + 5, hw * n
    max_det = max_det or total
    parent = np.ctypeslib.as_array(t.parent, (t.n,)).astype(np.int32)
    gsize = np.ctypeslib.as_array(t.group_size, (t.groups,)).astype(np.int32)
    goff = np.ctypeslib.as_array(t.group_offset, (t.groups,)).astype(np.int32)
    owner = np.where(parent[goff] < 0, t.n, parent[goff])          # node every group hangs under (t.n = virtual root)
    order = np.argsort(owner, kind="stable").astype(np.int32)
    child_ptr = np.zeros(t.n + 2, np.int32)
    np.add.at(child_ptr, owner + 1, 1)
    child_ptr = np.cumsum(child_ptr).astype(np.int32)
    lib.y2_tree_rec_bytes.restype = C.c_size_t
    vp, i, f = C.c_void_p, C.c_int, C.c_float
    lib.y2_region_tree_detect.restype = i
    lib.y2_region_tree_detect.argtypes = [vp, i, vp, i, i, i, i, i, f, i, vp, vp, vp, vp, vp, vp]
    lib.y2_tree_nms_collect.restype = i
    lib.y2_tree_nms_collect.argtypes = [vp, i, i, f, f, vp, vp, i, vp]
    bufs = []

    def dev(nbytes, host=None):
        b = _DevBuf(nbytes, host)
        bufs.append(b)
        return b

    try:
        xin = dev(region_in.nbytes, region_in.astype(np.float32))
        flat = dev(region_in.nbytes)
        _lib.check(lib.y2_nchw_to_flat_f32(xin.ptr, flat.ptr, B, n * size, hw, None), "nchw_to_flat")
        biases = dev(n * 2 * 4, np.ctypeslib.as_array(l.biases, (n * 2,)).astype(np.float32))
        rec = dev(B * total * lib.y2_tree_rec_bytes())
        det = dev(B * max_det * C.sizeof(Detection))
        cnt = dev(B * 4)
        _lib.check(lib.y2_region_tree_detect(flat.ptr, n * size, biases.ptr, B, l.w, l.h, n, classes, thresh, l.classfix,
                                             dev(gsize.nbytes, gsize).ptr, dev(goff.nbytes, goff).ptr,
                                             dev(child_ptr.nbytes, child_ptr).ptr, dev(order.nbytes, order).ptr, rec.ptr,
                                             None), "region_tree_detect")
        _lib.check(lib.y2_tree_nms_collect(rec.ptr, B, total, thresh, nms, det.ptr, cnt.ptr, max_det, None),
                   "tree_nms_collect")
        counts = cnt.get(np.int32, (B,))
        dets = det.get(np.dtype([("x", "f4"), ("y", "f4"), ("w", "f4"), ("h", "f4"), ("prob", "f4"), ("obj_id", "i4"),
                                 ("box_index", "i4")]), (B, max_det))
        return [dets[b, :min(counts[b], max_det)].copy() for b in range(B)], counts
    finally:
        for b in bufs:
            b.free()
