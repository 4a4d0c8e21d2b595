"""ctypes binding of libevk.so (the C ABI declared in include/evk.h).

There is NO CPU fallback: if the shared library is missing or the device is not a B200-class
(sm_100) GPU, every compute entry point raises.  Build with ``python -c "import
__graft_entry__ as g; g.build()"`` or ``make -C event_utils_b200/csrc``.
"""
import ctypes
import os
import threading

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
SO_PATH = os.environ.get("EVK_LIB") or os.path.join(_HERE, "libevk.so")  # EVK_LIB: development override

# flags (mirror include/evk.h)
ACCUMULATE = 0x1
BILINEAR = 0x2
CLIP = 0x4
NEGPOS_TRUTHY = 0x8
WINDOW_PAIRS = 0x100000
WINDOW_NEGPOS = 0x400000
NO_FOLD = 0x800000
PEER_MULTICAST = 0x1000000
AUTO_SPAN = 0x200000
VARIANT_AUTO = 0 << 8
VARIANT_GLOBAL_RED = 1 << 8
VARIANT_VECTOR_RED = 2 << 8
VARIANT_SMEM_TILE = 3 << 8
VARIANT_WARP_AGG = 4 << 8
VARIANT_ROUTED = 5 << 8
VARIANT_MASK = 0xF << 8
ROUTED_ABORT_MARK = 1 << 62       # evk.h: added to the oob counter when the routed kernel's watchdog fired
TS_REVERSE = 0x80
TS_RAW = 0x1000
CMAX_WANT_GRAD = 0x10
CMAX_ABS_POLARITY = 0x20
CMAX_NO_CHANNEL_MIX = 0x40
OBJ_VARIANCE, OBJ_SOS, OBJ_SOE, OBJ_MOA, OBJ_ISOA, OBJ_SOSA = range(6)
WARP_LINVEL, WARP_ROTATION, WARP_XYZTHETA = range(3)
WARP_MODELS = {"linvel": WARP_LINVEL, "rotation": WARP_ROTATION, "xyztheta": WARP_XYZTHETA}   # warp_function.fused_kind

_lib = None
_lock = threading.Lock()


class EvkError(RuntimeError):
    pass


def _declare(L):
    c = ctypes
    vp, i64, f32, f64, ci, cu, sz = c.c_void_p, c.c_int64, c.c_float, c.c_double, c.c_int, c.c_uint, c.c_size_t
    L.evk_version.restype = ci
    L.evk_last_error.restype = c.c_char_p
    L.evk_device_check.restype = ci
    L.evk_prof_enable.restype = ci
    L.evk_prof_enable.argtypes = [ci]
    L.evk_prof_collect.restype = ci
    L.evk_prof_collect.argtypes = [c.POINTER(c.c_double), c.POINTER(c.c_longlong), c.POINTER(c.c_longlong)]
    L.evk_voxel_workspace_bytes.restype = sz
    L.evk_voxel_workspace_bytes.argtypes = [ci, ci, ci, cu]
    L.evk_voxel_f32.restype = ci
    L.evk_voxel_f32.argtypes = [vp, vp, vp, vp, i64, f32, f32, ci, ci, ci, cu, vp, vp, sz, vp, vp]
    L.evk_voxel_negpos_f32.restype = ci
    L.evk_voxel_negpos_f32.argtypes = [vp, vp, vp, vp, i64, f32, f32, ci, ci, ci, cu, vp, vp, sz, vp, vp]
    L.evk_voxel_packed_f32.restype = ci
    L.evk_voxel_packed_f32.argtypes = [vp, vp, vp, vp, i64, f64, f64, ci, ci, ci, cu, vp, vp, sz, vp, vp]
    L.evk_voxel_aos_f32.restype = ci
    L.evk_voxel_aos_f32.argtypes = [vp, i64, f32, f32, ci, ci, ci, cu, vp, vp, sz, vp, vp]
    L.evk_voxel_windows_f32.restype = ci
    L.evk_voxel_windows_f32.argtypes = [vp, vp, vp, vp, vp, ci, i64, ci, ci, ci, cu, vp, vp, vp]
    L.evk_image_workspace_bytes.restype = sz
    L.evk_image_workspace_bytes.argtypes = [ci, ci, cu]
    L.evk_image_f32.restype = ci
    L.evk_image_f32.argtypes = [vp, vp, vp, i64, ci, ci, f32, f32, cu, f32, vp, vp, sz, vp, vp]
    L.evk_timestamp_image_workspace_bytes.restype = sz
    L.evk_timestamp_image_workspace_bytes.argtypes = [ci, ci]
    L.evk_timestamp_image_f32.restype = ci
    L.evk_timestamp_image_f32.argtypes = [vp, vp, vp, vp, i64, f32, f32, ci, ci, f32, f32, cu, vp, vp, vp, sz, vp, vp]
    L.evk_count_u32.restype = ci
    L.evk_count_u32.argtypes = [vp, vp, i64, ci, ci, f32, f32, cu, vp, vp, vp]
    L.evk_splat_idx_f32.restype = ci
    L.evk_splat_idx_f32.argtypes = [vp, vp, vp, vp, vp, i64, ci, ci, vp, vp, vp]
    L.evk_splat_drv_idx_f32.restype = ci
    L.evk_splat_drv_idx_f32.argtypes = [vp, vp, vp, vp, vp, vp, ci, i64, ci, ci, vp, vp, vp]
    L.evk_image_drv_f32.restype = ci
    L.evk_image_drv_f32.argtypes = [vp, vp, vp, vp, vp, ci, i64, ci, ci, f32, f32, cu, vp, vp, vp, vp]
    L.evk_gather_bilinear_f64.restype = ci
    L.evk_gather_bilinear_f64.argtypes = [vp, vp, i64, vp, ci, ci, vp, vp, vp]
    L.evk_warp_flow_f32.restype = ci
    L.evk_warp_flow_f32.argtypes = [vp, vp, vp, i64, vp, ci, ci, f32, vp, vp, vp, sz, vp]
    L.evk_voxel_fold_allreduce_f32.restype = ci
    L.evk_voxel_fold_allreduce_f32.argtypes = [vp, vp, ci, ci, ci, ci, ci, cu, vp]
    L.evk_warp_flow_workspace_bytes.restype = sz
    L.evk_warp_flow_workspace_bytes.argtypes = [ci, ci]
    L.evk_cmax_workspace_bytes.restype = sz
    L.evk_cmax_workspace_bytes.argtypes = [ci, ci]
    L.evk_cmax_linvel_variance_f64.restype = ci
    L.evk_cmax_linvel_variance_f64.argtypes = [vp, vp, vp, vp, i64, f64, f64, f64, f64, ci, ci, ci, ci, f64, cu,
                                               vp, vp, vp, vp, sz, vp]
    L.evk_cmax_linvel_variance_f32.restype = ci
    L.evk_cmax_linvel_variance_f32.argtypes = [vp, vp, vp, vp, i64, f32, f32, f32, ci, ci, ci, ci, f64, cu,
                                               vp, vp, vp, vp, sz, vp]
    L.evk_cmax_linvel_objective_f64.restype = ci
    L.evk_cmax_linvel_objective_f64.argtypes = [vp, vp, vp, vp, i64, f64, f64, f64, f64, ci, ci, ci, ci, f64, cu, ci, f64,
                                                vp, vp, vp, vp, sz, vp]
    L.evk_cmax_linvel_objective_f32.restype = ci
    L.evk_cmax_linvel_objective_f32.argtypes = [vp, vp, vp, vp, i64, f32, f32, f32, ci, ci, ci, ci, f64, cu, ci, f64,
                                                vp, vp, vp, vp, sz, vp]
    L.evk_cmax_linvel_objective_batch_f64.restype = ci
    L.evk_cmax_linvel_objective_batch_f64.argtypes = [vp, vp, vp, vp, i64, f64, vp, ci, f64, ci, ci, ci, ci, f64, cu, ci, f64,
                                                      vp, vp, sz, vp]
    L.evk_iwe_objective_f32.restype = ci
    L.evk_iwe_objective_f32.argtypes = [vp, vp, ci, ci, f64, cu, ci, f64, vp, vp, sz, vp]
    L.evk_cmax_model_objective_f64.restype = ci
    L.evk_cmax_model_objective_f64.argtypes = [ci, vp, ci, vp, vp, vp, vp, i64, f64, f64, ci, ci, ci, ci, f64, cu, ci, f64,
                                               vp, vp, vp, sz, vp]
    L.evk_cmax_model_objective_f32.restype = ci
    L.evk_cmax_model_objective_f32.argtypes = [ci, vp, ci, vp, vp, vp, vp, i64, f32, ci, ci, ci, ci, f64, cu, ci, f64,
                                               vp, vp, vp, sz, vp]
    L.evk_cmax_model_warp_f64.restype = ci
    L.evk_cmax_model_warp_f64.argtypes = [ci, vp, ci, vp, vp, vp, vp, i64, f64, ci, ci, cu, vp, vp, vp, vp, vp, vp]
    L.evk_iwe_objective_k_f32.restype = ci
    L.evk_iwe_objective_k_f32.argtypes = [vp, vp, ci, ci, ci, f64, cu, ci, f64, vp, vp, vp, sz, vp]
    L.evk_gaussian_blur_f32.restype = ci
    L.evk_gaussian_blur_f32.argtypes = [vp, ci, ci, f64, vp, vp, vp]
    L.evk_variance_objective_f32.restype = ci
    L.evk_variance_objective_f32.argtypes = [vp, vp, ci, ci, f64, cu, vp, vp, sz, vp]
    L.evk_peer_barrier.restype = ci
    L.evk_peer_barrier.argtypes = [vp, ci, ci, cu, vp]
    L.evk_cmax_linvel_partial_f64.restype = ci
    L.evk_cmax_linvel_partial_f64.argtypes = [vp, vp, vp, vp, i64, f64, f64, f64, f64, ci, ci, ci, ci, cu, vp, vp, vp, sz, vp]
    L.evk_cmax_linvel_partial_f32.restype = ci
    L.evk_cmax_linvel_partial_f32.argtypes = [vp, vp, vp, vp, i64, f32, f32, f32, ci, ci, ci, ci, cu, vp, vp, vp, sz, vp]
    L.evk_cmax_peer_tail_f32.restype = ci
    L.evk_cmax_peer_tail_f32.argtypes = [vp, vp, ci, ci, ci, f64, cu, vp, vp, sz, vp]
    L.evk_cmax_flow_variance_f32.restype = ci
    L.evk_cmax_flow_variance_f32.argtypes = [vp, vp, vp, vp, i64, vp, f32, ci, ci, f64, cu, vp, vp, vp, sz, vp]
    L.evk_robust_norm_workspace_bytes.restype = sz
    L.evk_robust_norm_workspace_bytes.argtypes = []
    L.evk_robust_norm_f32.restype = ci
    L.evk_robust_norm_f32.argtypes = [vp, i64, i64, i64, vp, vp, vp, sz, vp]
    L.evk_host_hash64.restype = c.c_uint64
    L.evk_host_hash64.argtypes = [vp, sz, c.c_uint64]
    L.evk_host_hash64_multi.restype = None
    L.evk_host_hash64_multi.argtypes = [c.POINTER(vp), c.POINTER(sz), ci, c.c_uint64, c.POINTER(c.c_uint64)]
    L.evk_host_copy.restype = None
    L.evk_host_copy.argtypes = [c.POINTER(vp), c.POINTER(vp), ci, sz]
    L.evk_host_upload.restype = ci
    L.evk_host_upload.argtypes = [vp, c.POINTER(vp), c.POINTER(vp), ci, c.POINTER(sz)]
    L.evk_pipeline_create.restype = ci
    L.evk_pipeline_create.argtypes = [c.POINTER(vp), i64]
    L.evk_pipeline_destroy.restype = None
    L.evk_pipeline_destroy.argtypes = [vp]
    L.evk_voxel_host_packed_f32.restype = ci
    L.evk_voxel_host_packed_f32.argtypes = [vp, vp, vp, vp, vp, i64, f64, f64, ci, ci, ci, cu, vp, c.POINTER(c.c_ulonglong)]
    L.evk_voxel_host_f32.restype = ci
    L.evk_voxel_host_f32.argtypes = [vp, vp, vp, vp, vp, i64, f32, f32, ci, ci, ci, cu, vp, c.POINTER(c.c_ulonglong)]


def load():
    """Load libevk.so (no GPU needed for this step) and declare the prototypes."""
    global _lib
    with _lock:
        if _lib is None:
            if not os.path.exists(SO_PATH):
                raise EvkError("libevk.so not found at %s -- build it (make -C event_utils_b200/csrc); "
                               "there is no CPU fallback" % SO_PATH)
            L = ctypes.CDLL(SO_PATH)
            _declare(L)
            _lib = L
    return _lib


_device_ok = {}


def lib():
    """Library handle for compute calls: requires a CUDA device of compute capability 10.x."""
    L = load()
    if not torch.cuda.is_available():
        raise EvkError("event_utils_b200 needs a CUDA device (B200, sm_100a); there is no CPU fallback")
    dev = torch.cuda.current_device()
    if dev not in _device_ok:
        check_device(dev)
    return L


def check_device(dev):
    """Capability check of the device that will run the kernels (not merely the current one)."""
    L = load()
    dev = dev.index if isinstance(dev, torch.device) else int(dev)
    if dev is None:
        dev = torch.cuda.current_device()
    if dev not in _device_ok:
        torch.cuda.init()
        with torch.cuda.device(dev):
            torch.empty(1, device="cuda")  # make sure the primary context exists
            check(L.evk_device_check())
        _device_ok[dev] = True


def check(rc):
    if rc != 0:
        msg = load().evk_last_error()
        raise EvkError("libevk error %d: %s" % (rc, msg.decode() if msg else "?"))


def host_hashes(arrays):
    """64-bit content hashes of contiguous numpy arrays (every byte enters), one library call for all of them."""
    k = len(arrays)
    ptrs = (ctypes.c_void_p * k)(*[a.ctypes.data for a in arrays])
    sizes = (ctypes.c_size_t * k)(*[a.nbytes for a in arrays])
    out = (ctypes.c_uint64 * k)()
    load().evk_host_hash64_multi(ptrs, sizes, k, 0, out)
    return tuple(out)


UPLOAD_MIN_BYTES = 4 << 20      # below this torch's own copy is as fast (one staged driver copy)


def upload(host_tensors, device):
    """CPU tensors -> new device tensors of the same dtype / shape.  Large ordinary (pageable) tensors -- what numpy hands
    over -- take evk_host_upload (pinned bounce slots filled by the library's worker pool, ~50 GB/s instead of the
    driver's ~10 GB/s staged copy); small or non-contiguous ones take torch's copy.  The result is complete on return."""
    host_tensors = list(host_tensors)
    big = [i for i, t in enumerate(host_tensors)
           if (not t.is_cuda) and t.is_contiguous() and t.numel() * t.element_size() >= UPLOAD_MIN_BYTES]
    out = [None] * len(host_tensors)
    for i, t in enumerate(host_tensors):
        if i not in big:
            out[i] = t.to(device, non_blocking=True)
    if big:
        with torch.cuda.device(device):
            for i in big:
                out[i] = torch.empty(host_tensors[i].shape, dtype=host_tensors[i].dtype, device=device)
            torch.cuda.current_stream().synchronize()      # the allocator may hand out memory with work still queued on it
            k = len(big)
            dst = (ctypes.c_void_p * k)(*[out[i].data_ptr() for i in big])
            src = (ctypes.c_void_p * k)(*[host_tensors[i].data_ptr() for i in big])
            nb = (ctypes.c_size_t * k)(*[host_tensors[i].numel() * host_tensors[i].element_size() for i in big])
            check(lib().evk_host_upload(pipeline(), dst, src, k, nb))
    return out


def stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def ptr(t):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else None


_scratch = {}


def _stream_key(key, device):
    """Scratch is reused call after call, which is only safe in stream order: one buffer per
    (purpose, device, stream, host thread) -- ctypes releases the GIL during a call, so two threads that
    share a stream (e.g. the default one) must not share a workspace either."""
    idx = device.index if device.index is not None else torch.cuda.current_device()
    if idx not in _device_ok:
        check_device(idx)
    return (key, idx, torch.cuda.current_stream(idx).cuda_stream, threading.get_ident())


def scratch(key, nbytes, device):
    """A cached 256-byte aligned device scratch buffer (uint8) of at least nbytes, private to the
    current stream of `device`."""
    k = _stream_key(key, device)
    buf = _scratch.get(k)
    if buf is None or buf.numel() < nbytes:
        buf = torch.empty(max(int(nbytes), 256), dtype=torch.uint8, device=device)
        _scratch[k] = buf
    return buf


def oob_counter(device):
    k = _stream_key("oob", device)
    buf = _scratch.get(k)
    if buf is None:
        buf = torch.zeros(1, dtype=torch.int64, device=device)
        _scratch[k] = buf
    else:
        buf.zero_()
    return buf


_pipelines = {}


def pipeline(chunk_events=4 << 20):
    """The host-input pipeline (staging buffers + two streams, csrc/evk_host.cu) of the calling THREAD on
    the current device: a pipeline serves one call at a time, and ctypes releases the GIL during it."""
    import threading
    k = (torch.cuda.current_device(), threading.get_ident())
    p = _pipelines.get(k)
    if p is None:
        h = ctypes.c_void_p()
        check(lib().evk_pipeline_create(ctypes.byref(h), chunk_events))
        p = h
        _pipelines[k] = p
    return p
