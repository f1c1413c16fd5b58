"""ctypes binding of libmvsf_b200.so (include/mvsf_b200.h).  There is no fallback: if the library is missing or a
call fails, a RuntimeError is raised (the reference's seams raise Python exceptions: SURVEY.md §8b)."""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("MVSF_LIB_PATH") or os.path.join(_HERE, "libmvsf_b200.so")   # override: A-B builds of the same library
_lib = None

P, I, F, Z = ctypes.c_void_p, ctypes.c_int, ctypes.c_float, ctypes.c_size_t
SIGNATURES = {
    "mvsf_abi_version": ([], I),
    "mvsf_launch_count": ([I], ctypes.c_longlong),
    "mvsf_ktimer_enable": ([I], I),
    "mvsf_ktimer_read": ([ctypes.c_char_p, ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_longlong)], I),
    "mvsf_nchw_to_nhwc": ([P, P, I, I, I, P], I),
    "mvsf_nhwc_to_nchw": ([P, P, I, I, I, P], I),
    "mvsf_compose_geometry": ([P, I, P, P, P], I),
    "mvsf_homography_from_proj": ([P, P, I, P, P], I),
    "mvsf_init_inverse_range": ([P, I, P, I, I, I, P], I),
    "mvsf_schedule_inverse_range": ([P, P, I, F, P, I, I, I, P], I),
    "mvsf_position3d": ([P, P, P, I, P, I, P, I, I, I, P], I),
    "mvsf_homo_warp": ([P, P, P, P, P, I, I, I, I, P], I),
    "mvsf_warp_corr_set_tile_path": ([I], I),
    "mvsf_warp_corr_last_selection": ([ctypes.POINTER(I), ctypes.POINTER(I)], I),
    "mvsf_warp_corr_plan": ([I, I, I, I, I, I, Z], I),
    "mvsf_warp_corr_entropy": ([P, P, P, P, I, I, I, I, I, I, P], I),
    "mvsf_vis_cnn": ([P, P, P, I, I, I, P], I),
    "mvsf_warp_corr_aggregate": ([P, P, P, P, P, I, I, I, I, I, I, P], I),
    "mvsf_warp_corr_entropy_store": ([P, P, P, P, P, I, I, I, I, I, I, P], I),
    "mvsf_corr_aggregate": ([P, P, P, I, I, I, I, I, P], I),
    "mvsf_costreg_unet_workspace_bytes": ([I, I, I, I, I, ctypes.POINTER(Z)], I),
    "mvsf_costreg_unet_tc_bytes": ([ctypes.POINTER(Z)], I),
    "mvsf_costreg_unet_pack_tc": ([I, P, P, Z, P], I),
    "mvsf_costreg_unet_forward": ([I, P, P, P, P, P, Z, I, I, I, I, P], I),
    "mvsf_conv3d_tc_layer": ([I, I, P, P, P, P, P, Z, I, I, I, I, I, P], I),
    "mvsf_costreg_tr_workspace_bytes": ([I, I, I, I, ctypes.POINTER(Z)], I),
    "mvsf_costreg_tr_forward": ([P, P, P, P, Z, P, P, Z, I, I, I, I, I, F, P], I),
    "mvsf_split_weights_f16": ([P, P, Z, P], I),
    "mvsf_attention_forward": ([P, P, P, Z, I, F, P], I),
    "mvsf_linear_tc_forward": ([P, P, P, P, P, Z, I, I, I, I, P], I),
    "mvsf_softargmax": ([P, P, F, P, P, P, I, I, I, P], I),
    "mvsf_conf_accumulate": ([P, I, I, P, I, I, F, I, P], I),
    "mvsf_fmt_workspace_bytes": ([I, I, I, ctypes.POINTER(Z)], I),
    "mvsf_fmt_forward": ([P] * 7 + [Z] + [P] * 5 + [Z, I, I, I, P], I),
}
# entry points that launch no kernel: profile_calls does not time them
NO_LAUNCH = {"mvsf_abi_version", "mvsf_launch_count", "mvsf_ktimer_enable", "mvsf_ktimer_read", "mvsf_warp_corr_plan",
             "mvsf_warp_corr_set_tile_path", "mvsf_warp_corr_last_selection", "mvsf_costreg_unet_workspace_bytes",
             "mvsf_costreg_unet_tc_bytes", "mvsf_costreg_tr_workspace_bytes", "mvsf_fmt_workspace_bytes"}


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(f"{LIB_PATH} is missing: build it with `python -m mvsformerplusplus_b200.build` "
                               "(the B200 hot path has no CPU/PyTorch fallback)")
        L = ctypes.CDLL(LIB_PATH)
        L.mvsf_last_error.restype = ctypes.c_char_p
        L.mvsf_last_error.argtypes = []
        for name, (argt, rest) in SIGNATURES.items():
            fn = getattr(L, name)  # AttributeError if the symbol is not exported
            fn.argtypes = argt
            fn.restype = rest
        _lib = L
    return _lib


def check(rc, what):
    if rc != 0:
        msg = lib().mvsf_last_error().decode(errors="replace")
        raise RuntimeError(f"{what} failed (status {rc}): {msg}")


def launch_count(reset=False):
    return int(lib().mvsf_launch_count(1 if reset else 0))


class profile_calls:
    """Context manager: brackets every library call with CUDA events on the current stream and reports device
    milliseconds per entry point (used by bench.py for the roofline of the warp+correlation kernels).
    Timing-only instrumentation; it does not change what is launched."""

    def __init__(self):
        self.records = []  # (name, start_event, end_event)

    def __enter__(self):
        import torch
        L = lib()
        self._orig = {}
        for name in SIGNATURES:
            if name in NO_LAUNCH:
                continue
            fn = getattr(L, name)
            self._orig[name] = fn

            def wrapped(*a, _fn=fn, _name=name):
                s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                s.record()
                rc = _fn(*a)
                e.record()
                self.records.append((_name, s, e))
                return rc
            setattr(L, name, wrapped)
        return self

    def __exit__(self, *exc):
        L = lib()
        for name, fn in self._orig.items():
            setattr(L, name, fn)
        return False

    def summary(self):
        import torch
        torch.cuda.synchronize()
        out = {}
        for name, s, e in self.records:
            d = out.setdefault(name, {"ms": 0.0, "calls": 0})
            d["ms"] += s.elapsed_time(e)
            d["calls"] += 1
        return out


def ktimer_enable(on):
    check(lib().mvsf_ktimer_enable(1 if on else 0), "ktimer_enable")


def ktimer_read(name):
    """(device ms, launches) recorded around the named kernel since the last read."""
    ms, n = ctypes.c_double(0.0), ctypes.c_longlong(0)
    check(lib().mvsf_ktimer_read(name.encode(), ctypes.byref(ms), ctypes.byref(n)), "ktimer_read")
    return ms.value, n.value
