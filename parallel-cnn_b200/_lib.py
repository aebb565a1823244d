"""ctypes declarations for every symbol of include/pcnn.h (kept in the same order as the header)."""
import ctypes as C
import os
import re

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
LIB_PATH = os.environ.get("PCNN_LIB_PATH") or os.path.join(HERE, "libpcnn.so")
HEADER = os.path.join(ROOT, "include", "pcnn.h")

NPARAM = 2343
OFF = dict(c1w=(0, 150), c1b=(150, 156), s1w=(156, 172), s1b=(172, 173), fw=(173, 2333), fb=(2333, 2343))
U8, F32 = 0, 1
MODE_AUTO, MODE_GRAPH, MODE_PERSISTENT = 0, 1, 2
TRAIN_SET, TEST_SET = 0, 1


class PcnnError(RuntimeError):
    """A libpcnn.so entry point returned a non-zero status (message = pcnn_last_error_string())."""

    def __init__(self, fn, code, msg):
        super().__init__(f"{fn} failed with status {code}: {msg}")
        self.fn, self.code, self.msg = fn, code, msg


_vp, _i, _l, _f, _sz = C.c_void_p, C.c_int, C.c_long, C.c_float, C.c_size_t
_pvp = C.POINTER(C.c_void_p)

# name -> argtypes (every function returns int unless listed in _RESTYPE)
_SIG = {
    "pcnn_version": [],
    "pcnn_last_error_string": [],
    "pcnn_create": [_pvp, _i, _vp],
    "pcnn_destroy": [_vp],
    "pcnn_sync": [_vp],
    "pcnn_device_info": [_vp, C.POINTER(_i), C.POINTER(_i), C.POINTER(_i), C.POINTER(_sz)],
    "pcnn_malloc": [_vp, _pvp, _sz],
    "pcnn_free": [_vp, _vp],
    "pcnn_memset0": [_vp, _vp, _sz],
    "pcnn_h2d": [_vp, _vp, _vp, _sz],
    "pcnn_d2h": [_vp, _vp, _vp, _sz],
    "pcnn_d2d": [_vp, _vp, _vp, _sz],
    "pcnn_init_params_reference": [_vp],
    "pcnn_set_params": [_vp, _vp],
    "pcnn_get_params": [_vp, _vp],
    "pcnn_get_grads": [_vp, _vp],
    "pcnn_params_dev": [_vp, _pvp],
    "pcnn_set_learning_rate": [_vp, _f],
    "pcnn_save_params": [_vp, C.c_char_p],
    "pcnn_load_params": [_vp, C.c_char_p],
    "pcnn_apply_step_function": [_vp, _vp, _vp, _l],
    "pcnn_make_error": [_vp, _vp, _vp, C.c_uint, _i],
    "pcnn_make_error_batch": [_vp, _vp, _vp, _vp, _i],
    "pcnn_apply_grad": [_vp, _vp, _vp, _l],
    "pcnn_apply_grad_scaled": [_vp, _vp, _vp, _l, _f],
    "pcnn_vector_norm": [_vp, _vp, _i, _i, _vp],
    "pcnn_fp_c1": [_vp, _vp, _vp, _vp, _vp, _i],
    "pcnn_fp_s1": [_vp, _vp, _vp, _vp, _vp, _i],
    "pcnn_fp_preact_f": [_vp, _vp, _vp, _vp, _i],
    "pcnn_fp_bias_f": [_vp, _vp, _vp, _i],
    "pcnn_bp_weight_f": [_vp, _vp, _vp, _vp, _i],
    "pcnn_bp_bias_f": [_vp, _vp, _vp, _i],
    "pcnn_bp_output_s1": [_vp, _vp, _vp, _vp, _i],
    "pcnn_bp_preact_s1": [_vp, _vp, _vp, _vp, _i],
    "pcnn_bp_weight_s1": [_vp, _vp, _vp, _vp, _i],
    "pcnn_bp_bias_s1": [_vp, _vp, _vp, _i],
    "pcnn_bp_output_c1": [_vp, _vp, _vp, _vp, _i],
    "pcnn_bp_preact_c1": [_vp, _vp, _vp, _vp, _i],
    "pcnn_bp_weight_c1": [_vp, _vp, _vp, _vp, _i],
    "pcnn_bp_bias_c1": [_vp, _vp, _vp, _i],
    "pcnn_mnist_load_u8": [C.c_char_p, C.c_char_p, _pvp, _pvp, C.POINTER(C.c_uint)],
    "pcnn_mnist_free": [_vp],
    "pcnn_dataset_upload": [_vp, _i, _vp, _i, _vp, _l],
    "pcnn_dataset_bind": [_vp, _i, _vp, _i, _vp, _l],
    "pcnn_train_step": [_vp, _l, _i],
    "pcnn_train_steps": [_vp, _l, _i, _i],
    "pcnn_train_steps_prepare": [_vp, _i, _i],
    "pcnn_train_step_dev": [_vp, _vp, _i, _vp, _i],
    "pcnn_train_step_host": [_vp, _vp, _i, _vp, _i, C.POINTER(_f)],
    "pcnn_compute_grads": [_vp, _vp, _i, _vp, _i],
    "pcnn_learn": [_vp, _i, _i, C.POINTER(_f)],
    "pcnn_learn_host": [_vp, _vp, _i, _vp, _l, _i, _i, C.POINTER(_f)],
    "pcnn_err_sum": [_vp, C.POINTER(C.c_double), _i],
    "pcnn_forward_batch": [_vp, _vp, _i, _i, _vp, _vp],
    "pcnn_test": [_vp, C.POINTER(_l)],
    "pcnn_launch_count": [_vp, C.POINTER(_l)],
    "pcnn_step_errs": [_vp, _vp, _l, C.POINTER(_l)],
    "pcnn_time_fused_kernel": [_vp, _i, _i, C.POINTER(_f)],
    "pcnn_measure_fp32_peak": [_vp, C.POINTER(_f)],
    "pcnn_measure_tma_read": [_vp, _vp, _i, _i, _i, _i, _i, C.POINTER(_f)],
    "pcnn_measure_tma_write": [_vp, _vp, _i, _i, _i, _i, _i, _i, _i, C.POINTER(_f)],
    "pcnn_measure_mma_rate": [_vp, _i, _i, _i, _i, _i, _i, C.POINTER(_f)],
    "pcnn_comm_unique_id": [_vp, C.POINTER(_sz)],
    "pcnn_comm_init_rank": [_vp, _vp, _i, _i],
    "pcnn_comm_destroy": [_vp],
    "pcnn_allreduce_grads": [_vp],
    "pcnn_p2p_export": [_vp, _vp, C.POINTER(_sz)],
    "pcnn_p2p_attach": [_vp, _vp, _i, _i],
    "pcnn_p2p_detach": [_vp],
    "pcnn_set_step_mode": [_vp, _i],
    "pcnn_persist_trace": [_vp, _vp, _i],
    "pcnn_persist_trace_ctas": [_vp, _vp, _i],
    "pcnn_persist_info": [_vp, _vp],
    "pcnn_conv_bwd_select": [_vp, _i],
    "pcnn_l5_compute_grads": [_vp, _vp, _vp, _i, _vp, _i, _vp],
    "pcnn_l5_train_step": [_vp, _vp, _vp, _i, _vp, _i, _vp],
    "pcnn_l5_forward": [_vp, _vp, _vp, _i, _i, _vp],
    "pcnn_persist_tune": [_vp, _i],
    "pcnn_maxpool_fwd": [_vp, _vp, _vp, _vp, _i, _i, _i, _i],
    "pcnn_maxpool_bwd": [_vp, _vp, _vp, _vp, _i, _i, _i, _i],
    "pcnn_softmax_ce": [_vp, _vp, _vp, _i, _i, _vp, _vp, _vp],
    "pcnn_conv_tc_plan_create": [_vp, _i, _i, _i, _i, _i, _i, _i, _i, _i, _i, _vp, _vp, _pvp],
    "pcnn_conv_tc_plan_create_strided": [_vp, _i, _i, _i, _i, _i, _i, _i, _i, _i, _i, _i, _vp, _vp, _pvp],
    "pcnn_conv_tc_plan_destroy": [_vp, _vp],
    "pcnn_conv_tc_fwd": [_vp, _vp, _vp, _vp],
    "pcnn_f32_to_bf16_rows": [_vp, _vp, _vp, _l, _i, _i],
    "pcnn_conv_bwd_plan_info": [_i, _i, _i, _i, _i, _i, _i, _vp],
    "pcnn_conv_bwd_plan_info_strided": [_i, _i, _i, _i, _i, _i, _i, _i, _vp],
    "pcnn_pad_nhwc_bf16": [_vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _i],
    "pcnn_crop_nhwc_bf16": [_vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _i],
    "pcnn_conv_wgrad": [_vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _i, _i],
    "pcnn_conv_dgrad": [_vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _i, _i],
    "pcnn_conv_wgrad_strided": [_vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _i, _i, _i],
    "pcnn_conv_dgrad_strided": [_vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _i, _i, _i],
}
_RESTYPE = {"pcnn_last_error_string": C.c_char_p, "pcnn_mnist_free": None}

_lib = None


def declared_symbols():
    """Every function name declared in include/pcnn.h (parsed from the header text)."""
    text = open(HEADER).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(pcnn_[a-z0-9_]+)\s*\(", text)))


def lib():
    """Load libpcnn.so (built in-tree by `make -C parallel-cnn_b200/csrc` / __graft_entry__.build()).  Fails loudly."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise PcnnError("dlopen", -1, f"{LIB_PATH} not built: run `python -c 'import __graft_entry__ as g; g.build()'`; "
                            "there is no CPU fallback")
        L = C.CDLL(LIB_PATH)
        for name, args in _SIG.items():
            fn = getattr(L, name)
            fn.argtypes = args
            fn.restype = _RESTYPE.get(name, C.c_int)
        _lib = L
    return _lib


def check(fn, code):
    if code != 0:
        raise PcnnError(fn, code, lib().pcnn_last_error_string().decode())


def init_params_reference():
    """The reference's static-constructor parameters (glibc rand(), seed 1) as a packed float32[2343] (host only)."""
    p = np.empty(NPARAM, np.float32)
    check("pcnn_init_params_reference", lib().pcnn_init_params_reference(p.ctypes.data))
    return p


def mnist_load_u8(image_file, label_file):
    """mnist_load's contract (return codes 0, -1..-4) on raw u8; returns (code, images[n,784] u8, labels[n] u8)."""
    L = lib()
    img, lab, cnt = C.c_void_p(), C.c_void_p(), C.c_uint(0)
    rc = L.pcnn_mnist_load_u8(os.fsencode(image_file), os.fsencode(label_file), C.byref(img), C.byref(lab), C.byref(cnt))
    if rc != 0:
        return rc, None, None
    n = cnt.value
    images = np.ctypeslib.as_array(C.cast(img, C.POINTER(C.c_uint8)), shape=(n * 784,)).reshape(n, 784).copy()
    labels = np.ctypeslib.as_array(C.cast(lab, C.POINTER(C.c_uint8)), shape=(n,)).copy()
    L.pcnn_mnist_free(img)
    L.pcnn_mnist_free(lab)
    return 0, images, labels
