"""Engine: a thin object wrapper over one pcnn_ctx.  Method names follow include/pcnn.h minus the pcnn_ prefix, which
in turn follow /root/reference/Sequential/layer.h and Main.cpp (fp_c1, bp_weight_c1, learn, test ...)."""
import ctypes as C

import numpy as np

from ._lib import F32, NPARAM, TEST_SET, TRAIN_SET, U8, PcnnError, check, lib


def _pixel_type(arr_or_dtype):
    dt = np.dtype(getattr(arr_or_dtype, "dtype", arr_or_dtype))
    if dt == np.uint8:
        return U8
    if dt == np.float32:
        return F32
    raise PcnnError("pixel_type", -1, f"images must be uint8 or float32, got {dt}")


class DeviceArray:
    """A device buffer obtained from pcnn_malloc (zero-initialised like the reference's `new float[n]()`)."""

    def __init__(self, engine, shape, dtype=np.float32):
        self.engine = engine
        self.shape = tuple(int(s) for s in (shape if isinstance(shape, (tuple, list)) else (shape,)))
        self.dtype = np.dtype(dtype)
        self.nbytes = int(np.prod(self.shape, dtype=np.int64)) * self.dtype.itemsize
        p = C.c_void_p()
        check("pcnn_malloc", lib().pcnn_malloc(engine.ctx, C.byref(p), self.nbytes))
        self.ptr = p.value

    @classmethod
    def from_host(cls, engine, host):
        host = np.ascontiguousarray(host)
        d = cls(engine, host.shape, host.dtype)
        d.copy_from(host)
        return d

    def copy_from(self, host):
        host = np.ascontiguousarray(host, self.dtype)
        assert host.nbytes == self.nbytes, (host.shape, self.shape)
        check("pcnn_h2d", lib().pcnn_h2d(self.engine.ctx, self.ptr, host.ctypes.data, self.nbytes))
        return self

    def to_host(self):
        out = np.empty(self.shape, self.dtype)
        check("pcnn_d2h", lib().pcnn_d2h(self.engine.ctx, out.ctypes.data, self.ptr, self.nbytes))
        return out

    def zero(self):
        check("pcnn_memset0", lib().pcnn_memset0(self.engine.ctx, self.ptr, self.nbytes))

    def free(self):
        if self.ptr and self.engine.ctx:
            lib().pcnn_free(self.engine.ctx, self.ptr)
        self.ptr = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


def _p(x):
    """device pointer of a DeviceArray / raw int / torch tensor (data_ptr) / None"""
    if x is None:
        return None
    if isinstance(x, DeviceArray):
        return x.ptr
    if hasattr(x, "data_ptr"):
        return x.data_ptr()
    return int(x)


class Engine:
    def __init__(self, device=-1, stream=None):
        self.ctx = None
        ctx = C.c_void_p()
        check("pcnn_create", lib().pcnn_create(C.byref(ctx), int(device), stream))
        self.ctx = ctx

    def close(self):
        if self.ctx:
            lib().pcnn_destroy(self.ctx)
            self.ctx = None

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _call(self, name, *args):
        check(name, getattr(lib(), name)(self.ctx, *args))

    # ------------------------------------------------------------------ context / parameters
    def sync(self):
        self._call("pcnn_sync")

    def device_info(self):
        sm, ma, mi, hb = C.c_int(), C.c_int(), C.c_int(), C.c_size_t()
        self._call("pcnn_device_info", C.byref(sm), C.byref(ma), C.byref(mi), C.byref(hb))
        return dict(sm_count=sm.value, cc=(ma.value, mi.value), hbm_bytes=hb.value)

    def array(self, shape, dtype=np.float32):
        return DeviceArray(self, shape, dtype)

    def to_device(self, host):
        return DeviceArray.from_host(self, host)

    def set_params(self, p):
        p = np.ascontiguousarray(p, np.float32)
        assert p.size == NPARAM
        self._call("pcnn_set_params", p.ctypes.data)

    def get_params(self):
        p = np.empty(NPARAM, np.float32)
        self._call("pcnn_get_params", p.ctypes.data)
        return p

    def get_grads(self):
        g = np.empty(NPARAM, np.float32)
        self._call("pcnn_get_grads", g.ctypes.data)
        return g

    def params_dev(self):
        p = C.c_void_p()
        self._call("pcnn_params_dev", C.byref(p))
        return p.value

    def set_learning_rate(self, dt):
        self._call("pcnn_set_learning_rate", float(dt))

    def save_params(self, path):
        self._call("pcnn_save_params", str(path).encode())

    def load_params(self, path):
        self._call("pcnn_load_params", str(path).encode())

    def err_sum(self, reset=False):
        s = C.c_double()
        self._call("pcnn_err_sum", C.byref(s), 1 if reset else 0)
        return s.value

    def launch_count(self):
        n = C.c_long()
        self._call("pcnn_launch_count", C.byref(n))
        return n.value

    # ------------------------------------------------------------------ per-operator API (layer.h names)
    def apply_step_function(self, inp, out, n):
        self._call("pcnn_apply_step_function", _p(inp), _p(out), int(n))

    def makeError(self, err, out, Y, n=10):
        self._call("pcnn_make_error", _p(err), _p(out), int(Y), int(n))

    def makeError_batch(self, err, out, labels, B):
        self._call("pcnn_make_error_batch", _p(err), _p(out), _p(labels), int(B))

    def apply_grad(self, w, g, n):
        self._call("pcnn_apply_grad", _p(w), _p(g), int(n))

    def vectorNorm(self, v, n, B, norms):
        self._call("pcnn_vector_norm", _p(v), int(n), int(B), _p(norms))

    def fp_c1(self, inp, pre, w, b, B=1):
        self._call("pcnn_fp_c1", _p(inp), _p(pre), _p(w), _p(b), int(B))

    def fp_s1(self, inp, pre, w, b, B=1):
        self._call("pcnn_fp_s1", _p(inp), _p(pre), _p(w), _p(b), int(B))

    def fp_preact_f(self, inp, pre, w, B=1):
        self._call("pcnn_fp_preact_f", _p(inp), _p(pre), _p(w), int(B))

    def fp_bias_f(self, pre, b, B=1):
        self._call("pcnn_fp_bias_f", _p(pre), _p(b), int(B))

    def bp_weight_f(self, dw, dpre, pout, B=1):
        self._call("pcnn_bp_weight_f", _p(dw), _p(dpre), _p(pout), int(B))

    def bp_bias_f(self, bias, dpre, B=1):
        self._call("pcnn_bp_bias_f", _p(bias), _p(dpre), int(B))

    def bp_output_s1(self, dout, nw, ndpre, B=1):
        self._call("pcnn_bp_output_s1", _p(dout), _p(nw), _p(ndpre), int(B))

    def bp_preact_s1(self, dpre, dout, pre, B=1):
        self._call("pcnn_bp_preact_s1", _p(dpre), _p(dout), _p(pre), int(B))

    def bp_weight_s1(self, dw, dpre, pout, B=1):
        self._call("pcnn_bp_weight_s1", _p(dw), _p(dpre), _p(pout), int(B))

    def bp_bias_s1(self, bias, dpre, B=1):
        self._call("pcnn_bp_bias_s1", _p(bias), _p(dpre), int(B))

    def bp_output_c1(self, dout, nw, ndpre, B=1):
        self._call("pcnn_bp_output_c1", _p(dout), _p(nw), _p(ndpre), int(B))

    def bp_preact_c1(self, dpre, dout, pre, B=1):
        self._call("pcnn_bp_preact_c1", _p(dpre), _p(dout), _p(pre), int(B))

    def bp_weight_c1(self, dw, dpre, pout, B=1):
        self._call("pcnn_bp_weight_c1", _p(dw), _p(dpre), _p(pout), int(B))

    def bp_bias_c1(self, bias, dpre, B=1):
        self._call("pcnn_bp_bias_c1", _p(bias), _p(dpre), int(B))

    # ------------------------------------------------------------------ data + fused path (Main.cpp names)
    def dataset_upload(self, split, images, labels):
        images = np.ascontiguousarray(images)
        labels = np.ascontiguousarray(labels, np.uint8)
        n = labels.shape[0]
        assert images.size == n * 784
        self._call("pcnn_dataset_upload", int(split), images.ctypes.data, _pixel_type(images), labels.ctypes.data, n)

    def dataset_bind(self, split, images_dev, pixel_type, labels_dev, n):
        self._call("pcnn_dataset_bind", int(split), _p(images_dev), int(pixel_type), _p(labels_dev), int(n))

    def train_step(self, first, B):
        self._call("pcnn_train_step", int(first), int(B))

    def train_steps(self, first, B, nsteps):
        self._call("pcnn_train_steps", int(first), int(B), int(nsteps))

    def train_steps_prepare(self, B, nsteps):
        self._call("pcnn_train_steps_prepare", int(B), int(nsteps))

    def train_step_dev(self, images_dev, pixel_type, labels_dev, B):
        self._call("pcnn_train_step_dev", _p(images_dev), int(pixel_type), _p(labels_dev), int(B))

    def train_step_host(self, images, labels):
        images = np.ascontiguousarray(images)
        labels = np.ascontiguousarray(labels, np.uint8)
        e = C.c_float()
        self._call("pcnn_train_step_host", images.ctypes.data, _pixel_type(images), labels.ctypes.data,
                   labels.shape[0], C.byref(e))
        return e.value

    def compute_grads(self, images_dev, pixel_type, labels_dev, B):
        self._call("pcnn_compute_grads", _p(images_dev), int(pixel_type), _p(labels_dev), int(B))

    def learn(self, B=1, epochs=1):
        e = C.c_float()
        self._call("pcnn_learn", int(B), int(epochs), C.byref(e))
        return e.value

    def learn_host(self, images, labels, B=1, epochs=1):
        images = np.ascontiguousarray(images)
        labels = np.ascontiguousarray(labels, np.uint8)
        e = C.c_float()
        self._call("pcnn_learn_host", images.ctypes.data, _pixel_type(images), labels.ctypes.data, labels.shape[0],
                   int(B), int(epochs), C.byref(e))
        return e.value

    def forward_batch(self, images_dev, pixel_type, B, f_out_dev=None, pred_dev=None):
        self._call("pcnn_forward_batch", _p(images_dev), int(pixel_type), int(B), _p(f_out_dev), _p(pred_dev))

    def test(self):
        w = C.c_long()
        self._call("pcnn_test", C.byref(w))
        return w.value

    def step_errs(self):
        n = C.c_long()
        self._call("pcnn_step_errs", None, 0, C.byref(n))
        out = np.empty(n.value, np.float32)
        self._call("pcnn_step_errs", out.ctypes.data, n.value, C.byref(n))
        return out

    def time_fused_kernel(self, B, iters):
        ms = C.c_float()
        self._call("pcnn_time_fused_kernel", int(B), int(iters), C.byref(ms))
        return ms.value

    def measure_fp32_peak(self):
        t = C.c_float()
        self._call("pcnn_measure_fp32_peak", C.byref(t))
        return t.value

    def measure_mma_rate(self, M, N, a_mn=0, b_mn=0, nacc=1, reps=2000):
        t = C.c_float()
        self._call("pcnn_measure_mma_rate", int(M), int(N), int(a_mn), int(b_mn), int(nacc), int(reps), C.byref(t))
        return t.value

    def measure_tma_read(self, dev_bf16, N, P, Q, mode, iters=10):
        t = C.c_float()
        self._call("pcnn_measure_tma_read", _p(dev_bf16), int(N), int(P), int(Q), int(mode), int(iters), C.byref(t))
        return t.value

    def measure_tma_write(self, dev_bf16, N, P, H, row_elems, mode, hot=0, iters=10):
        t = C.c_float()
        self._call("pcnn_measure_tma_write", _p(dev_bf16), int(N), int(P), int(H), int(row_elems), int(mode), int(hot), int(iters), C.byref(t))
        return t.value

    # ------------------------------------------------------------------ data parallel
    @staticmethod
    def comm_unique_id():
        buf = (C.c_char * 256)()
        n = C.c_size_t()
        check("pcnn_comm_unique_id", lib().pcnn_comm_unique_id(buf, C.byref(n)))
        return bytes(buf[: n.value])

    def comm_init_rank(self, uid, rank, world):
        self._call("pcnn_comm_init_rank", C.c_char_p(uid), int(rank), int(world))

    def comm_destroy(self):
        self._call("pcnn_comm_destroy")

    def allreduce_grads(self):
        self._call("pcnn_allreduce_grads")

    def p2p_export(self):
        buf = (C.c_char * 128)()
        n = C.c_size_t()
        self._call("pcnn_p2p_export", buf, C.byref(n))
        return bytes(buf[: n.value])

    def p2p_attach(self, handles, rank, world):
        """handles: list of the `world` byte strings returned by every rank's p2p_export(), in rank order"""
        blob = b"".join(handles)
        self._call("pcnn_p2p_attach", C.c_char_p(blob), int(rank), int(world))

    def p2p_detach(self):
        self._call("pcnn_p2p_detach")

    def set_step_mode(self, mode):
        self._call("pcnn_set_step_mode", int(mode))

    def persist_trace_ctas(self, ctas):
        out = np.zeros((int(ctas), 8), np.int64)
        self._call("pcnn_persist_trace_ctas", out.ctypes.data, int(ctas))
        return out

    def persist_info(self):
        out = np.zeros(6, np.int32)
        self._call("pcnn_persist_info", out.ctypes.data)
        return {"grid": int(out[0]), "cluster": int(out[1]), "cta_capacity": int(out[2]), "cta_capacity_clustered": int(out[3]),
                "cluster_size_used_when_possible": int(out[4]), "cooperative": bool(out[5] & 1), "direct_exchange": bool(out[5] & 2)}

    def persist_tune(self, max_cluster=0):
        self._call("pcnn_persist_tune", int(max_cluster))

    def persist_trace_arm(self):
        self._call("pcnn_persist_trace", None, 0)

    def persist_trace_read(self, steps=256):
        out = np.zeros((steps, 6), np.int64)
        self._call("pcnn_persist_trace", out.ctypes.data, int(steps))
        return out

    # ------------------------------------------------------------------ extension ops
    def maxpool_fwd(self, inp, out, argmax, planes, H, W, k):
        self._call("pcnn_maxpool_fwd", _p(inp), _p(out), _p(argmax), int(planes), int(H), int(W), int(k))

    def maxpool_bwd(self, dout, argmax, din, planes, H, W, k):
        self._call("pcnn_maxpool_bwd", _p(dout), _p(argmax), _p(din), int(planes), int(H), int(W), int(k))

    # LeNet-5-style variant (second convolution layer); all arguments are DeviceArrays
    def l5_compute_grads(self, params, images, pixel_type, labels, B, grads):
        self._call("pcnn_l5_compute_grads", _p(params), _p(images), int(pixel_type), _p(labels), int(B), _p(grads))

    def l5_train_step(self, params, images, pixel_type, labels, B, grads=None):
        self._call("pcnn_l5_train_step", _p(params), _p(images), int(pixel_type), _p(labels), int(B), _p(grads) if grads is not None else None)

    def l5_forward(self, params, images, pixel_type, B, f_out):
        self._call("pcnn_l5_forward", _p(params), _p(images), int(pixel_type), int(B), _p(f_out))

    def conv_bwd_select(self, reference=False):
        """reference=True: the FMA-pipe reference kernels for every shape (explicit opt-in); False: tensor cores only"""
        self._call("pcnn_conv_bwd_select", 1 if reference else 0)

    def conv_wgrad(self, x_bf16, dy_bf16, dw_f32, N, H, W, Cin, K, R, S, row_pitch=0, image_rows=0, stride=1):
        """weight gradient; stride > 1: the window step of a strided forward plan (dy [N][(H-R)//stride+1][(W-S)//stride+1][K])"""
        if stride == 1:
            self._call("pcnn_conv_wgrad", _p(x_bf16), _p(dy_bf16), _p(dw_f32), N, H, W, Cin, K, R, S, int(row_pitch), int(image_rows))
        else:
            self._call("pcnn_conv_wgrad_strided", _p(x_bf16), _p(dy_bf16), _p(dw_f32), N, H, W, Cin, K, R, S, int(stride), int(row_pitch),
                       int(image_rows))

    def conv_dgrad(self, dy_bf16, filt_f32, dx_bf16, N, H, W, Cin, K, R, S, row_pitch=0, image_rows=0, stride=1):
        """input gradient; stride as for conv_wgrad (every dx element is written, those no tap reaches as 0)"""
        if stride == 1:
            self._call("pcnn_conv_dgrad", _p(dy_bf16), _p(filt_f32), _p(dx_bf16), N, H, W, Cin, K, R, S, int(row_pitch), int(image_rows))
        else:
            self._call("pcnn_conv_dgrad_strided", _p(dy_bf16), _p(filt_f32), _p(dx_bf16), N, H, W, Cin, K, R, S, int(stride), int(row_pitch),
                       int(image_rows))

    def pad_nhwc(self, src_bf16, dst_bf16, N, H, W, Cin, pad_h, pad_w, dst_row_pitch=0, dst_image_rows=0):
        self._call("pcnn_pad_nhwc_bf16", _p(src_bf16), _p(dst_bf16), N, H, W, Cin, int(pad_h), int(pad_w), int(dst_row_pitch), int(dst_image_rows))

    def crop_nhwc(self, src_bf16, dst_bf16, N, H, W, Cin, pad_h, pad_w, src_row_pitch=0, src_image_rows=0):
        self._call("pcnn_crop_nhwc_bf16", _p(src_bf16), _p(dst_bf16), N, H, W, Cin, int(pad_h), int(pad_w), int(src_row_pitch), int(src_image_rows))

    def softmax_ce(self, logits, labels, B, n, prob=None, d=None, loss=None):
        self._call("pcnn_softmax_ce", _p(logits), _p(labels), int(B), int(n), _p(prob), _p(d), _p(loss))


class ConvPlan:
    """bf16 tensor-core convolution plan (pcnn_conv_tc_*): filters fp32 KRSC on the host, activations NHWC bf16."""

    def __init__(self, engine, N, H, W, C, K, R, S, filt, bias=None, act=0, row_pitch=None, image_rows=0, stride=1):
        self.engine = engine
        self.shape = (N, H, W, C, K, R, S)
        self.row_pitch = int(row_pitch if row_pitch is not None else (W * C + 7) // 8 * 8)
        filt = np.ascontiguousarray(filt, np.float32)
        assert filt.size == K * R * S * C
        b = None if bias is None else np.ascontiguousarray(bias, np.float32)
        plan = C_.c_void_p()
        check("pcnn_conv_tc_plan_create_strided",
              lib().pcnn_conv_tc_plan_create_strided(engine.ctx, N, H, W, C, K, R, S, int(stride), self.row_pitch, int(image_rows), int(act),
                                                     filt.ctypes.data, None if b is None else b.ctypes.data, C_.byref(plan)))
        self.plan = plan
        self.out_shape = (N, (H - R) // stride + 1, (W - S) // stride + 1, K)

    def fwd(self, x_bf16_dev, y_bf16_dev):
        check("pcnn_conv_tc_fwd", lib().pcnn_conv_tc_fwd(self.engine.ctx, self.plan, _p(x_bf16_dev), _p(y_bf16_dev)))

    def close(self):
        if self.plan and self.engine.ctx:
            lib().pcnn_conv_tc_plan_destroy(self.engine.ctx, self.plan)
        self.plan = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def f32_to_bf16_bits(a):
    """numpy float32 -> uint16 bf16 bit patterns (round to nearest even), the rounding the kernels use"""
    u = np.ascontiguousarray(a, np.float32).view(np.uint32).astype(np.uint64)
    u = u + 0x7FFF + ((u >> 16) & 1)
    return (u >> 16).astype(np.uint16)


def bf16_bits_to_f32(b):
    return (np.ascontiguousarray(b, np.uint16).astype(np.uint32) << 16).view(np.float32)


C_ = C
__all__ = ["Engine", "DeviceArray", "ConvPlan", "f32_to_bf16_bits", "bf16_bits_to_f32", "TRAIN_SET", "TEST_SET", "U8", "F32"]
