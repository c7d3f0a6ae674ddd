"""ctypes binding of include/gtn_b200.h (the C-ABI shared library).

This module never computes anything itself: every call goes into
``gtn_b200/lib/libgtn_b200.so`` (hand-written sm_100a CUDA).  If the library is
missing, or no CUDA device is usable, it raises -- there is no CPU fallback.
"""
import ctypes as C
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "lib", "libgtn_b200.so")

OK = 0
ERR_INVALID_ARGUMENT = 2
ERR_LOGIC = 3
ERR_RUNTIME = 4
ERR_UNSUPPORTED = 5
EPSILON = -1

_f32p = C.POINTER(C.c_float)
_i32p = C.POINTER(C.c_int32)
_u8p = C.POINTER(C.c_uint8)
_vp = C.c_void_p


class GraphView(C.Structure):
    _fields_ = [
        ("num_nodes", C.c_int32), ("num_arcs", C.c_int32),
        ("node_flags", _u8p),
        ("arc_src", _i32p), ("arc_dst", _i32p), ("arc_ilabel", _i32p), ("arc_olabel", _i32p),
        ("weights", _f32p),
        ("in_ptr", _i32p), ("in_arcs", _i32p), ("out_ptr", _i32p), ("out_arcs", _i32p),
        ("start", _i32p), ("num_start", C.c_int32),
        ("accept", _i32p), ("num_accept", C.c_int32),
    ]


# every symbol include/gtn_b200.h declares: (name, restype, argtypes)
SYMBOLS = [
    ("gtnb_version", C.c_int, []),
    ("gtnb_ctx_create", C.c_int, [C.c_int, _vp, C.POINTER(_vp)]),
    ("gtnb_ctx_destroy", None, [_vp]),
    ("gtnb_last_error", C.c_char_p, [_vp]),
    ("gtnb_ctx_synchronize", C.c_int, [_vp]),
    ("gtnb_ctx_stream", _vp, [_vp]),
    ("gtnb_ctx_device", C.c_int, [_vp]),
    ("gtnb_ctx_launch_count", C.c_int64, [_vp]),
    ("gtnb_ctx_set_flag", C.c_int, [_vp, C.c_char_p, C.c_int]),
    ("gtnb_device_alloc", C.c_int, [_vp, C.c_size_t, C.POINTER(_vp)]),
    ("gtnb_device_free", C.c_int, [_vp, _vp]),
    ("gtnb_host_alloc", C.c_int, [_vp, C.c_size_t, C.POINTER(_vp)]),
    ("gtnb_host_free", C.c_int, [_vp, _vp]),
    ("gtnb_memcpy_h2d", C.c_int, [_vp, _vp, _vp, C.c_size_t]),
    ("gtnb_memcpy_d2h", C.c_int, [_vp, _vp, _vp, C.c_size_t]),
    ("gtnb_memset", C.c_int, [_vp, _vp, C.c_int, C.c_size_t]),
    ("gtnb_timer_start", C.c_int, [_vp]),
    ("gtnb_timer_stop", C.c_int, [_vp, _f32p]),
    ("gtnb_flush_l2", C.c_int, [_vp]),
    ("gtnb_profile_enable", C.c_int, [_vp, C.c_int]),
    ("gtnb_profile_read", C.c_char_p, [_vp]),
    ("gtnb_pack", C.c_int, [_vp, C.c_int, C.POINTER(GraphView), C.POINTER(_vp)]),
    ("gtnb_compose_linear", C.c_int,
     [_vp, C.c_int, C.POINTER(GraphView), C.c_int, C.c_int, _i32p, C.c_int, _vp, C.c_int64,
      C.POINTER(_vp)]),
    ("gtnb_compose_graphs", C.c_int,
     [_vp, C.c_int, C.POINTER(GraphView), C.c_int, C.POINTER(GraphView), C.c_int, _i32p, C.POINTER(_vp)]),
    ("gtnb_composed_sizes", C.c_int, [_vp, C.c_int, _i32p, _i32p]),
    ("gtnb_composed_download", C.c_int,
     [_vp, _vp, C.c_int, _u8p, _i32p, _i32p, _i32p, _i32p, _f32p, _i32p, _i32p]),
    ("gtnb_composed_destroy", None, [_vp, _vp]),
    ("gtnb_lattice_destroy", None, [_vp, _vp]),
    ("gtnb_lattice_batch", C.c_int, [_vp]),
    ("gtnb_lattice_sizes", C.c_int, [_vp, _vp, _i32p, _i32p]),
    ("gtnb_lattice_download", C.c_int,
     [_vp, _vp, C.c_int, _u8p, _i32p, _i32p, _i32p, _i32p, _f32p, _i32p, _i32p]),
    ("gtnb_forward", C.c_int, [_vp, _vp, C.c_int, _f32p, _i32p]),
    ("gtnb_backward", C.c_int, [_vp, _vp, C.c_int, _f32p]),
    ("gtnb_lattice_arc_grads", C.c_int, [_vp, _vp, C.c_int, _f32p]),
    ("gtnb_lattice_arc_grads_dev", _vp, [_vp]),
    ("gtnb_lattice_set_arc_grads", C.c_int, [_vp, _vp, C.c_int, _f32p]),
    ("gtnb_compose_grad", C.c_int, [_vp, _vp, _vp, _vp, C.c_int64]),
    ("gtnb_viterbi_path", C.c_int, [_vp, _vp, C.c_int, _i32p, _i32p, _i32p, _f32p, _i32p, _i32p]),
    ("gtnb_linear_forward", C.c_int,
     [_vp, C.c_int, _i32p, C.c_int, _vp, C.c_int64, C.c_int, _vp, _vp, C.c_int64, _vp, C.c_float]),
    ("gtnb_asg_loss", C.c_int,
     [_vp, C.c_int, C.c_int, C.c_int, _vp, C.c_int, _f32p, _i32p, _i32p, _f32p, _vp, C.c_int, _f32p]),
    ("gtnb_viterbi_dense", C.c_int,
     [_vp, C.c_int, C.c_int, C.c_int, _vp, C.c_int, _i32p, _f32p, _i32p, _f32p]),
    ("gtnb_ctc_loss", C.c_int,
     [_vp, C.c_int, C.c_int, C.c_int, _vp, C.c_int, _i32p, _i32p, _i32p, C.c_int, _f32p, _vp,
      C.c_int]),
    ("gtnb_ctc_align", C.c_int,
     [_vp, C.c_int, C.c_int, C.c_int, _vp, C.c_int, _i32p, _i32p, _i32p, C.c_int, C.c_int, _vp, _vp, C.c_int,
      _f32p]),
]

_lib = None


def lib():
    """Load the shared library (once) and declare every prototype."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                "gtn_b200: %s is missing -- run `python -c 'import __graft_entry__ as g; g.build()'` "
                "(there is no CPU fallback)" % LIB_PATH)
        L = C.CDLL(LIB_PATH)
        for name, res, args in SYMBOLS:
            fn = getattr(L, name)
            fn.restype = res
            fn.argtypes = args
        _lib = L
    return _lib


class GtnbError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(msg)
        self.code = code


class GtnbInvalidArgument(GtnbError, ValueError):
    """std::invalid_argument in the reference -> ValueError through pybind11."""


def _raise(code, msg):
    if code == ERR_INVALID_ARGUMENT:
        raise GtnbInvalidArgument(code, msg)
    raise GtnbError(code, msg)


def _p(a, t):
    return None if a is None else a.ctypes.data_as(t)


def make_view(flags, src, dst, ilabel, olabel, weights=None, in_ptr=None, in_arcs=None,
              out_ptr=None, out_arcs=None, start=None, accept=None):
    """Build a GraphView over numpy arrays; returns (view, keepalive list)."""
    keep = []

    def arr(a, dt):
        if a is None:
            return None
        a = np.ascontiguousarray(a, dtype=dt)
        keep.append(a)
        return a

    flags = arr(flags, np.uint8)
    src, dst = arr(src, np.int32), arr(dst, np.int32)
    ilabel, olabel = arr(ilabel, np.int32), arr(olabel, np.int32)
    weights = arr(weights, np.float32)
    in_ptr, in_arcs = arr(in_ptr, np.int32), arr(in_arcs, np.int32)
    out_ptr, out_arcs = arr(out_ptr, np.int32), arr(out_arcs, np.int32)
    start, accept = arr(start, np.int32), arr(accept, np.int32)
    v = GraphView()
    v.num_nodes = len(flags)
    v.num_arcs = len(src)
    v.node_flags = _p(flags, _u8p)
    v.arc_src, v.arc_dst = _p(src, _i32p), _p(dst, _i32p)
    v.arc_ilabel, v.arc_olabel = _p(ilabel, _i32p), _p(olabel, _i32p)
    v.weights = _p(weights, _f32p)
    v.in_ptr, v.in_arcs = _p(in_ptr, _i32p), _p(in_arcs, _i32p)
    v.out_ptr, v.out_arcs = _p(out_ptr, _i32p), _p(out_arcs, _i32p)
    v.start = _p(start, _i32p)
    v.num_start = 0 if start is None else len(start)
    v.accept = _p(accept, _i32p)
    v.num_accept = 0 if accept is None else len(accept)
    return v, keep


class DeviceBuffer:
    def __init__(self, ctx, nbytes):
        self.ctx = ctx
        self.nbytes = int(nbytes)
        p = _vp()
        ctx._check(lib().gtnb_device_alloc(ctx.h, self.nbytes, C.byref(p)))
        self.ptr = p.value

    def free(self):
        if self.ptr and self.ctx.h:
            lib().gtnb_device_free(self.ctx.h, self.ptr)
        self.ptr = None

    def upload(self, a):
        a = np.ascontiguousarray(a)
        assert a.nbytes <= self.nbytes
        self.ctx._check(lib().gtnb_memcpy_h2d(self.ctx.h, self.ptr, a.ctypes.data, a.nbytes))
        self.ctx.synchronize()
        return self

    def download(self, shape, dtype=np.float32):
        out = np.empty(shape, dtype=dtype)
        assert out.nbytes <= self.nbytes
        self.ctx._check(lib().gtnb_memcpy_d2h(self.ctx.h, out.ctypes.data, self.ptr, out.nbytes))
        self.ctx.synchronize()
        return out

    def zero(self):
        self.ctx._check(lib().gtnb_memset(self.ctx.h, self.ptr, 0, self.nbytes))


class Ctx:
    def __init__(self, device=0, stream=None):
        h = _vp()
        rc = lib().gtnb_ctx_create(device, stream, C.byref(h))
        if rc:
            _raise(rc, lib().gtnb_last_error(None).decode())
        self.h = h.value
        self.device = device

    def close(self):
        if self.h:
            lib().gtnb_ctx_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc):
        if rc:
            _raise(rc, lib().gtnb_last_error(self.h).decode())

    def synchronize(self):
        self._check(lib().gtnb_ctx_synchronize(self.h))

    @property
    def launches(self):
        return lib().gtnb_ctx_launch_count(self.h)

    def alloc(self, nbytes):
        return DeviceBuffer(self, nbytes)

    def to_device(self, a):
        a = np.ascontiguousarray(a)
        return DeviceBuffer(self, max(a.nbytes, 16)).upload(a)

    def timer_start(self):
        self._check(lib().gtnb_timer_start(self.h))

    def timer_stop(self):
        ms = C.c_float()
        self._check(lib().gtnb_timer_stop(self.h, C.byref(ms)))
        return ms.value

    def set_flag(self, name, value):
        self._check(lib().gtnb_ctx_set_flag(self.h, name.encode(), int(value)))

    def profile(self, on=True):
        self._check(lib().gtnb_profile_enable(self.h, int(on)))

    def profile_read(self):
        """-> {kernel name: (launches, total_ms)} since the last read."""
        out = {}
        for line in lib().gtnb_profile_read(self.h).decode().splitlines():
            name, n, ms = line.split()
            out[name] = (int(n), float(ms))
        return out

    def flush_l2(self):
        self._check(lib().gtnb_flush_l2(self.h))

    # ---- graph batches -------------------------------------------------
    def pack(self, views):
        arr = (GraphView * max(len(views), 1))(*[v for v, _ in views])
        h = _vp()
        self._check(lib().gtnb_pack(self.h, len(views), arr, C.byref(h)))
        return Lattice(self, h.value, keep=views)

    def compose_linear(self, views, T, Cn, emissions_dev, stride, linear_first=False, B=None):
        B = len(T) if B is None else B
        arr = (GraphView * max(len(views), 1))(*[v for v, _ in views])
        Tn = np.ascontiguousarray(T, dtype=np.int32)
        h = _vp()
        ptr = emissions_dev.ptr if isinstance(emissions_dev, DeviceBuffer) else emissions_dev
        self._check(lib().gtnb_compose_linear(
            self.h, B, arr, len(views), int(linear_first), _p(Tn, _i32p), Cn, ptr, stride,
            C.byref(h)))
        return Lattice(self, h.value, keep=(views, emissions_dev))

    def linear_forward(self, T, Cn, emissions_dev, stride, tropical=False, grad_dev=None,
                       grad_stride=0, delta=1.0):
        B = len(T)
        Tn = np.ascontiguousarray(T, dtype=np.int32)
        scores = self.alloc(4 * max(B, 1))
        self._check(lib().gtnb_linear_forward(
            self.h, B, _p(Tn, _i32p), Cn, emissions_dev.ptr, stride, int(tropical), scores.ptr,
            None if grad_dev is None else grad_dev.ptr, grad_stride, None, float(delta)))
        out = scores.download((B,))
        scores.free()
        return out

    def asg_loss(self, emissions, trans_w, targets, want_grad=True):
        """Host-buffer entry: -> (losses [B], grads [B,T,C] or None, trans_grad [C + C*C] or None)."""
        e = np.ascontiguousarray(emissions, dtype=np.float32)
        B, T, Cn = e.shape
        tw = np.ascontiguousarray(trans_w, dtype=np.float32)
        lens = np.asarray([len(t) for t in targets], np.int32)
        cat = np.ascontiguousarray(
            np.concatenate([np.asarray(t, np.int32) for t in targets]) if B else np.zeros(0, np.int32), np.int32)
        losses = np.zeros(B, np.float32)
        grads = np.zeros_like(e) if want_grad else None
        tg = np.zeros(Cn + Cn * Cn, np.float32) if want_grad else None
        self._check(lib().gtnb_asg_loss(
            self.h, B, T, Cn, e.ctypes.data, 0, _p(tw, _f32p), _p(cat, _i32p), _p(lens, _i32p),
            _p(losses, _f32p), None if grads is None else grads.ctypes.data, 0, _p(tg, _f32p)))
        return losses, grads, tg

    def viterbi_dense(self, emissions, trans_w, input_lens=None):
        """Host-buffer entry: emissions [B,T,C], trans_w [C + C*C] -> (paths [B,T], scores [B])."""
        e = np.ascontiguousarray(emissions, dtype=np.float32)
        B, T, Cn = e.shape
        tw = np.ascontiguousarray(trans_w, dtype=np.float32)
        assert tw.size == Cn + Cn * Cn
        il = None if input_lens is None else np.ascontiguousarray(input_lens, np.int32)
        paths = np.full((B, max(T, 1)), -1, np.int32)
        scores = np.zeros(max(B, 1), np.float32)
        self._check(lib().gtnb_viterbi_dense(
            self.h, B, T, Cn, e.ctypes.data, 0, _p(il, _i32p), _p(tw, _f32p), _p(paths, _i32p),
            _p(scores, _f32p)))
        return paths[:, :T], scores[:B]

    def ctc_loss(self, emissions, targets, blank=0, want_grad=True, input_lens=None):
        """Host-buffer entry point: emissions [B,T,C] float32 numpy -> (losses, grads)."""
        e = np.ascontiguousarray(emissions, dtype=np.float32)
        B, T, Cn = e.shape
        lens = np.asarray([len(t) for t in targets], np.int32)
        cat = (np.concatenate([np.asarray(t, np.int32) for t in targets])
               if B else np.zeros(0, np.int32))
        cat = np.ascontiguousarray(cat, np.int32)
        il = None if input_lens is None else np.ascontiguousarray(input_lens, np.int32)
        losses = np.zeros(B, np.float32)
        grads = np.zeros_like(e) if want_grad else None
        self._check(lib().gtnb_ctc_loss(
            self.h, B, T, Cn, e.ctypes.data, 0, _p(il, _i32p), _p(cat, _i32p), _p(lens, _i32p),
            blank, _p(losses, _f32p), None if grads is None else grads.ctypes.data, 0))
        return losses, grads

    def ctc_loss_dev(self, emissions, targets, blank=0, input_lens=None):
        """Device-buffer entry point: uploads once, runs gtnb_ctc_loss on device pointers (emissions
        in HBM in, gradients in HBM out), downloads the gradients afterwards -> (losses, grads)."""
        e = np.ascontiguousarray(emissions, dtype=np.float32)
        B, T, Cn = e.shape
        lens = np.asarray([len(t) for t in targets], np.int32)
        cat = np.ascontiguousarray(np.concatenate([np.asarray(t, np.int32) for t in targets]), np.int32)
        il = None if input_lens is None else np.ascontiguousarray(input_lens, np.int32)
        losses = np.zeros(B, np.float32)
        e_dev = self.to_device(e)
        g_dev = self.alloc(e.nbytes)
        try:
            self._check(lib().gtnb_ctc_loss(
                self.h, B, T, Cn, e_dev.ptr, 1, _p(il, _i32p), _p(cat, _i32p), _p(lens, _i32p),
                blank, _p(losses, _f32p), g_dev.ptr, 1))
            grads = g_dev.download(e.shape)
        finally:
            e_dev.free()
            g_dev.free()
        return losses, grads

    @staticmethod
    def _align_args(emissions, targets, input_lens):
        e = np.ascontiguousarray(emissions, dtype=np.float32)
        lens = np.asarray([len(t) for t in targets], np.int32)
        cat = np.ascontiguousarray(
            np.concatenate([np.asarray(t, np.int32) for t in targets]) if len(targets) else np.zeros(0, np.int32),
            np.int32)
        il = None if input_lens is None else np.ascontiguousarray(input_lens, np.int32)
        return e, lens, cat, il

    def ctc_align(self, emissions, targets, blank=0, input_lens=None, arc_sorted=True, want_states=False):
        """Host-buffer entry of gtnb_ctc_align: emissions [B,T,C] -> (labels [B,T], scores [B], states [B,T] or
        None): the best path of intersect(ctcGraph(target_b), emissions_b), -1 past input_lens[b] or without a path."""
        e, lens, cat, il = self._align_args(emissions, targets, input_lens)
        B, T, Cn = e.shape
        labels = np.full((B, max(T, 1)), -7, np.int32)
        states = np.full_like(labels, -7) if want_states else None
        scores = np.zeros(max(B, 1), np.float32)
        self._check(lib().gtnb_ctc_align(
            self.h, B, T, Cn, e.ctypes.data, 0, _p(il, _i32p), _p(cat, _i32p), _p(lens, _i32p), int(blank),
            int(arc_sorted), labels.ctypes.data, None if states is None else states.ctypes.data, 0,
            _p(scores, _f32p)))
        return labels[:, :T], scores[:B], None if states is None else states[:, :T]

    def ctc_align_dev(self, emissions, targets, blank=0, input_lens=None, arc_sorted=True, want_states=False):
        """Device-buffer entry of gtnb_ctc_align: emissions uploaded once, labels / states written to device
        buffers and downloaded afterwards -> the same as ctc_align."""
        e, lens, cat, il = self._align_args(emissions, targets, input_lens)
        B, T, Cn = e.shape
        scores = np.zeros(max(B, 1), np.float32)
        e_dev = self.to_device(e)
        l_dev = self.alloc(4 * max(B * T, 1))
        s_dev = self.alloc(4 * max(B * T, 1)) if want_states else None
        try:
            self._check(lib().gtnb_ctc_align(
                self.h, B, T, Cn, e_dev.ptr, 1, _p(il, _i32p), _p(cat, _i32p), _p(lens, _i32p), int(blank),
                int(arc_sorted), l_dev.ptr, None if s_dev is None else s_dev.ptr, 1, _p(scores, _f32p)))
            labels = l_dev.download((B, T), np.int32)
            states = None if s_dev is None else s_dev.download((B, T), np.int32)
        finally:
            e_dev.free()
            l_dev.free()
            if s_dev is not None:
                s_dev.free()
        return labels, scores[:B], states


class Lattice:
    def __init__(self, ctx, h, keep=None):
        self.ctx = ctx
        self.h = h
        self._keep = keep
        self.B = lib().gtnb_lattice_batch(h)

    def free(self):
        if self.h and self.ctx.h:
            lib().gtnb_lattice_destroy(self.ctx.h, self.h)
        self.h = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass

    def sizes(self):
        n = np.zeros(max(self.B, 1), np.int32)
        a = np.zeros(max(self.B, 1), np.int32)
        self.ctx._check(lib().gtnb_lattice_sizes(self.ctx.h, self.h, _p(n, _i32p), _p(a, _i32p)))
        return n[:self.B], a[:self.B]

    def download(self, b):
        nn, na = self.sizes()
        N, A = int(nn[b]), int(na[b])
        flags = np.zeros(max(N, 1), np.uint8)
        src, dst, il, ol, gg, gl = (np.zeros(max(A, 1), np.int32) for _ in range(6))
        w = np.zeros(max(A, 1), np.float32)
        self.ctx._check(lib().gtnb_lattice_download(
            self.ctx.h, self.h, b, _p(flags, _u8p), _p(src, _i32p), _p(dst, _i32p), _p(il, _i32p),
            _p(ol, _i32p), _p(w, _f32p), _p(gg, _i32p), _p(gl, _i32p)))
        return dict(flags=flags[:N], src=src[:A], dst=dst[:A], ilabel=il[:A], olabel=ol[:A],
                    w=w[:A], gi_graph=gg[:A], gi_linear=gl[:A])

    def forward(self, tropical=False, want_status=False):
        scores = np.zeros(max(self.B, 1), np.float32)
        status = np.zeros(max(self.B, 1), np.int32)
        rc = lib().gtnb_forward(self.ctx.h, self.h, int(tropical), _p(scores, _f32p), _p(status, _i32p))
        if want_status:
            if rc not in (OK, ERR_INVALID_ARGUMENT):
                self.ctx._check(rc)
            return scores[:self.B], status[:self.B]
        self.ctx._check(rc)
        return scores[:self.B]

    def backward(self, tropical=False, deltas=None):
        d = None if deltas is None else np.ascontiguousarray(deltas, np.float32)
        self.ctx._check(lib().gtnb_backward(self.ctx.h, self.h, int(tropical), _p(d, _f32p)))

    def arc_grads(self, b, num_arcs):
        out = np.zeros(max(num_arcs, 1), np.float32)
        self.ctx._check(lib().gtnb_lattice_arc_grads(self.ctx.h, self.h, b, _p(out, _f32p)))
        return out[:num_arcs]

    def compose_grad(self, grad_graph_dev=None, grad_emissions_dev=None, grad_stride=0):
        self.ctx._check(lib().gtnb_compose_grad(
            self.ctx.h, self.h,
            None if grad_graph_dev is None else grad_graph_dev.ptr,
            None if grad_emissions_dev is None else grad_emissions_dev.ptr, grad_stride))

    def viterbi_path(self, max_len, want_status=False):
        B = self.B
        arcs = np.full((max(B, 1), max(max_len, 1)), -1, np.int32)
        il = np.full_like(arcs, -1)
        ol = np.full_like(arcs, -1)
        lens = np.zeros(max(B, 1), np.int32)
        status = np.zeros(max(B, 1), np.int32)
        pw = np.zeros(arcs.shape, np.float32)
        rc = lib().gtnb_viterbi_path(
            self.ctx.h, self.h, max_len, _p(arcs, _i32p), _p(il, _i32p), _p(ol, _i32p),
            _p(pw, _f32p), _p(lens, _i32p), _p(status, _i32p))
        if want_status:
            if rc not in (OK, ERR_INVALID_ARGUMENT):
                self.ctx._check(rc)
        else:
            self.ctx._check(rc)
        out = dict(arcs=arcs[:B], ilabels=il[:B], olabels=ol[:B], lens=lens[:B], weights=pw[:B])
        return (out, status[:B]) if want_status else out
