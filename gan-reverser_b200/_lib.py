"""ctypes binding of libganrev_cuda.so (include/ganrev.h).  No fallback: if the CUDA library
is missing or no sm_100 GPU is present, every entry point raises."""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
# GANREV_CUDA_LIB: another build of the SAME library (e.g. `make trace`), never a different backend
SO_PATH = os.environ.get("GANREV_CUDA_LIB") or os.path.join(_HERE, "libganrev_cuda.so")

OK, EINVAL, ECUDA, ENODEV, ESTATE, ENCCL, ENOMEM = range(7)
BUF_NOISE, BUF_IMAGES, BUF_ATTRS0, BUF_ATTRS1, BUF_FIXED, BUF_MASK = range(6)


class GanrevError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"ganrev error {code}: {msg}")
        self.code = code


_lib = None
_vp, _i, _i64, _sz = C.c_void_p, C.c_int, C.c_int64, C.c_size_t

_SIGS = {
    "ganrev_version": (_i, []),
    "ganrev_create": (_i, [C.POINTER(_vp), _i]),
    "ganrev_destroy": (None, [_vp]),
    "ganrev_last_error": (C.c_char_p, [_vp]),
    "ganrev_comm_unique_id": (_i, [_vp, _vp, _sz, C.POINTER(_sz)]),
    "ganrev_comm_init": (_i, [_vp, _i, _i, _vp, _sz]),
    "ganrev_load_G": (_i, [_vp, _i, _i, _i, _i, _vp, _sz]),
    "ganrev_load_R": (_i, [_vp, _i, _i, _i, _i, _i, _i, _vp, _sz]),
    "ganrev_forward_G": (_i, [_vp, _vp, _i64, _vp]),
    "ganrev_forward_R": (_i, [_vp, _i, _vp, _vp, _i64, _vp]),
    "ganrev_fix_l2": (_i, [_vp, _i, _vp, _vp, _i64, _vp, _vp, _vp]),
    "ganrev_l2": (_i, [_vp, _vp, _vp, _i64, _i, _vp]),
    "ganrev_nearest_l2": (_i, [_vp, _vp, _i, _vp, _i64, _i, _vp, _vp]),
    "ganrev_refine_l2": (_i, [_vp, _i, _vp, _vp, _i64, _i, _vp, _vp, _vp, _vp]),
    "ganrev_debug_refine_grad": (_i, [_vp, _vp, _vp, _i64, C.c_float, _vp, _vp]),
    "ganrev_debug_refine_stage": (_i, [_vp, _vp, _vp, _i64, _i, _vp, _sz]),
    "ganrev_refine_masked_l2": (_i, [_vp, _i, _vp, _vp, _vp, _i64, _i, _vp, _vp, _vp, _vp]),
    "ganrev_debug_refine_masked_stage": (_i, [_vp, _vp, _vp, _vp, _i64, _i, _vp, _sz]),
    "ganrev_debug_G_stage": (_i, [_vp, _vp, _i64, _i, _vp, _sz]),
    "ganrev_debug_R_stage": (_i, [_vp, _i, _vp, _vp, _i64, _i, _vp, _sz]),
    "ganrev_train_R_init": (_i, [_vp, _i, _i, _i, _i, _i, _i, _vp, _sz]),
    "ganrev_train_R_step": (_i, [_vp, _vp, _i, _vp, _sz, _vp, _vp]),
    "ganrev_train_R_state": (_i, [_vp, _i, _vp, _sz]),
    "ganrev_anomaly_flags": (_i, [_vp, _vp, _i64, _i64, C.c_double, _vp, C.POINTER(C.c_double)]),
    "ganrev_buffer_put": (_i, [_vp, _i, _vp, _i64]),
    "ganrev_buffer_get": (_i, [_vp, _i, _vp, _i64, _i64]),
    "ganrev_db_set": (_i, [_vp, _vp, _i64, _i]),
    "ganrev_cosine": (_i, [_vp, _vp, _vp, _i, C.POINTER(C.c_float)]),
    "ganrev_search_cosine": (_i, [_vp, _vp, _i, _i, _vp, _vp]),
    "ganrev_search_rows": (_i, [_vp, _vp, _i, _i, _vp, _vp]),
    "ganrev_kmeans": (_i, [_vp, _i, _i, _vp, _vp, _vp, _vp]),
    "ganrev_assign_cosine_min": (_i, [_vp, _vp, _i, _vp, _vp]),
    "ganrev_cluster_members": (_i, [_vp, _i, _i, _vp, _i, _vp, _vp, _vp]),
    "ganrev_stream": (_vp, [_vp]),
    "ganrev_sync": (_i, [_vp]),
    "ganrev_launch_count": (C.c_uint64, [_vp]),
    "ganrev_profile_enable": (_i, [_vp, _i]),
    "ganrev_profile_reset": (_i, [_vp]),
    "ganrev_profile_count": (_i, [_vp]),
    "ganrev_profile_get": (_i, [_vp, _i, C.POINTER(C.c_char_p), C.POINTER(C.c_uint64), C.POINTER(C.c_double),
                                C.POINTER(C.c_double), C.POINTER(C.c_double)]),
    "ganrev_set_option": (_i, [_vp, C.c_char_p, _i64]),
    "ganrev_debug_db_synthetic": (_i, [_vp, _i64, _i, C.c_uint64, _i64]),
    "ganrev_debug_fma_peak": (_i, [_vp, C.POINTER(C.c_double)]),
    "ganrev_debug_tc_scores": (_i, [_vp, _vp, _i, _vp, C.POINTER(C.c_float)]),
    "ganrev_debug_tc_counters": (_i, [_vp, _vp]),
    "ganrev_debug_tfs_stats": (_i, [_vp, _vp]),
    "ganrev_debug_trace_arm": (_i, [_vp, C.c_char_p]),
    "ganrev_debug_trace_read": (_i, [_vp, _vp]),
}
EXPORTS = sorted(_SIGS)


def lib():
    """Load the CUDA library (loudly failing if it has not been built)."""
    global _lib
    if _lib is None:
        if not os.path.exists(SO_PATH):
            raise GanrevError(ENODEV, f"{SO_PATH} is missing -- run __graft_entry__.build(); there is no CPU fallback")
        L = C.CDLL(SO_PATH)
        for name, (res, args) in _SIGS.items():
            fn = getattr(L, name)
            fn.restype = res
            fn.argtypes = args
        _lib = L
    return _lib


def _ptr(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def _arr(a, dtype):
    if a is None:
        return None
    return np.ascontiguousarray(a, dtype=dtype)


class Context:
    """One GPU (ganrev_ctx).  All array arguments are numpy arrays on the host."""

    def __init__(self, device=0):
        self._h = C.c_void_p()
        rc = lib().ganrev_create(C.byref(self._h), int(device))
        if rc != OK:
            self._h = None
            raise GanrevError(rc, "ganrev_create failed (needs an sm_100 GPU; there is no CPU fallback)")
        self.device = int(device)
        self.geom = None       # (C, H, W, nd)
        self.db_shape = None   # (N local rows, d) of the database set by db_set
        self.world, self.rank = 1, 0

    def close(self):
        if getattr(self, "_h", None):
            lib().ganrev_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _chk(self, rc):
        if rc != OK:
            raise GanrevError(rc, lib().ganrev_last_error(self._h).decode())

    # ---- multi-GPU
    def comm_unique_id(self):
        buf = C.create_string_buffer(256)
        n = C.c_size_t(0)
        self._chk(lib().ganrev_comm_unique_id(self._h, buf, 256, C.byref(n)))
        return buf.raw[:n.value]

    def comm_init(self, world, rank, uid):
        self._chk(lib().ganrev_comm_init(self._h, world, rank, uid, len(uid)))
        self.world, self.rank = world, rank

    # ---- models
    def load_G(self, Cc, H, W, nd, blob):
        blob = _arr(blob, np.float32)
        self._chk(lib().ganrev_load_G(self._h, Cc, H, W, nd, _ptr(blob), blob.size))
        self.geom = (Cc, H, W, nd)

    def load_R(self, slot, Cc, H, W, nd, blob, tanh_out=False):
        blob = _arr(blob, np.float32)
        self._chk(lib().ganrev_load_R(self._h, slot, Cc, H, W, nd, int(bool(tanh_out)), _ptr(blob), blob.size))
        self.geom = (Cc, H, W, nd)     # one geometry per context (ganrev.h): a different one unloaded the old models

    def forward_G(self, noise, N=None, want_images=True, out=None):
        Cc, H, W, nd = self.geom
        noise = _arr(noise, np.float32)
        if noise is not None:
            N = noise.shape[0]
            assert noise.shape[1] == nd
        images = None
        if want_images:
            images = out if out is not None else np.empty((N, Cc, H, W), np.float32)
        self._chk(lib().ganrev_forward_G(self._h, _ptr(noise), N, _ptr(images)))
        return images

    def forward_R(self, slot, images, mask=None, N=None, want_attrs=True, out=None):
        Cc, H, W, nd = self.geom
        images = _arr(images, np.float32)
        mask = _arr(mask, np.uint8)
        if images is not None:
            N = images.shape[0]
            assert images.shape[1:] == (Cc, H, W), images.shape
        if mask is not None:
            assert mask.size == N * Cc * H * W
        attrs = None
        if want_attrs:
            attrs = out if out is not None else np.empty((N, nd), np.float32)
        self._chk(lib().ganrev_forward_R(self._h, slot, _ptr(images), _ptr(mask), N, _ptr(attrs)))
        return attrs

    def fix_l2(self, slot, images, mask=None, N=None, want_attrs=True, want_fixed=True):
        Cc, H, W, nd = self.geom
        images = _arr(images, np.float32)
        mask = _arr(mask, np.uint8)
        if images is not None:
            N = images.shape[0]
        attrs = np.empty((N, nd), np.float32) if want_attrs else None
        fixed = np.empty((N, Cc, H, W), np.float32) if want_fixed else None
        l2 = np.empty((N,), np.float64)
        self._chk(lib().ganrev_fix_l2(self._h, slot, _ptr(images), _ptr(mask), N, _ptr(attrs), _ptr(fixed), _ptr(l2)))
        return attrs, fixed, l2

    def l2(self, a, b):
        a, b = _arr(a, np.float32), _arr(b, np.float32)
        N = a.shape[0]
        px = a.size // max(N, 1)
        assert a.size == b.size
        out = np.empty((N,), np.float64)
        self._chk(lib().ganrev_l2(self._h, _ptr(a), _ptr(b), N, px, _ptr(out)))
        return out

    def nearest_l2(self, queries, images=None, N=None):
        """sample.lua:128-148: per query image the set image with the first strictly smallest torch.dist.
        images=None scans the first N resident IMAGES.  Returns (ids int64 [Q], dist float64 [Q])."""
        q = _arr(queries, np.float32)
        Q = q.shape[0]
        px = q.size // max(Q, 1)
        if images is not None:
            x = _arr(images, np.float32)
            N = x.shape[0]
            assert N == 0 or x.size // N == px
            xp = _ptr(x) if N else None
        else:
            assert N is not None
            xp = None
        ids = np.empty((Q,), np.int64)
        dist = np.empty((Q,), np.float64)
        if images is not None and N == 0:
            xp = _ptr(np.zeros((1,), np.float32))   # any non-NULL pointer: an EMPTY explicit set, not the resident images
        self._chk(lib().ganrev_nearest_l2(self._h, _ptr(q), Q, xp, N, px, _ptr(ids), _ptr(dist)))
        return ids, dist

    # ---- noise-vector refinement (new work: gradient descent through G from R's guess)
    def refine_l2(self, slot, images, z0=None, iters=100, N=None, lr=0.01, beta1=0.9, beta2=0.999, eps=1e-8, prior=0.0, zclamp=0.0,
                  want_attrs=True, want_fixed=True):
        """`iters` Adam steps per image on ||G(z) - x||^2 + prior ||z||^2 from z0 (None: the resident ATTRS_slot rows), |z| <= zclamp
        after each step if zclamp > 0.  images=None uses the resident IMAGES (then N is required).  Returns (z_final, G(z_final), l2)."""
        Cc, H, W, nd = self.geom
        images = _arr(images, np.float32)
        z0 = _arr(z0, np.float32)
        if images is not None:
            N = images.shape[0]
            assert images.shape[1:] == (Cc, H, W), images.shape
        if z0 is not None:
            assert z0.shape == (N, nd), z0.shape
        hy = np.array([lr, beta1, beta2, eps, prior, zclamp], np.float32)
        attrs = np.empty((N, nd), np.float32) if want_attrs else None
        fixed = np.empty((N, Cc, H, W), np.float32) if want_fixed else None
        l2 = np.empty((N,), np.float64)
        self._chk(lib().ganrev_refine_l2(self._h, slot, _ptr(images), _ptr(z0), N, int(iters), _ptr(hy), _ptr(attrs), _ptr(fixed), _ptr(l2)))
        return attrs, fixed, l2

    def debug_refine_grad(self, images, z, prior=0.0):
        """Tests: (gradient of ||G(z) - x||^2 + prior ||z||^2 [N x nd], f [N]) from one forward + backward pass of G."""
        images, z = _arr(images, np.float32), _arr(z, np.float32)
        N = z.shape[0]
        grad = np.empty_like(z)
        f = np.empty((N,), np.float64)
        self._chk(lib().ganrev_debug_refine_grad(self._h, _ptr(images), _ptr(z), N, float(prior), _ptr(grad), _ptr(f)))
        return grad, f

    REFINE_STAGES = ("h0", "h1", "h2", "y", "e2", "e1", "e0", "glin")

    def _refine_stage_out(self, N, stage):
        Cc, H, W, nd = self.geom
        s = self.REFINE_STAGES.index(stage) if isinstance(stage, str) else int(stage)
        shapes = {0: ((H // 4, W // 4, 512), np.uint16), 1: ((H // 2, W // 2, 256), np.uint16), 2: ((H, W, 128), np.uint16),
                  3: ((Cc, H, W), np.float32), 4: ((H, W, 128), np.uint16), 5: ((H // 2, W // 2, 256), np.uint16),
                  6: ((H // 4, W // 4, 512), np.uint16), 7: ((nd,), np.float32)}
        shape, dt = shapes.get(s, ((1,), np.uint8))
        return s, np.empty((N,) + shape, dt)

    def debug_refine_stage(self, images, z, stage):
        """Tests: the buffer of one stage of refine_l2's forward + backward pass of G (ganrev.h), rows in input order.  bf16 stages
        come back as their uint16 bits, NHWC; y is float32 NCHW, glin float32 [N x nd].  `stage` is an index or a name."""
        images, z = _arr(images, np.float32), _arr(z, np.float32)
        N = z.shape[0]
        s, out = self._refine_stage_out(N, stage)
        self._chk(lib().ganrev_debug_refine_stage(self._h, _ptr(images), _ptr(z), N, s, _ptr(out), out.nbytes))
        return out

    # ---- face completion (new work: refinement against the known pixels only)
    def refine_masked_l2(self, slot, images, mask, z0=None, iters=100, N=None, lr=0.01, beta1=0.9, beta2=0.999, eps=1e-8, prior=0.0,
                         zclamp=0.0, want_attrs=True, want_fixed=True):
        """refine_l2 on sum over mask = 1 of (G(z) - x)^2 + prior ||z||^2; mask is a uint8 keep-mask shaped like images (1 = keep,
        R's input-mask convention).  images / mask / z0 = None use the resident IMAGES / MASK / ATTRS_slot rows (then N is required).
        Returns (z_final, G(z_final), masked l2 = sqrt(sum over mask = 1 of (x - G(z_final))^2), not normalised by the kept count)."""
        Cc, H, W, nd = self.geom
        images = _arr(images, np.float32)
        mask = _arr(mask, np.uint8)
        z0 = _arr(z0, np.float32)
        if images is not None:
            N = images.shape[0]
            assert images.shape[1:] == (Cc, H, W), images.shape
        if mask is not None:
            assert mask.shape == (N, Cc, H, W), mask.shape
        if z0 is not None:
            assert z0.shape == (N, nd), z0.shape
        hy = np.array([lr, beta1, beta2, eps, prior, zclamp], np.float32)
        attrs = np.empty((N, nd), np.float32) if want_attrs else None
        fixed = np.empty((N, Cc, H, W), np.float32) if want_fixed else None
        l2 = np.empty((N,), np.float64)
        self._chk(lib().ganrev_refine_masked_l2(self._h, slot, _ptr(images), _ptr(mask), _ptr(z0), N, int(iters), _ptr(hy),
                                                _ptr(attrs), _ptr(fixed), _ptr(l2)))
        return attrs, fixed, l2

    def debug_refine_masked_stage(self, images, mask, z, stage):
        """Tests: debug_refine_stage with the masked objective (mask: uint8 keep-mask shaped like images)."""
        images, mask, z = _arr(images, np.float32), _arr(mask, np.uint8), _arr(z, np.float32)
        N = z.shape[0]
        assert mask.size == images.size
        s, out = self._refine_stage_out(N, stage)
        self._chk(lib().ganrev_debug_refine_masked_stage(self._h, _ptr(images), _ptr(mask), _ptr(z), N, s, _ptr(out), out.nbytes))
        return out

    G_STAGES = ("lin", "c1", "c2", "taps", "y")
    R_STAGES = ("c1", "c2", "c3", "c4", "c5", "c6", "l1", "out")

    def debug_G_stage(self, noise, stage):
        """Tests: the output of one layer of forward_G (ganrev.h), rows in input order.  bf16 stages come back as their uint16 bits,
        NHWC; taps float32 [N][9C][H][W], y float32 NCHW.  `stage` is an index or a name."""
        Cc, H, W, nd = self.geom
        s = self.G_STAGES.index(stage) if isinstance(stage, str) else int(stage)
        noise = _arr(noise, np.float32)
        shapes = {0: ((H // 4, W // 4, 512), np.uint16), 1: ((H // 2, W // 2, 256), np.uint16), 2: ((H, W, 128), np.uint16),
                  3: ((9 * Cc, H, W), np.float32), 4: ((Cc, H, W), np.float32)}
        shape, dt = shapes.get(s, ((1,), np.uint8))
        out = np.empty((noise.shape[0],) + shape, dt)
        self._chk(lib().ganrev_debug_G_stage(self._h, _ptr(noise), noise.shape[0], s, _ptr(out), out.nbytes))
        return out

    def debug_R_stage(self, slot, images, stage, mask=None):
        """Tests: the output of one layer of forward_R (ganrev.h), rows in input order: bf16 stages as uint16 bits (NHWC; l1 [N][512]),
        out float32 [N][nd]."""
        Cc, H, W, nd = self.geom
        s = self.R_STAGES.index(stage) if isinstance(stage, str) else int(stage)
        images, mask = _arr(images, np.float32), _arr(mask, np.uint8)
        shapes = {0: ((H, W, 64), np.uint16), 1: ((H, W, 64), np.uint16), 2: ((H // 2, W // 2, 64), np.uint16),
                  3: ((H // 2, W // 2, 128), np.uint16), 4: ((H // 2, W // 2, 128), np.uint16), 5: ((H // 4, W // 4, 128), np.uint16),
                  6: ((512,), np.uint16), 7: ((nd,), np.float32)}
        shape, dt = shapes.get(s, ((1,), np.uint8))
        out = np.empty((images.shape[0],) + shape, dt)
        self._chk(lib().ganrev_debug_R_stage(self._h, slot, _ptr(images), _ptr(mask), images.shape[0], s, _ptr(out), out.nbytes))
        return out

    # ---- R training step (train_r.lua:138-170)
    def train_R_init(self, C, H, W, nd, blob, tanh_out=False, fixer=False):
        b = _arr(blob, np.float32)
        self._train_floats = b.size
        self._chk(lib().ganrev_train_R_init(self._h, C, H, W, nd, int(bool(tanh_out)), int(bool(fixer)), _ptr(b), b.size))

    def train_R_step(self, noise, masks, lr=1e-3, beta1=0.9, beta2=0.999, eps=1e-8, l1=0.0, l2=1e-4, clamp=1.0):
        """masks: list of uint8 keep-masks in module order (ganrev.h).  Returns (criterion output, f with penalties)."""
        z = _arr(noise, np.float32)
        m = np.ascontiguousarray(np.concatenate([np.asarray(a, np.uint8).ravel() for a in masks]))
        hy = np.array([lr, beta1, beta2, eps, l1, l2, clamp], np.float32)
        out = np.zeros((2,), np.float64)
        self._chk(lib().ganrev_train_R_step(self._h, _ptr(z), z.shape[0], _ptr(m), m.size, _ptr(hy), _ptr(out)))
        return float(out[0]), float(out[1])

    def train_R_state(self, what=0):
        """0: parameters + running statistics as a weight blob, 1: last gradients (after penalties / clamp), 2 / 3: Adam's m / v."""
        out = np.empty((self._train_floats,), np.float32)
        self._chk(lib().ganrev_train_R_state(self._h, what, _ptr(out), out.size))
        return out

    def anomaly_flags(self, l2, n_calc, n_show, quantile):
        l2 = _arr(l2, np.float64)
        flags = np.zeros((n_show,), np.uint8)
        thr = C.c_double(0.0)
        self._chk(lib().ganrev_anomaly_flags(self._h, _ptr(l2), n_calc, n_show, float(quantile), _ptr(flags), C.byref(thr)))
        return flags, thr.value

    # ---- resident buffers
    def buffer_put(self, which, host):
        dt = np.uint8 if which == BUF_MASK else np.float32
        host = _arr(host, dt)
        self._chk(lib().ganrev_buffer_put(self._h, which, _ptr(host), host.shape[0]))

    def buffer_get(self, which, row0, rows):
        Cc, H, W, nd = self.geom
        if which in (BUF_NOISE, BUF_ATTRS0, BUF_ATTRS1):
            out = np.empty((rows, nd), np.float32)
        elif which == BUF_MASK:
            out = np.empty((rows, Cc, H, W), np.uint8)
        else:
            out = np.empty((rows, Cc, H, W), np.float32)
        self._chk(lib().ganrev_buffer_get(self._h, which, _ptr(out), row0, rows))
        return out

    # ---- database
    def db_set(self, vecs=None, N=None, d=None):
        vecs = _arr(vecs, np.float32)
        if vecs is not None:
            N, d = vecs.shape
        self._chk(lib().ganrev_db_set(self._h, _ptr(vecs), N, d))
        self.db_shape = (N, d)

    def db_synthetic(self, N, d, seed=8, global_row0=0):
        """bench.py: N(0,1) rows generated on the device and adopted as the database."""
        self._chk(lib().ganrev_debug_db_synthetic(self._h, int(N), int(d), int(seed), int(global_row0)))
        self.db_shape = (int(N), int(d))

    def tc_scores(self, queries):
        """Tests: approximate cosines of the tensor-core filter for every (query, row) pair, and the assumed bound eps(d)."""
        q = _arr(queries, np.float32)
        out = np.empty((q.shape[0], self.db_shape[0]), np.float32)
        eps = C.c_float(0.0)
        self._chk(lib().ganrev_debug_tc_scores(self._h, _ptr(q), q.shape[0], _ptr(out), C.byref(eps)))
        return out, eps.value

    def tc_counters(self):
        out = np.zeros((2,), np.uint64)
        self._chk(lib().ganrev_debug_tc_counters(self._h, _ptr(out)))
        return int(out[0]), int(out[1])

    def tfs_stats(self):
        """Counters of the tf32 filter pipeline since the last call: chains on top of the filter, rows sent to the list
        kernel, largest observed error / bound (measured under dbg bit 18), launches."""
        out = np.zeros((4,), np.uint64)
        self._chk(lib().ganrev_debug_tfs_stats(self._h, _ptr(out)))
        return {"chains": int(out[0]), "listed_rows": int(out[1]),
                "max_error_over_bound": float(np.array([int(out[2]) & 0xFFFFFFFF], np.uint32).view(np.float32)[0]), "launches": int(out[3])}

    def fma_peak(self):
        out = C.c_double(0.0)
        self._chk(lib().ganrev_debug_fma_peak(self._h, C.byref(out)))
        return out.value

    def cosine(self, a, b):
        a, b = _arr(a, np.float32).ravel(), _arr(b, np.float32).ravel()
        out = C.c_float(0.0)
        self._chk(lib().ganrev_cosine(self._h, _ptr(a), _ptr(b), a.size, C.byref(out)))
        return out.value

    def search_cosine(self, queries, k):
        queries = _arr(queries, np.float32)
        Q = queries.shape[0]
        ids = np.empty((Q, k), np.int64)
        scores = np.empty((Q, k), np.float32)
        self._chk(lib().ganrev_search_cosine(self._h, _ptr(queries), Q, k, _ptr(ids), _ptr(scores)))
        return ids, scores

    def search_rows(self, rows, k):
        rows = _arr(rows, np.int64)
        Q = rows.shape[0]
        ids = np.empty((Q, k), np.int64)
        scores = np.empty((Q, k), np.float32)
        self._chk(lib().ganrev_search_rows(self._h, _ptr(rows), Q, k, _ptr(ids), _ptr(scores)))
        return ids, scores

    def kmeans(self, k, niter, init, want_labels=True):
        init = _arr(init, np.float32)
        if self.db_shape is None:
            raise GanrevError(ESTATE, "database not set (call db_set first)")
        N, d = self.db_shape
        assert init.shape == (k, d)
        cen = np.empty((k, d), np.float32)
        tot = np.empty((k,), np.float32)
        lab = np.empty((N,), np.int32) if want_labels else None
        self._chk(lib().ganrev_kmeans(self._h, k, niter, _ptr(init), _ptr(cen), _ptr(tot), _ptr(lab)))
        return cen, tot, lab

    def assign_cosine_min(self, centroids):
        centroids = _arr(centroids, np.float32)
        if self.db_shape is None:
            raise GanrevError(ESTATE, "database not set (call db_set first)")
        N, d = self.db_shape
        k = centroids.shape[0]
        cl = np.empty((N,), np.int32)
        cv = np.empty((N,), np.float32)
        self._chk(lib().ganrev_assign_cosine_min(self._h, _ptr(centroids), k, _ptr(cl), _ptr(cv)))
        return cl, cv

    def cluster_members(self, k, m, images=None, px=None, want_mean=True):
        images = _arr(images, np.float32)
        if images is not None:
            px = images.size // images.shape[0]
        ids = np.empty((k, m), np.int64)
        cnt = np.empty((k,), np.int32)
        mean = np.empty((k, px), np.float32) if want_mean else None
        self._chk(lib().ganrev_cluster_members(self._h, k, m, _ptr(images), px or 0, _ptr(ids), _ptr(cnt), _ptr(mean)))
        return ids, cnt, mean

    # ---- measurement
    def stream(self):
        return lib().ganrev_stream(self._h)

    def sync(self):
        self._chk(lib().ganrev_sync(self._h))

    def launch_count(self):
        return int(lib().ganrev_launch_count(self._h))

    def profile_enable(self, on=True):
        self._chk(lib().ganrev_profile_enable(self._h, int(on)))

    def profile_reset(self):
        self._chk(lib().ganrev_profile_reset(self._h))

    def profile(self):
        out = {}
        n = lib().ganrev_profile_count(self._h)
        for i in range(n):
            name, cnt = C.c_char_p(), C.c_uint64()
            ms, fl, by = C.c_double(), C.c_double(), C.c_double()
            self._chk(lib().ganrev_profile_get(self._h, i, C.byref(name), C.byref(cnt), C.byref(ms), C.byref(fl), C.byref(by)))
            out[name.value.decode()] = {"launches": cnt.value, "ms": ms.value, "flops": fl.value, "bytes": by.value}
        return out

    def trace_arm(self, layer):
        self._chk(lib().ganrev_debug_trace_arm(self._h, layer.encode()))

    def trace_read(self):
        out = np.zeros((8, 256), np.int64)
        self._chk(lib().ganrev_debug_trace_read(self._h, _ptr(out)))
        return out

    def set_option(self, name, value):
        self._chk(lib().ganrev_set_option(self._h, name.encode(), int(value)))
