"""Thin Python handle on one `idc_ctx` (one device, one geometry).

Host-side plumbing only: pointer marshalling, torch tensors as device memory, streams.
All arithmetic of the forward happens in libidc_b200.so.
"""
import ctypes

import numpy as np

from . import _lib


def _np_ptr(a):
    return ctypes.c_void_p(a.ctypes.data)


class LhnContext(object):
    """Local Hints Network forward context (the B200 stand-in for
    `SIGGRAPHGenerator(...).cuda().eval()`, /root/reference/data/colorize_image.py:221-232)."""

    def __init__(self, device=0, max_n=1, H=256, W=256, dist=False, engine="tcgen05", fast_fp16=False,
                 global_hints=False, use_graph=True, keep_conv10=False, caffe313=False, options=None):
        """options: {name: int} plan-time switches; the names and values are listed at idc_set_option in
        include/idc_b200.h."""
        self.lib = _lib.load()
        flags = 0
        if dist:
            flags |= _lib.FLAG_DIST
        if engine == "simt":
            flags |= _lib.FLAG_ENGINE_SIMT
        elif engine != "tcgen05":
            raise ValueError("engine must be 'tcgen05' or 'simt'")
        if fast_fp16:
            flags |= _lib.FLAG_FAST_FP16
        if global_hints:
            flags |= _lib.FLAG_GLOBAL_HINTS
        if not use_graph:
            flags |= _lib.FLAG_NO_GRAPH
        if keep_conv10:
            flags |= _lib.FLAG_KEEP_CONV10
        if caffe313:
            flags |= _lib.FLAG_CAFFE313
        self.device, self.max_n, self.H, self.W = int(device), int(max_n), int(H), int(W)
        self.dist, self.global_hints, self.flags = bool(dist), bool(global_hints), flags
        h = ctypes.c_void_p()
        rc = self.lib.idc_create(self.device, self.max_n, self.H, self.W, flags, ctypes.byref(h))
        if rc != _lib.IDC_OK:
            raise _lib.IdcError(rc, "idc_create(device=%d, max_n=%d, %dx%d) failed -- a CUDA sm_100 device is "
                                    "required; there is no CPU fallback" % (device, max_n, H, W))
        self.h = h
        self.ready = False
        self._pinned = []
        # bookkeeping of the reference-facing wrappers that share this context (colorize_image.py: _click)
        self._wrapper_click, self._wrapper_staged_l, self._wrapper_last, self._wrapper_shared = None, [], None, False
        self._dist_resident = False
        for k, v in (options or {}).items():
            self.set_option(k, v)

    def set_option(self, name, value):
        _lib.check(self.h, self.lib.idc_set_option(self.h, name.encode(), int(value)))

    # ---- weights ---------------------------------------------------------------------------
    def load_state_dict(self, sd):
        """sd: {reference state_dict key: torch.Tensor | ndarray}.  Packs + uploads."""
        for k, v in sd.items():
            a = v.detach().cpu().numpy() if hasattr(v, "detach") else np.asarray(v)
            if a.dtype == np.float32:
                dt = _lib.F32
            elif a.dtype == np.float64:
                dt = _lib.F64
            elif a.dtype == np.int64:
                dt = _lib.I64
            else:
                a = a.astype(np.float32)
                dt = _lib.F32
            a = np.ascontiguousarray(a)
            dims = (ctypes.c_int64 * max(a.ndim, 1))(*a.shape)
            _lib.check(self.h, self.lib.idc_load_tensor(self.h, k.encode(), _np_ptr(a), dt, a.ndim, dims))
        _lib.check(self.h, self.lib.idc_finalize_weights(self.h))
        self.ready = True

    def weights_arena(self):
        p, n = ctypes.c_void_p(), ctypes.c_size_t()
        _lib.check(self.h, self.lib.idc_weights_arena(self.h, ctypes.byref(p), ctypes.byref(n)))
        return p.value, n.value

    def reserve_weights(self):
        _lib.check(self.h, self.lib.idc_reserve_weights(self.h))

    def adopt_weights(self):
        _lib.check(self.h, self.lib.idc_adopt_weights(self.h))
        self.ready = True

    # ---- forward ---------------------------------------------------------------------------
    def forward_device(self, L_mc, ab, mask, maskcent=0.0, glob=None, want_dist=False, want_rgb=False,
                       out_ab=None, out_dist=None, out_rgb=None):
        """torch CUDA float32 tensors [n,1,H,W], [n,2,H,W], [n,1,H,W] -> dict of torch tensors.
        Asynchronous on torch's current stream."""
        import torch
        n = L_mc.shape[0]
        for t in (L_mc, ab, mask):
            assert t.is_cuda and t.dtype == torch.float32 and t.is_contiguous()
        dev = L_mc.device
        if out_ab is None:
            out_ab = torch.empty((n, 2, self.H, self.W), dtype=torch.float32, device=dev)
        if want_dist and out_dist is None:
            out_dist = torch.empty((n, 529, self.H // 4, self.W // 4), dtype=torch.float32, device=dev)
        if want_rgb and out_rgb is None:
            out_rgb = torch.empty((n, self.H, self.W, 3), dtype=torch.uint8, device=dev)
        st = torch.cuda.current_stream(dev).cuda_stream
        rc = self.lib.idc_forward(self.h, n, self.H, self.W, L_mc.data_ptr(), ab.data_ptr(), mask.data_ptr(),
                                  float(maskcent), glob.data_ptr() if glob is not None else None,
                                  out_ab.data_ptr(), out_dist.data_ptr() if want_dist else None,
                                  out_rgb.data_ptr() if want_rgb else None, st)
        _lib.check(self.h, rc)
        return {"ab": out_ab, "dist": out_dist if want_dist else None, "rgb": out_rgb if want_rgb else None}

    def set_image(self, L_mc):
        """Upload the mean-centred L planes [n,1,H,W] once (the reference's set_image / load_image half of a session);
        forward_host(None, ab, mask, ...) then reuses them.  None forgets the image."""
        if L_mc is None:
            _lib.check(self.h, self.lib.idc_set_image(self.h, 0, self.H, self.W, None))
            return
        assert L_mc.dtype == np.float32 and L_mc.flags["C_CONTIGUOUS"]
        _lib.check(self.h, self.lib.idc_set_image(self.h, int(L_mc.shape[0]), self.H, self.W, _np_ptr(L_mc)))

    def forward_host(self, L_mc, ab, mask, maskcent=0.0, glob=None, want_dist=False, want_rgb=False,
                     out_ab=None, out_dist=None, out_rgb=None, want_abq=False, out_abq=None):
        """numpy float32 C-contiguous host arrays (pinned or pageable) -> dict of numpy arrays.
        Synchronous; includes H2D + D2H.  want_abq: also the reference's quantised output_ab
        (rgb2lab(rgb)[1:], float64; implies want_rgb).  L_mc None = the image uploaded by set_image."""
        want_rgb = want_rgb or want_abq
        n = ab.shape[0]
        if L_mc is not None:                 # an explicit L replaces the resident image: wrappers must re-stage theirs
            self._wrapper_staged_l, self._wrapper_last = [], None
        for a in (ab, mask) + (() if L_mc is None else (L_mc,)):
            assert a.dtype == np.float32 and a.flags["C_CONTIGUOUS"]
        if out_ab is None:
            out_ab = np.empty((n, 2, self.H, self.W), np.float32)
        if want_dist and out_dist is None:
            out_dist = np.empty((n, 529, self.H // 4, self.W // 4), np.float32)
        if want_rgb and out_rgb is None:
            out_rgb = np.empty((n, self.H, self.W, 3), np.uint8)
        if want_abq and out_abq is None:
            out_abq = np.empty((n, 2, self.H, self.W), np.float64)
        rc = self.lib.idc_forward_host_q(self.h, n, self.H, self.W, None if L_mc is None else _np_ptr(L_mc), _np_ptr(ab), _np_ptr(mask),
                                         float(maskcent), _np_ptr(glob) if glob is not None else None,
                                         _np_ptr(out_ab), _np_ptr(out_dist) if want_dist else None,
                                         _np_ptr(out_rgb) if want_rgb else None,
                                         _np_ptr(out_abq) if want_abq else None)
        _lib.check(self.h, rc)
        return {"ab": out_ab, "dist": out_dist if want_dist else None, "rgb": out_rgb if want_rgb else None,
                "abq": out_abq}

    # ---- zero-copy click path ---------------------------------------------------------------
    def click_buffers(self, n=1, glob=False):
        """Page-locked I/O arrays for the interactive call (n <= 4), laid out back to back so that a click is one H2D and
        one D2H with NO copy by the CPU: pass them to forward_host (L_mc / ab / mask (/ glob) as inputs, out_ab / out_rgb /
        out_abq as outputs).  -> dict of numpy views; they stay valid until close()."""
        HW = self.H * self.W
        n_in = n * 4 * HW + (n * 316 if glob else 0)
        b_ab, b_rgb, b_q = n * 2 * HW * 4, n * 3 * HW, n * 2 * HW * 8
        sizes = (n_in * 4, b_ab + b_rgb + b_q)
        blocks = []
        for nbytes in sizes:
            p = self.lib.idc_host_alloc(nbytes)
            if not p:
                raise _lib.IdcError(-2, "idc_host_alloc(%d) failed" % nbytes)
            self._pinned.append(p)
            blocks.append(np.frombuffer((ctypes.c_char * nbytes).from_address(p), dtype=np.uint8))
        fin = blocks[0].view(np.float32)
        out = {"L_mc": fin[:n * HW].reshape(n, 1, self.H, self.W),
               "ab": fin[n * HW:3 * n * HW].reshape(n, 2, self.H, self.W),
               "mask": fin[3 * n * HW:4 * n * HW].reshape(n, 1, self.H, self.W),
               "glob": fin[4 * n * HW:].reshape(n, 316) if glob else None,
               "out_ab": blocks[1][:b_ab].view(np.float32).reshape(n, 2, self.H, self.W),
               "out_rgb": blocks[1][b_ab:b_ab + b_rgb].reshape(n, self.H, self.W, 3),
               "out_abq": blocks[1][b_ab + b_rgb:].view(np.float64).reshape(n, 2, self.H, self.W)}
        return out

    def set_dist_resident(self, on=True):
        """Interactive mode: the dist head runs on every forward_host but stays on the device."""
        _lib.check(self.h, self.lib.idc_set_dist_resident(self.h, 1 if on else 0))
        self._dist_resident = bool(on)

    def set_click(self, img=0, y4=-1, x4=0, K=0):
        """Announce the clicked pixel of the (H/4 x W/4) grid before forward_host: its pmf and K colour suggestions
        come back with the same graph launch (fetch_dist / ab_reccs for that pixel are then host-side reads).
        y4 < 0 switches the mode off."""
        _lib.check(self.h, self.lib.idc_set_click(self.h, int(img), int(y4), int(x4), int(K)))

    def fetch_dist(self, img=0, y4=None, x4=None):
        """dist[img, :, y4, x4] (529 floats), or the whole [529, H/4, W/4] plane when y4 is None."""
        if y4 is None:
            out = np.empty((529, self.H // 4, self.W // 4), np.float32)
            _lib.check(self.h, self.lib.idc_fetch_dist(self.h, img, -1, 0, _np_ptr(out)))
        else:
            out = np.empty((529,), np.float32)
            _lib.check(self.h, self.lib.idc_fetch_dist(self.h, img, int(y4), int(x4), _np_ptr(out)))
        return out

    def ab_reccs(self, img, y4, x4, K=5, max_iter=100, n_init=8, pts=None):
        """Colour suggestions at dist[img, :, y4, x4] (reference get_ab_reccs, data/colorize_image.py:322-354)
        computed on the device: (centres [K,2], mass [K], Lloyd iterations)."""
        centers, conf, iters = np.empty((K, 2), np.float32), np.empty((K,), np.float32), ctypes.c_int(0)
        p = None if pts is None else np.ascontiguousarray(pts, np.float32)
        assert p is None or p.shape == (529, 2)
        _lib.check(self.h, self.lib.idc_ab_reccs(self.h, int(img), int(y4), int(x4), int(K), int(max_iter), int(n_init),
                                                 None if p is None else _np_ptr(p), _np_ptr(centers), _np_ptr(conf),
                                                 ctypes.byref(iters)))
        return centers, conf, iters.value

    # ---- Caffe-spec 313-bin head (IDC_FLAG_CAFFE313) ----------------------------------------
    def caffe313_pred_ab(self, n, T=2.6):
        """Annealed-mean ab [n,2,H,W] (device tensor) from the 313-bin logits of the last forward."""
        import torch
        out = torch.empty((n, 2, self.H, self.W), dtype=torch.float32, device="cuda:%d" % self.device)
        st = torch.cuda.current_stream(self.device).cuda_stream
        _lib.check(self.h, self.lib.idc_caffe313_pred_ab(self.h, n, float(T), out.data_ptr(), st))
        return out

    def caffe313_dist_pixel(self, img, y, x, S=0.2):
        """dist_ab_S[:, y, x] (313 floats) at one full-resolution pixel."""
        out = np.empty((313,), np.float32)
        _lib.check(self.h, self.lib.idc_caffe313_dist_pixel(self.h, int(img), int(y), int(x), float(S), _np_ptr(out)))
        return out

    # ---- introspection (tests) -------------------------------------------------------------
    def op_names(self):
        return [self.lib.idc_op_name(self.h, i).decode() for i in range(self.lib.idc_num_ops(self.h))]

    def activation_shape(self, name):
        c, h, w = ctypes.c_int(), ctypes.c_int(), ctypes.c_int()
        _lib.check(self.h, self.lib.idc_get_activation(self.h, name.encode(), None, 0, ctypes.byref(c),
                                                       ctypes.byref(h), ctypes.byref(w)))
        return c.value, h.value, w.value

    def get_activation(self, name, n):
        import torch
        c, h, w = self.activation_shape(name)
        out = torch.empty((n, c, h, w), dtype=torch.float32, device="cuda:%d" % self.device)
        _lib.check(self.h, self.lib.idc_get_activation(self.h, name.encode(), out.data_ptr(), out.numel(), None, None, None))
        return out

    def set_activation(self, name, t):
        assert t.is_cuda and t.is_contiguous()
        _lib.check(self.h, self.lib.idc_set_activation(self.h, name.encode(), t.shape[0], t.data_ptr()))

    def run_op(self, op_name, n):
        import torch
        st = torch.cuda.current_stream(self.device).cuda_stream
        _lib.check(self.h, self.lib.idc_run_op(self.h, op_name.encode(), n, st))

    def set_profiling(self, on):
        _lib.check(self.h, self.lib.idc_set_profiling(self.h, 1 if on else 0))

    def get_profile(self):
        """-> list of (slot name, mean ms per forward, FLOPs per image) since profiling was enabled."""
        names = ["pack+conv1_1"] + self.op_names() + ["heads+post"]
        buf = (ctypes.c_float * len(names))()
        rc = self.lib.idc_get_profile(self.h, buf, len(names))
        if rc < 0:
            _lib.check(self.h, rc)
        flops = [2.0 * self.H * self.W * 64 * 36] + [self.lib.idc_op_flops(self.h, i) for i in range(len(names) - 2)] + [0.0]
        return [(names[i], float(buf[i]), flops[i]) for i in range(len(names))]

    def last_launch_count(self):
        return self.lib.idc_last_launch_count(self.h)

    def flops_per_image(self):
        return self.lib.idc_flops_per_image(self.h)

    def close(self):
        if getattr(self, "h", None):
            self.lib.idc_destroy(self.h)
            self.h = None
            for p in getattr(self, "_pinned", []):
                self.lib.idc_host_free(p)
            self._pinned = []

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
