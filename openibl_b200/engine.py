"""Torch-facing wrapper of the C-ABI engine: tensors in, tensors out, raw device pointers and
the current CUDA stream across the boundary.  PyTorch is used for device memory, streams and
torch.distributed only; every FLOP of the hot path runs in libiblb200.so."""
from __future__ import annotations

import ctypes
from ctypes import byref, c_float, c_int, c_uint64, c_void_p
from typing import Optional, Sequence

import torch

from . import _cabi
from ._cabi import CONV_SIMT_FP32, CONV_TC_BF16X3, OUT_PCA, OUT_POOL, OUT_VLAD, check

_engines = {}


def invalidate_caches() -> None:
    """Forget the re-laid-out VGG16 / PCA parameters cached by every engine of this process.

    The cache key is (data_ptr, Tensor._version).  In-place writes through `.data` (EMA / mean-teacher
    updates, the reference's own `_init_params`, netvlad.py:41-42) do not bump `_version`, so code that
    mutates parameters that way must call this (the model mirror does so from `_init_params`,
    `load_state_dict` and `reset_params`, and re-binds on every forward in training mode)."""
    for eng in _engines.values():
        eng.invalidate()


def _require_cuda(t: torch.Tensor, name: str, dtype=torch.float32) -> torch.Tensor:
    if not isinstance(t, torch.Tensor):
        raise TypeError(f"{name} must be a torch.Tensor")
    if not t.is_cuda:
        raise RuntimeError(
            f"{name} is on '{t.device}': the OpenIBL-B200 hot path runs only on an sm_100 GPU "
            "(there is no CPU fallback); move the tensor/model to CUDA")
    if t.dtype != dtype:
        raise TypeError(f"{name} must be {dtype}, got {t.dtype}")
    return t if t.is_contiguous() else t.contiguous()


def _stream(device) -> c_void_p:
    return c_void_p(torch.cuda.current_stream(device).cuda_stream)


def _ptr(t: Optional[torch.Tensor]) -> c_void_p:
    return c_void_p(0 if t is None else t.data_ptr())


class Engine:
    """One per (process, GPU).  Use Engine.get(device)."""

    def __init__(self, device: int):
        if not torch.cuda.is_available():
            raise RuntimeError("no CUDA device: the OpenIBL-B200 engine has no CPU fallback")
        self.lib = _cabi.load()
        self.device = int(device)
        h = c_void_p()
        check(self.lib.ibl_engine_create(self.device, byref(h)), "ibl_engine_create")
        self.h = h
        self._vgg_key = None
        self._pca_key = None
        self._keep = {}

    @staticmethod
    def get(device=None) -> "Engine":
        if isinstance(device, torch.device) and device.type != "cuda":
            raise RuntimeError(
                f"tensor/model is on '{device}': the OpenIBL-B200 hot path runs only on an sm_100 GPU "
                "(there is no CPU fallback); move it to CUDA")
        if not torch.cuda.is_available():
            raise RuntimeError("no CUDA device: the OpenIBL-B200 engine has no CPU fallback")
        if device is None:
            device = torch.cuda.current_device()
        if isinstance(device, torch.device):
            device = device.index if device.index is not None else torch.cuda.current_device()
        device = int(device)
        if device not in _engines:
            _engines[device] = Engine(device)
        return _engines[device]

    def __del__(self):
        try:
            if getattr(self, "h", None):
                self.lib.ibl_engine_destroy(self.h)
                self.h = None
        except Exception:
            pass

    # ---- configuration -------------------------------------------------------------------
    @property
    def conv_mode(self) -> int:
        m = c_int()
        check(self.lib.ibl_engine_get_conv_mode(self.h, byref(m)), "ibl_engine_get_conv_mode")
        return m.value

    @conv_mode.setter
    def conv_mode(self, mode: int) -> None:
        check(self.lib.ibl_engine_set_conv_mode(self.h, int(mode)), "ibl_engine_set_conv_mode")

    def set_gemm_mode(self, mode: int) -> None:
        check(self.lib.ibl_engine_set_gemm_mode(self.h, int(mode)), "ibl_engine_set_gemm_mode")

    @property
    def launch_count(self) -> int:
        c = c_uint64()
        check(self.lib.ibl_engine_launch_count(self.h, byref(c)), "ibl_engine_launch_count")
        return c.value

    # ---- parameters ----------------------------------------------------------------------
    def invalidate(self) -> None:
        """Drop the (address, version) keys: the next set_vgg16 / set_pca re-lays the parameters out."""
        self._vgg_key = None
        self._pca_key = None

    def set_vgg16(self, weights: Sequence[torch.Tensor], biases: Sequence[torch.Tensor], force: bool = False) -> None:
        assert len(weights) == 13 and len(biases) == 13
        key = tuple((w.data_ptr(), w._version, b.data_ptr(), b._version) for w, b in zip(weights, biases))
        if key == self._vgg_key and not force:
            return
        self._vgg_key = None
        ws = [_require_cuda(w.detach(), "vgg weight") for w in weights]
        bs = [_require_cuda(b.detach(), "vgg bias") for b in biases]
        wa = (c_void_p * 13)(*[w.data_ptr() for w in ws])
        ba = (c_void_p * 13)(*[b.data_ptr() for b in bs])
        check(self.lib.ibl_engine_set_vgg16(self.h, wa, ba, _stream(self.device)), "ibl_engine_set_vgg16")
        self._vgg_key = key
        # keep the tensors alive: the key is (address, version), so the addresses must not be recycled
        self._keep["vgg"] = (list(weights), list(biases), ws, bs)

    def set_netvlad(self, conv_w: torch.Tensor, centroids: torch.Tensor) -> None:
        K, C = centroids.shape
        w = _require_cuda(conv_w.detach().reshape(K, C), "net_vlad.conv.weight")
        c = _require_cuda(centroids.detach(), "net_vlad.centroids")
        self._keep["nv"] = (w, c)
        check(self.lib.ibl_engine_set_netvlad(self.h, _ptr(w), _ptr(c), K, C, _stream(self.device)),
              "ibl_engine_set_netvlad")

    def set_pca(self, weight: torch.Tensor, bias: torch.Tensor, force: bool = False) -> None:
        key = (weight.data_ptr(), weight._version, bias.data_ptr(), bias._version)
        if key == self._pca_key and not force:
            return
        self._pca_key = None                      # stays unset if validation or the C call fails
        P = weight.shape[0]
        w = _require_cuda(weight.detach().reshape(P, -1), "pca weight")
        b = _require_cuda(bias.detach().reshape(-1), "pca bias")
        check(self.lib.ibl_engine_set_pca(self.h, _ptr(w), _ptr(b), P, w.shape[1], _stream(self.device)),
              "ibl_engine_set_pca")
        self._keep["pca"] = (weight, bias, w, b)   # the originals too: their addresses are in the key
        self._pca_key = key

    # ---- stages --------------------------------------------------------------------------
    def vgg16_forward(self, x: torch.Tensor, want_nchw=True, want_pool=True, want_nhwc=False):
        x = _require_cuda(x, "input images")
        N, C, H, W = x.shape
        if C != 3:
            raise ValueError("VGG16 trunk expects [N,3,H,W]")
        fh, fw = H // 16, W // 16
        nhwc = torch.empty(N, fh, fw, 512, device=x.device) if want_nhwc else None
        nchw = torch.empty(N, 512, fh, fw, device=x.device) if want_nchw else None
        pool = torch.empty(N, 512, device=x.device) if want_pool else None
        check(self.lib.ibl_vgg16_forward(self.h, _ptr(x), N, H, W, _ptr(nhwc), _ptr(nchw), _ptr(pool),
                                         _stream(self.device)), "ibl_vgg16_forward")
        return nhwc, nchw, pool

    def netvlad_forward(self, feat: torch.Tensor, conv_w: torch.Tensor, centroids: torch.Tensor,
                        nhwc=False, normalize_input=True, want_raw=True, want_norm=False):
        feat = _require_cuda(feat, "feature map")
        K, C = centroids.shape
        if nhwc:
            N, S = feat.shape[0], feat[0].numel() // C
        else:
            N, S = feat.shape[0], feat[0].numel() // C
            if feat.shape[1] != C:
                raise ValueError(f"feature map has {feat.shape[1]} channels, NetVLAD dim is {C}")
        w = _require_cuda(conv_w.detach().reshape(K, C), "net_vlad.conv.weight")
        c = _require_cuda(centroids.detach(), "net_vlad.centroids")
        raw = torch.empty(N, K, C, device=feat.device) if want_raw else None
        nrm = torch.empty(N, K * C, device=feat.device) if want_norm else None
        check(self.lib.ibl_netvlad_forward(self.h, _ptr(feat), 1 if nhwc else 0, N, C, S, _ptr(w), _ptr(c), K,
                                           1 if normalize_input else 0, _ptr(raw), _ptr(nrm),
                                           _stream(self.device)), "ibl_netvlad_forward")
        return raw, nrm

    def netvlad_backward(self, feat: torch.Tensor, conv_w: torch.Tensor, centroids: torch.Tensor,
                         grad_vlad: torch.Tensor, nhwc=False, normalize_input=True):
        """-> (grad_feat like feat, grad_conv_w [K,C], grad_centroids [K,C])"""
        feat = _require_cuda(feat, "feature map")
        g = _require_cuda(grad_vlad, "grad_vlad")
        K, C = centroids.shape
        N, S = feat.shape[0], feat[0].numel() // C
        w = _require_cuda(conv_w.detach().reshape(K, C), "net_vlad.conv.weight")
        c = _require_cuda(centroids.detach(), "net_vlad.centroids")
        dx = torch.empty_like(feat)
        dw = torch.empty(K, C, device=feat.device)
        dc = torch.empty(K, C, device=feat.device)
        check(self.lib.ibl_netvlad_backward(self.h, _ptr(feat), 1 if nhwc else 0, N, C, S, _ptr(w), _ptr(c), K,
                                            1 if normalize_input else 0, _ptr(g), _ptr(dx), _ptr(dw), _ptr(dc),
                                            _stream(self.device)), "ibl_netvlad_backward")
        return dx, dw, dc

    def vlad_normalize(self, raw: torch.Tensor) -> torch.Tensor:
        raw = _require_cuda(raw, "vlad")
        N, K, C = raw.shape
        out = torch.empty(N, K * C, device=raw.device)
        check(self.lib.ibl_vlad_normalize(self.h, _ptr(raw), N, K, C, _ptr(out), _stream(self.device)),
              "ibl_vlad_normalize")
        return out

    def pca_l2(self, v: torch.Tensor, weight: torch.Tensor, bias: torch.Tensor) -> torch.Tensor:
        v = _require_cuda(v, "descriptors")
        P = weight.shape[0]
        w = _require_cuda(weight.detach().reshape(P, -1), "pca weight")
        b = _require_cuda(bias.detach().reshape(-1), "pca bias")
        N, D = v.shape
        if w.shape[1] != D:
            raise ValueError(f"PCA expects dim {w.shape[1]}, got {D}")
        out = torch.empty(N, P, device=v.device)
        check(self.lib.ibl_pca_l2(self.h, _ptr(v), N, D, _ptr(w), _ptr(b), P, _ptr(out), _stream(self.device)),
              "ibl_pca_l2")
        return out

    def l2_normalize_rows(self, x: torch.Tensor) -> torch.Tensor:
        x = _require_cuda(x, "rows")
        N, D = x.shape
        out = torch.empty_like(x)
        check(self.lib.ibl_l2_normalize_rows(self.h, _ptr(x), N, D, _ptr(out), _stream(self.device)),
              "ibl_l2_normalize_rows")
        return out

    def extract(self, x: torch.Tensor, pca=False, want_pool=False):
        """Whole path with the parameters previously set on the engine."""
        x = _require_cuda(x, "input images")
        N, _, H, W = x.shape
        flags = OUT_VLAD | (OUT_PCA if pca else 0) | (OUT_POOL if want_pool else 0)
        dim = self._keep["pca"][0].shape[0] if pca else self._keep["nv"][0].numel()
        out = torch.empty(N, dim, device=x.device)
        pool = torch.empty(N, 512, device=x.device) if want_pool else None
        check(self.lib.ibl_extract(self.h, _ptr(x), N, H, W, flags, _ptr(out), _ptr(pool), _stream(self.device)),
              "ibl_extract")
        return out, pool

    def extract_host(self, x_host: torch.Tensor, out_host: torch.Tensor, pca=False,
                     pool_host: Optional[torch.Tensor] = None) -> torch.Tensor:
        """HOST in / HOST out (pinned recommended): H2D + path + D2H + sync inside the call."""
        assert not x_host.is_cuda and not out_host.is_cuda and x_host.is_contiguous() and out_host.is_contiguous()
        assert x_host.dtype == torch.float32 and out_host.dtype == torch.float32
        N, _, H, W = x_host.shape
        flags = OUT_VLAD | (OUT_PCA if pca else 0) | (OUT_POOL if pool_host is not None else 0)
        check(self.lib.ibl_extract_host(self.h, _ptr(x_host), N, H, W, flags, _ptr(out_host), _ptr(pool_host),
                                        _stream(self.device)), "ibl_extract_host")
        return out_host

    def extract_host_submit(self, slot: int, x_host: torch.Tensor, out_host: torch.Tensor, pca=False,
                            pool_host: Optional[torch.Tensor] = None) -> None:
        """Pipelined form of extract_host: enqueue H2D (copy stream), extraction and D2H for `slot` (0 or 1) and return
        without synchronising; `extract_host_wait(slot)` blocks until out_host holds the descriptors.  With two slots
        the copy of batch i+1 overlaps the compute of batch i.  Host tensors should be pinned and must stay alive."""
        assert not x_host.is_cuda and not out_host.is_cuda and x_host.is_contiguous() and out_host.is_contiguous()
        assert x_host.dtype == torch.float32 and out_host.dtype == torch.float32
        N, _, H, W = x_host.shape
        flags = OUT_VLAD | (OUT_PCA if pca else 0) | (OUT_POOL if pool_host is not None else 0)
        self._keep[("pipe", slot)] = (x_host, out_host, pool_host)
        check(self.lib.ibl_extract_host_submit(self.h, int(slot), _ptr(x_host), N, H, W, flags, _ptr(out_host),
                                               _ptr(pool_host), _stream(self.device)), "ibl_extract_host_submit")

    def extract_host_wait(self, slot: int) -> None:
        check(self.lib.ibl_extract_host_wait(self.h, int(slot)), "ibl_extract_host_wait")
        self._keep.pop(("pipe", slot), None)

    def extract_host_stream(self, batches, pca=False):
        """Iterate (x_host, out_host) pairs through the two-slot pipeline; yields each out_host once it is complete."""
        pending = []
        for i, (x_host, out_host) in enumerate(batches):
            slot = i & 1
            if len(pending) == 2:
                s0, o0 = pending.pop(0)
                self.extract_host_wait(s0)
                yield o0
            self.extract_host_submit(slot, x_host, out_host, pca=pca)
            pending.append((slot, out_host))
        for s0, o0 in pending:
            self.extract_host_wait(s0)
            yield o0

    # ---- input side: ToTensor + Normalize on the device (utils/data/__init__.py:37-42) ------
    @staticmethod
    def _norm_consts(mean, std):
        import ctypes
        m = (ctypes.c_float * 3)(*[float(v) for v in mean])
        s = (ctypes.c_float * 3)(*[float(v) for v in std])
        return m, s

    def preprocess_u8(self, x_u8_nhwc: torch.Tensor, mean, std) -> torch.Tensor:
        """uint8 [N,H,W,3] on the GPU -> fp32 [N,3,H,W] = ((x/255) - mean) / std, bit-identical to torchvision."""
        x = _require_cuda(x_u8_nhwc, "images", dtype=torch.uint8)
        N, H, W, C = x.shape
        assert C == 3
        out = torch.empty(N, 3, H, W, device=x.device)
        m, s = self._norm_consts(mean, std)
        check(self.lib.ibl_preprocess_u8(self.h, _ptr(x), N, H, W, m, s, _ptr(out), _stream(self.device)),
              "ibl_preprocess_u8")
        return out

    def resize_u8(self, x_u8_nhwc: torch.Tensor, out_h: int, out_w: int) -> torch.Tensor:
        """uint8 [N,H,W,3] on the GPU -> uint8 [N,out_h,out_w,3], bit-identical to PIL.Image.resize(..., BILINEAR)."""
        from .utils.data.gpu_resize import pil_bilinear_coeffs
        x = _require_cuda(x_u8_nhwc, "images", dtype=torch.uint8)
        N, H, W, C = x.shape
        assert C == 3
        tabs = self._keep.setdefault("resize_tabs", {})

        def table(n_in, n_out):
            if n_in == n_out:
                return None, None, 0
            key = (n_in, n_out)
            if key not in tabs:
                b, k, ks = pil_bilinear_coeffs(n_in, n_out)
                tabs[key] = (torch.from_numpy(b).to(x.device), torch.from_numpy(k).to(x.device), ks)
            return tabs[key]

        bh, kh, ksh = table(W, out_w)
        bv, kv, ksv = table(H, out_h)
        out = torch.empty(N, out_h, out_w, 3, dtype=torch.uint8, device=x.device)
        check(self.lib.ibl_resize_bilinear_u8(self.h, _ptr(x), N, H, W, int(out_h), int(out_w), _ptr(bh), _ptr(kh), ksh,
                                              _ptr(bv), _ptr(kv), ksv, _ptr(out), _stream(self.device)),
              "ibl_resize_bilinear_u8")
        return out

    def argsort_rows(self, dist: torch.Tensor) -> torch.Tensor:
        """torch.argsort(dist, dim=1) on the engine's own sort kernels: [m,n] fp32 -> [m,n] int64, ties by index."""
        dist = _require_cuda(dist, "distance matrix")
        m, n = dist.shape
        out = torch.empty(m, n, dtype=torch.int64, device=dist.device)
        check(self.lib.ibl_argsort_rows(self.h, _ptr(dist), m, n, _ptr(out), _stream(self.device)), "ibl_argsort_rows")
        return out

    def extract_host_u8(self, x_u8_host: torch.Tensor, out_host: torch.Tensor, mean, std, pca=False,
                        pool_host: Optional[torch.Tensor] = None) -> torch.Tensor:
        """HOST uint8 [N,H,W,3] in / HOST descriptors out: a quarter of extract_host's H2D bytes."""
        assert not x_u8_host.is_cuda and not out_host.is_cuda and x_u8_host.is_contiguous() and out_host.is_contiguous()
        assert x_u8_host.dtype == torch.uint8 and out_host.dtype == torch.float32
        N, H, W, C = x_u8_host.shape
        assert C == 3
        flags = OUT_VLAD | (OUT_PCA if pca else 0) | (OUT_POOL if pool_host is not None else 0)
        m, s = self._norm_consts(mean, std)
        check(self.lib.ibl_extract_host_u8(self.h, _ptr(x_u8_host), N, H, W, m, s, flags, _ptr(out_host),
                                           _ptr(pool_host), _stream(self.device)), "ibl_extract_host_u8")
        return out_host

    # ---- retrieval -----------------------------------------------------------------------
    def l2dist_dense(self, q: torch.Tensor, db: torch.Tensor) -> torch.Tensor:
        q = _require_cuda(q, "queries")
        db = _require_cuda(db, "database")
        m, d = q.shape
        n = db.shape[0]
        out = torch.empty(m, n, device=q.device)
        check(self.lib.ibl_l2dist_dense(self.h, _ptr(q), m, _ptr(db), n, d, _ptr(out), _stream(self.device)),
              "ibl_l2dist_dense")
        return out

    def l2dist_self(self, x: torch.Tensor) -> torch.Tensor:
        x = _require_cuda(x, "features")
        n, d = x.shape
        out = torch.empty(n, n, device=x.device)
        check(self.lib.ibl_l2dist_self(self.h, _ptr(x), n, d, _ptr(out), _stream(self.device)), "ibl_l2dist_self")
        return out

    def l2dist_topk(self, q: torch.Tensor, db: torch.Tensor, k: int, idx_base: int = 0,
                    n_valid: Optional[int] = None):
        q = _require_cuda(q, "queries")
        db = _require_cuda(db, "database")
        m, d = q.shape
        n = db.shape[0]
        if n_valid is None:
            n_valid = n
        od = torch.empty(m, k, device=q.device)
        oi = torch.empty(m, k, device=q.device, dtype=torch.int64)
        check(self.lib.ibl_l2dist_topk(self.h, _ptr(q), m, _ptr(db), n, int(n_valid), d, int(k), int(idx_base),
                                       _ptr(od), _ptr(oi), _stream(self.device)), "ibl_l2dist_topk")
        return od, oi

    def topk_rows(self, dist: torch.Tensor, k: int):
        dist = _require_cuda(dist, "distance matrix")
        m, n = dist.shape
        od = torch.empty(m, k, device=dist.device)
        oi = torch.empty(m, k, device=dist.device, dtype=torch.int64)
        check(self.lib.ibl_topk_rows(self.h, _ptr(dist), m, n, int(k), _ptr(od), _ptr(oi), _stream(self.device)),
              "ibl_topk_rows")
        return od, oi

    def topk_merge(self, cand_dist: torch.Tensor, cand_idx: torch.Tensor, k_out: int):
        cand_dist = _require_cuda(cand_dist, "candidate distances")
        cand_idx = _require_cuda(cand_idx, "candidate indices", torch.int64)
        parts, m, k_in = cand_dist.shape
        od = torch.empty(m, k_out, device=cand_dist.device)
        oi = torch.empty(m, k_out, device=cand_dist.device, dtype=torch.int64)
        check(self.lib.ibl_topk_merge(self.h, _ptr(cand_dist), _ptr(cand_idx), parts, m, k_in, int(k_out),
                                      _ptr(od), _ptr(oi), _stream(self.device)), "ibl_topk_merge")
        return od, oi

    def l2dist_topk_host(self, q_host: torch.Tensor, db_host: torch.Tensor, k: int,
                         out_dist_host: torch.Tensor, out_idx_host: torch.Tensor):
        m, d = q_host.shape
        n = db_host.shape[0]
        check(self.lib.ibl_l2dist_topk_host(self.h, _ptr(q_host), m, _ptr(db_host), n, d, int(k),
                                            _ptr(out_dist_host), _ptr(out_idx_host), _stream(self.device)),
              "ibl_l2dist_topk_host")
        return out_dist_host, out_idx_host

    def dist_flagged(self) -> int:
        """Queries re-ranked by exact brute force in the last l2dist_topk call (-1: CUDA-core path)."""
        c = c_int()
        check(self.lib.ibl_debug_dist_flagged(self.h, byref(c), _stream(self.device)), "ibl_debug_dist_flagged")
        return c.value

    def gemm_nt(self, a: torch.Tensor, b: torch.Tensor, alpha: float = 1.0, mode: int = CONV_SIMT_FP32) -> torch.Tensor:
        """alpha * a @ b.T on the engine's own GEMM kernels (PCA.train's products, pca.py:38-67)."""
        a = _require_cuda(a, "A")
        b = _require_cuda(b, "B")
        m, k = a.shape
        n = b.shape[0]
        if b.shape[1] != k:
            raise ValueError("gemm_nt: inner dimensions differ")
        pad = (-k) % 64
        if pad:                                   # zero columns do not change the products
            a = torch.nn.functional.pad(a, (0, pad))
            b = torch.nn.functional.pad(b, (0, pad))
        out = torch.empty(m, n, device=a.device)
        rows = max(1, min(m, (2 ** 31 - 1) // max(n, 1)))
        for r0 in range(0, m, rows):
            r1 = min(m, r0 + rows)
            check(self.lib.ibl_gemm_nt(self.h, _ptr(a[r0:r1]), r1 - r0, _ptr(b), n, k + pad, c_float(alpha), _ptr(out[r0:r1]),
                                       int(mode), _stream(self.device)), "ibl_gemm_nt")
        return out

    # ---- training surface of the trunk (SURVEY 8 f1) ------------------------------------------
    def vgg16_prefix_forward(self, x: torch.Tensor, n_layers: int) -> torch.Tensor:
        """Frozen layers [0, n_layers) -> fp32 NHWC activation entering layer n_layers."""
        from .synth import VGG16_PLAN
        x = _require_cuda(x, "input images")
        N, _, H, W = x.shape
        h, w, c, seen = H, W, 3, 0
        for item in VGG16_PLAN:
            if item == "P":
                h, w = h // 2, w // 2
            else:
                if seen == n_layers:
                    break
                c = item[2]
                seen += 1
        out = torch.empty(N, h, w, c, device=x.device)
        check(self.lib.ibl_vgg16_prefix_forward(self.h, _ptr(x), N, H, W, int(n_layers), _ptr(out), _stream(self.device)),
              "ibl_vgg16_prefix_forward")
        return out

    def vgg16_layer_forward(self, layer: int, x: torch.Tensor, cout: int) -> torch.Tensor:
        x = _require_cuda(x, "layer input")
        if layer == 0:
            N, _, H, W = x.shape
        else:
            N, H, W, _ = x.shape
        y = torch.empty(N, H, W, cout, device=x.device)
        check(self.lib.ibl_vgg16_layer_forward(self.h, int(layer), _ptr(x), N, H, W, _ptr(y), _stream(self.device)),
              "ibl_vgg16_layer_forward")
        return y

    def vgg16_layer_backward(self, layer: int, x: torch.Tensor, y: Optional[torch.Tensor], gy: torch.Tensor,
                             w_shape, need_gx: bool):
        x = _require_cuda(x, "layer input")
        gy = _require_cuda(gy, "grad output")
        N, H, W, cout = gy.shape
        gx = torch.empty_like(x) if need_gx else None
        gw = torch.empty(w_shape, device=x.device)
        gb = torch.empty(cout, device=x.device)
        check(self.lib.ibl_vgg16_layer_backward(self.h, int(layer), _ptr(x), _ptr(y), _ptr(gy), N, H, W, _ptr(gx), _ptr(gw),
                                                _ptr(gb), _stream(self.device)), "ibl_vgg16_layer_backward")
        return gx, gw, gb

    def maxpool2x2(self, x: torch.Tensor) -> torch.Tensor:
        x = _require_cuda(x, "pool input")
        N, H, W, C = x.shape
        y = torch.empty(N, H // 2, W // 2, C, device=x.device)
        check(self.lib.ibl_maxpool2x2_forward(self.h, _ptr(x), N, H, W, C, _ptr(y), _stream(self.device)), "ibl_maxpool2x2_forward")
        return y

    def maxpool2x2_backward(self, x: torch.Tensor, gy: torch.Tensor) -> torch.Tensor:
        x = _require_cuda(x, "pool input")
        gy = _require_cuda(gy, "pool grad")
        N, H, W, C = x.shape
        gx = torch.empty_like(x)
        check(self.lib.ibl_maxpool2x2_backward(self.h, _ptr(x), _ptr(gy), N, H, W, C, _ptr(gx), _stream(self.device)),
              "ibl_maxpool2x2_backward")
        return gx

    # ---- test hooks ----------------------------------------------------------------------
    def debug_conv3x3(self, x_nhwc, w_oihw, bias, relu=True, pool=False, mode=CONV_TC_BF16X3, bn=0):
        x = _require_cuda(x_nhwc, "x")
        w = _require_cuda(w_oihw, "w")
        b = _require_cuda(bias, "bias")
        N, H, W, cin = x.shape
        cout = w.shape[0]
        oh, ow = (H // 2, W // 2) if pool else (H, W)
        y = torch.empty(N, oh, ow, cout, device=x.device)
        check(self.lib.ibl_debug_conv3x3(self.h, _ptr(x), N, H, W, cin, _ptr(w), _ptr(b), cout, int(relu),
                                         int(pool), int(mode), int(bn), _ptr(y), _stream(self.device)),
              "ibl_debug_conv3x3")
        return y
