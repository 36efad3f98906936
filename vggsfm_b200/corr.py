"""CorrBlock / EfficientCorrBlock with the reference's interface (vggsfm/models/track_modules/blocks.py:338-471),
backed by the fused correlation+sampling kernel (csrc/corr.cu).  The correlation volume is never built.

Drop-in: `vggsfm.models.track_modules.base_track_predictor.CorrBlock = vggsfm_b200.corr.CorrBlock`
(the class is looked up at base_track_predictor.py:117-124)."""
from __future__ import annotations

import ctypes

import torch

from . import _lib


def _stream(dev):
    return torch.cuda.current_stream(dev).cuda_stream


class _Pyramid:
    def __init__(self, fmaps, num_levels, radius, half=None, tc=None):
        if not fmaps.is_cuda:
            raise RuntimeError("vggsfm_b200.CorrBlock needs CUDA tensors (no CPU fallback)")
        B, S, C, H, W = fmaps.shape
        self.B, self.S, self.C, self.H, self.W = B, S, C, H, W
        self.num_levels, self.radius = num_levels, radius
        # half pyramid when the reference would have run its matmul under fp16 autocast (runner.py:418)
        if half is None:
            half = fmaps.dtype in (torch.float16, torch.bfloat16) or torch.is_autocast_enabled()
        self.elem = 2 if half else 4
        L = _lib.lib()
        dev = fmaps.device
        pb, sb = ctypes.c_size_t(), ctypes.c_size_t()
        _lib.check(L.vgg_corr_pyramid_bytes(B * S, C, H, W, num_levels, self.elem, ctypes.byref(pb), ctypes.byref(sb)),
                   "vgg_corr_pyramid_bytes")
        self.pyr = torch.empty(pb.value, dtype=torch.uint8, device=dev)
        scratch = torch.empty(max(sb.value, 1), dtype=torch.uint8, device=dev)
        src = fmaps.reshape(B * S, C, H, W).float().contiguous()
        with torch.cuda.device(dev):
            _lib.check(L.vgg_corr_build_pyramid(B * S, C, H, W, num_levels, src.data_ptr(), self.elem, self.pyr.data_ptr(),
                                                scratch.data_ptr() if sb.value else None, _stream(dev)),
                       "vgg_corr_build_pyramid")
        self.dev = dev
        # coarse tracker (C = 128, power-of-two maps, half pyramid): operand tile images for the tcgen05 kernel
        # (csrc/corr_tc.cu); tc=False keeps the CUDA-core footprint kernel
        self.tc_tiles = None
        want_tc = True if tc is None else bool(tc)
        if self.elem == 2 and want_tc and L.vgg_corr_tc_supported(C, H, W, num_levels, radius):
            tb = ctypes.c_size_t()
            _lib.check(L.vgg_corr_tc_bytes(B * S, C, H, W, num_levels, 0, ctypes.byref(tb), None), "vgg_corr_tc_bytes")
            self.tc_tiles = torch.empty(tb.value, dtype=torch.uint8, device=dev)
            with torch.cuda.device(dev):
                _lib.check(L.vgg_corr_tc_build(B * S, C, H, W, num_levels, self.pyr.data_ptr(), self.tc_tiles.data_ptr(),
                                               _stream(dev)), "vgg_corr_tc_build")
        self._tc_scratch = None

    def sample(self, coords, targets, border):
        B, S, N, D = coords.shape
        assert D == 2
        assert targets.shape == (B, S, N, self.C)
        assert S == self.S
        r = self.radius
        K = 2 * r + 1
        out = torch.empty(B, S, N, self.num_levels * K * K, dtype=torch.float32, device=self.dev)
        tg = targets.float().contiguous()
        co = coords.float().contiguous()
        if self.tc_tiles is not None and not border:
            L = _lib.lib()
            ab = ctypes.c_size_t()
            _lib.check(L.vgg_corr_tc_bytes(B * S, self.C, self.H, self.W, self.num_levels, N, None, ctypes.byref(ab)),
                       "vgg_corr_tc_bytes")
            if self._tc_scratch is None or self._tc_scratch.numel() < ab.value:
                self._tc_scratch = torch.empty(ab.value, dtype=torch.uint8, device=self.dev)
            with torch.cuda.device(self.dev):
                _lib.check(L.vgg_corr_tc_sample(B * S, N, self.C, self.H, self.W, self.num_levels, r, self.tc_tiles.data_ptr(),
                                                tg.data_ptr(), co.data_ptr(), self._tc_scratch.data_ptr(), out.data_ptr(),
                                                _stream(self.dev)), "vgg_corr_tc_sample")
            return out
        with torch.cuda.device(self.dev):
            _lib.check(_lib.lib().vgg_corr_sample(B * S, N, self.C, self.H, self.W, self.num_levels, r, self.pyr.data_ptr(),
                                                  self.elem, tg.data_ptr(), co.data_ptr(), 1 if border else 0,
                                                  out.data_ptr(), _stream(self.dev)), "vgg_corr_sample")
        return out


class CorrBlock:
    """blocks.py:338-416.  corr(targets) records the targets; sample(coords) runs the fused kernel."""

    def __init__(self, fmaps, num_levels=4, radius=4, multiple_track_feats=False, padding_mode="zeros", half=None, tc=None):
        if multiple_track_feats:
            raise NotImplementedError("multiple_track_feats=True is not used by the reference configs")
        if padding_mode not in ("zeros", "border"):
            raise ValueError(f"unsupported padding_mode {padding_mode}")
        self.padding_mode = padding_mode
        self.num_levels, self.radius = num_levels, radius
        B, S, C, H, W = fmaps.shape
        self.S, self.C, self.H, self.W = S, C, H, W
        self._pyr = _Pyramid(fmaps, num_levels, radius, half, tc if padding_mode == "zeros" else False)
        self._targets = None

    def corr(self, targets):
        B, S, N, C = targets.shape
        assert C == self.C
        assert S == self.S
        self._targets = targets

    def sample(self, coords):
        if self._targets is None:
            raise RuntimeError("CorrBlock.sample called before CorrBlock.corr")
        return self._pyr.sample(coords, self._targets, self.padding_mode == "border")


class EfficientCorrBlock:
    """blocks.py:419-471: sample(coords, target) with border padding."""

    def __init__(self, fmaps, num_levels=4, radius=4, half=None):
        self.num_levels, self.radius = num_levels, radius
        self._pyr = _Pyramid(fmaps, num_levels, radius, half)

    def sample(self, coords, target):
        return self._pyr.sample(coords, target, True)


def sample_features4d(input, coords):
    """vggsfm/models/utils.py:415-447: input [B,C,H,W], coords [B,R,2] (x,y) -> [B,R,C]; bilinear,
    align_corners=True, border padding (``vgg_sample_features4d``)."""
    if not input.is_cuda:
        raise RuntimeError("vggsfm_b200.sample_features4d needs CUDA tensors (no CPU fallback)")
    B, C, H, W = input.shape
    R = coords.shape[1]
    inp = input.float().contiguous()
    crd = coords.float().contiguous()
    out = torch.empty(B, R, C, dtype=torch.float32, device=input.device)
    with torch.cuda.device(input.device):
        _lib.check(_lib.lib().vgg_sample_features4d(B, C, H, W, R, inp.data_ptr(), crd.data_ptr(), out.data_ptr(),
                                                    _stream(input.device)), "vgg_sample_features4d")
    return out.to(input.dtype)
