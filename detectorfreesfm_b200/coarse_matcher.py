"""HP-1 host side: a drop-in for the reference's ``LoFTR`` module behind the NEUSFM_coarse_matcher hook.

Mirrors third_party/LoFTR/src/loftr/loftr.py:11-81: ``B200LoFTR(config)`` is called as ``matcher(data)`` under
``torch.no_grad()`` from src/coarse_match/coarse_match_worker.py:94-100, mutates ``data`` in place and adds the same
keys (``m_bids, mkpts0_f, mkpts1_f, mconf`` are the ones the worker reads, :85-89).  All compute runs in
libdfsfm_b200.so (hand-written sm_100a CUDA); this file only moves pointers and keeps the per-image feature cache
(the backbone is exact per image because BatchNorm is in eval mode, so features are reusable across pairs).
"""
import ctypes
from collections import OrderedDict

import torch

from . import _lib
from .packing import pack_loftr, position_encoding


class B200LoFTR(torch.nn.Module):
    def __init__(self, config, device=None, feature_cache_size=64, feature_cache_bytes=8 << 30):
        super().__init__()
        self.config = config
        mc = config["match_coarse"]
        if mc["match_type"] != "dual_softmax":
            raise NotImplementedError("only match_type='dual_softmax' is built (the shipped loftr_ds configs)")
        self.fine = bool(config["fine"]["enable"])
        if self.fine:
            fcfg = config["fine"]
            if (fcfg["d_model"] != 128 or fcfg["nhead"] != 8 or list(fcfg["layer_names"]) != ["self", "cross"] or config["fine_window_size"] != 5
                    or not config["fine_concat_coarse_feat"] or tuple(config["resolution"]) != (8, 2)):
                raise NotImplementedError("fine stage is specialised for the outdoor_ds LoFTR (window 5, d_model 128, ['self','cross'])")
        c = config["coarse"]
        if c["d_model"] != 256 or c["nhead"] != 8 or list(c["layer_names"]) != ["self", "cross"] * 4 or c["attention"] != "linear":
            raise NotImplementedError("engine is specialised for the outdoor_ds LoFTR (d_model 256, 8 heads, 8 layers, linear)")
        if c.get("temp_bug_fix", False):
            raise NotImplementedError("temp_bug_fix=True position encoding is not used by DetectorFreeSfM (coarse_match_worker.py:35)")
        self.thr = float(mc["thr"])
        self.border_rm = int(mc["border_rm"])
        self.temperature = float(mc["dsmax_temperature"])
        self._lib = _lib.load_library()
        self._h = ctypes.c_void_p()
        self._device = None
        self._pe = {}
        # per-image feature cache (exact: BatchNorm is in eval mode).  Key contract: (pair_key name, H, W) -- the caller guarantees that a
        # name keeps its pixels for the life of the cache (one scene); call clear_cache() between scenes that reuse relative paths.
        # Bounded by entries AND bytes (with the fine stage an entry holds the 1/2-resolution 128-channel map: 140-270 MB at 1200-1600 px).
        self._cache = OrderedDict()
        self._cache_size = feature_cache_size
        self._cache_bytes_max = int(feature_cache_bytes)
        self._cache_bytes = 0
        self._packed = None
        if device is not None:
            self.cuda(device)

    # ---------------------------------------------------------------- nn.Module-compatible plumbing
    def cuda(self, device=None):
        if device is None:
            idx = torch.cuda.current_device()
        elif isinstance(device, int):
            idx = device
        else:
            idx = torch.device(device).index
            idx = torch.cuda.current_device() if idx is None else idx
        dev = torch.device("cuda", idx)
        if self._device != dev:
            self._destroy()
            self._device = dev
            _lib.check(self._lib.dfsfm_coarse_create(ctypes.byref(self._h), dev.index))
            if self._packed is not None:
                self._upload()
        return self

    def load_state_dict(self, state_dict, strict=True):
        """Accepts the reference checkpoint layout (``matcher.`` prefix stripped like loftr.py:83-87)."""
        self._packed = pack_loftr(state_dict, fine=self.fine)
        if self._h:
            self._upload()
        self.clear_cache()
        return self

    def _upload(self):
        for name, (t, kind) in self._packed.items():
            _lib.check(self._lib.dfsfm_coarse_set_param(self._h, name.encode(), ctypes.c_void_p(t.data_ptr()), t.shape[0], t.shape[1], kind))

    def _destroy(self):
        if self._h:
            self._lib.dfsfm_coarse_destroy(self._h)
            self._h = ctypes.c_void_p()
        self._pe.clear()
        self._cache.clear()
        self._cache_bytes = 0

    def __del__(self):
        try:
            self._destroy()
        except Exception:
            pass

    # ------------------------------------------------------------------------------ stages
    def _pe_tokens(self, h, w):
        key = (h, w)
        if key not in self._pe:
            self._pe[key] = position_encoding(h, w).to(self._device)
        return self._pe[key]

    @staticmethod
    def _cache_key(image, cache_key):
        assert image.is_cuda and image.dtype == torch.float32 and image.dim() == 4 and image.shape[0] == 1 and image.shape[1] == 1
        return None if cache_key is None else (cache_key, image.shape[2], image.shape[3])

    def extract_features(self, image, cache_key=None):
        """ResNetFPN_8_2 coarse branch + position encoding -> tokens [(H/8)*(W/8), 256] fp32 (loftr.py:45-59)."""
        key = self._cache_key(image, cache_key)
        if key is not None and key in self._cache:
            self._cache.move_to_end(key)
            return self._cache[key]
        H, W = image.shape[2:]
        image = image.contiguous()
        h, w = H // 8, W // 8
        tokens = torch.empty(h * w, 256, device=self._device, dtype=torch.float32)
        if self.fine:
            feat_f = torch.empty((H // 2) * (W // 2), 128, device=self._device, dtype=torch.float32)
            _lib.check(self._lib.dfsfm_coarse_features_fine(self._h, _lib.ptr(image), H, W, _lib.ptr(self._pe_tokens(h, w)), _lib.ptr(tokens),
                                                            _lib.ptr(feat_f), _lib.stream_ptr(self._device)))
            out = (tokens, feat_f)
        else:
            _lib.check(self._lib.dfsfm_coarse_features(self._h, _lib.ptr(image), H, W, _lib.ptr(self._pe_tokens(h, w)), _lib.ptr(tokens),
                                                       _lib.stream_ptr(self._device)))
            out = tokens
        self._cache_put(key, out)
        return out

    def extract_features_pair(self, image0, image1, cache_key0=None, cache_key1=None):
        """``extract_features`` of both images of a pair in one backbone pass (one launch per layer for both) -> (tokens0, tokens1),
        bitwise equal to two ``extract_features`` calls.  Coarse-only matcher, images of the same size, neither of them cached."""
        key0, key1 = self._cache_key(image0, cache_key0), self._cache_key(image1, cache_key1)
        assert self._pair_applies(image0, image1, key0, key1)
        H, W = image0.shape[2:]
        image0, image1 = image0.contiguous(), image1.contiguous()
        h, w = H // 8, W // 8
        tokens0 = torch.empty(h * w, 256, device=self._device, dtype=torch.float32)
        tokens1 = torch.empty(h * w, 256, device=self._device, dtype=torch.float32)
        _lib.check(self._lib.dfsfm_coarse_features_pair(self._h, _lib.ptr(image0), _lib.ptr(image1), H, W, _lib.ptr(self._pe_tokens(h, w)),
                                                        _lib.ptr(tokens0), _lib.ptr(tokens1), _lib.stream_ptr(self._device)))
        self._cache_put(key0, tokens0)
        self._cache_put(key1, tokens1)
        return tokens0, tokens1

    def _pair_applies(self, image0, image1, key0, key1):
        # the same name twice is one extraction and one cache entry: the one-image path does that
        return (not self.fine and image0.shape == image1.shape and (key0 is None or (key0 not in self._cache and key0 != key1))
                and (key1 is None or key1 not in self._cache))

    def _cache_put(self, key, out):
        if key is None:
            return
        nbytes = sum(t.numel() * t.element_size() for t in (out if isinstance(out, tuple) else (out,)))
        self._cache[key] = out
        self._cache_bytes += nbytes
        while len(self._cache) > 1 and (len(self._cache) > self._cache_size or self._cache_bytes > self._cache_bytes_max):
            _, old = self._cache.popitem(last=False)
            self._cache_bytes -= sum(t.numel() * t.element_size() for t in (old if isinstance(old, tuple) else (old,)))

    def fine_match(self, feat_f0, hw0_f, feat_f1, hw1_f, feat_c0, hw0_c, feat_c1, hw1_c, i_ids, j_ids):
        """FinePreprocess + loftr_fine + FineMatching -> (coords_normed * (W // 2) [M,2], std [M])."""
        M = int(i_ids.shape[0])
        coords = torch.zeros(M, 2, device=self._device, dtype=torch.float32)
        std = torch.zeros(M, device=self._device, dtype=torch.float32)
        if M > 0:
            i32, j32 = i_ids.to(torch.int32).contiguous(), j_ids.to(torch.int32).contiguous()
            _lib.check(self._lib.dfsfm_coarse_fine_match(self._h, _lib.ptr(feat_f0), hw0_f[0], hw0_f[1], _lib.ptr(feat_f1), hw1_f[0], hw1_f[1],
                                                         _lib.ptr(feat_c0), hw0_c[1], _lib.ptr(feat_c1), hw1_c[1], _lib.ptr(i32), _lib.ptr(j32), M,
                                                         _lib.ptr(coords), _lib.ptr(std), _lib.stream_ptr(self._device)))
        return coords, std

    def transform(self, feat0, feat1):
        """LocalFeatureTransformer (8 layers) in place on [L,256], [S,256] fp32 tokens."""
        _lib.check(self._lib.dfsfm_coarse_transformer(self._h, _lib.ptr(feat0), feat0.shape[0], _lib.ptr(feat1), feat1.shape[0],
                                                      _lib.stream_ptr(self._device)))
        return feat0, feat1

    def coarse_match(self, feat0, hw0_c, feat1, hw1_c, return_conf=False):
        L, S = hw0_c[0] * hw0_c[1], hw1_c[0] * hw1_c[1]
        cap = min(L, S)
        i_ids = torch.empty(cap, device=self._device, dtype=torch.int32)
        j_ids = torch.empty(cap, device=self._device, dtype=torch.int32)
        mconf = torch.empty(cap, device=self._device, dtype=torch.float32)
        count = torch.zeros(1, device=self._device, dtype=torch.int32)
        conf = torch.empty(L, S, device=self._device, dtype=torch.float32) if return_conf else None
        _lib.check(self._lib.dfsfm_coarse_match(self._h, _lib.ptr(feat0), hw0_c[0], hw0_c[1], _lib.ptr(feat1), hw1_c[0], hw1_c[1],
                                                self.thr, self.border_rm, self.temperature, _lib.ptr(i_ids), _lib.ptr(j_ids),
                                                _lib.ptr(mconf), _lib.ptr(count), cap, _lib.ptr(conf), _lib.stream_ptr(self._device)))
        n = int(count.item())  # the one device sync per pair (the reference's torch.where does the same)
        return i_ids[:n].long(), j_ids[:n].long(), mconf[:n], conf

    # ------------------------------------------------------------------------------ forward
    @torch.no_grad()
    def forward(self, data):
        """Same contract as LoFTR.forward (loftr.py:29-81): updates ``data`` in place."""
        if not self._h:
            raise _lib.DfsfmError("B200LoFTR: call .cuda() before forward (there is no CPU path)")
        with torch.cuda.device(self._device):   # the engine's kernels, workspaces and stream all belong to its own device
            return self._forward(data)

    def clear_cache(self):
        """Drop the per-image feature cache.  Entries are keyed by (pair_key name, H, W): a caller that re-uses a name for
        different pixels (another dataset root with the same relative paths) must clear it between scenes."""
        self._cache.clear()
        self._cache_bytes = 0

    def _forward(self, data):
        if not self._h:
            raise _lib.DfsfmError("B200LoFTR: call .cuda() before forward (there is no CPU path)")
        if self._packed is None:
            raise _lib.DfsfmError("B200LoFTR: load_state_dict() has not been called")
        im0, im1 = data["image0"], data["image1"]
        if im0.size(0) != 1:
            raise NotImplementedError("bs must be 1 (coarse_match_worker.py:86 asserts the same)")
        if "mask0" in data:
            raise NotImplementedError("padding masks are a training-time feature (loftr.py:61-63)")
        data.update({"bs": 1, "hw0_i": im0.shape[2:], "hw1_i": im1.shape[2:]})
        names = data.get("pair_key")
        k0 = k1 = None
        if names is not None:
            k0 = names[0][0] if isinstance(names[0], (list, tuple)) else names[0]
            k1 = names[1][0] if isinstance(names[1], (list, tuple)) else names[1]
        if self._pair_applies(im0, im1, self._cache_key(im0, k0), self._cache_key(im1, k1)):
            f0, f1 = self.extract_features_pair(im0, im1, k0, k1)
        else:
            f0 = self.extract_features(im0, k0)
            f1 = self.extract_features(im1, k1)
        if self.fine:
            (f0, ff0), (f1, ff1) = f0, f1
        hw0_c = (im0.shape[2] // 8, im0.shape[3] // 8)
        hw1_c = (im1.shape[2] // 8, im1.shape[3] // 8)
        data.update({"hw0_c": torch.Size(hw0_c), "hw1_c": torch.Size(hw1_c)})
        f0, f1 = self.transform(f0.clone(), f1.clone())
        keep_conf = bool(data.get("_return_conf_matrix", False))
        i_ids, j_ids, mconf, conf = self.coarse_match(f0, hw0_c, f1, hw1_c, keep_conf)
        if keep_conf:
            data["conf_matrix"] = conf[None]
            data["feat_c0"], data["feat_c1"] = f0[None], f1[None]
        b_ids = torch.zeros_like(i_ids)
        # coordinates in original-image pixels, same op order as coarse_matching.py:239-247
        scale = data["hw0_i"][0] / hw0_c[0]
        scale0 = scale * data["scale0"][b_ids][:, [1, 0]] if "scale0" in data else scale
        scale1 = scale * data["scale1"][b_ids][:, [1, 0]] if "scale1" in data else scale
        mkpts0_c = torch.stack([i_ids % hw0_c[1], i_ids // hw0_c[1]], dim=1) * scale0
        mkpts1_c = torch.stack([j_ids % hw1_c[1], j_ids // hw1_c[1]], dim=1) * scale1
        keep = mconf != 0
        data.update({
            "b_ids": b_ids, "i_ids": i_ids, "j_ids": j_ids, "gt_mask": mconf == 0,
            "m_bids": b_ids[keep], "mkpts0_c": mkpts0_c[keep], "mkpts1_c": mkpts1_c[keep], "mconf": mconf[keep],
        })
        if not self.fine:
            data.update({"mkpts0_f": data["mkpts0_c"], "mkpts1_f": data["mkpts1_c"]})
            return None
        # fine-level refinement (loftr.py:75-81, utils/fine_matching.py:63-74)
        hw0_f = (im0.shape[2] // 2, im0.shape[3] // 2)
        hw1_f = (im1.shape[2] // 2, im1.shape[3] // 2)
        data.update({"hw0_f": torch.Size(hw0_f), "hw1_f": torch.Size(hw1_f), "W": 5})
        coords2, std = self.fine_match(ff0, hw0_f, ff1, hw1_f, f0, hw0_c, f1, hw1_c, i_ids, j_ids)
        data["expec_f"] = torch.cat([coords2 / 2, std[:, None]], -1)
        scale_f = data["hw0_i"][0] / hw0_f[0]
        scale1_f = scale_f * data["scale1"][b_ids][:, [1, 0]] if "scale0" in data else scale_f
        data.update({"mkpts0_f": data["mkpts0_c"], "mkpts1_f": data["mkpts1_c"] + (coords2 * scale1_f)[:len(data["mconf"])]})
        return None
