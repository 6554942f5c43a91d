"""Host-side mirror of the reference's model API for the hot path (src/models/image_model.py:126-217,
src/models/common_model.py:33-70,102-108,152-155): same method names, arguments and return values,
so scripts written against `DMCI` (test_video.py:226-238, 312-317) read the same.  It owns the
parameters as a plain state_dict; all inference goes through `inference_extensions_cuda`.
"""
from __future__ import annotations

from collections import OrderedDict

import numpy as np
import torch

from . import entropy
from .spec import QP_NUM, dmci_spec, synth_state_dict


class DMCI:
    def __init__(self):
        self._spec = dmci_spec()
        self._sd = OrderedDict((k, torch.zeros(v)) for k, v in self._spec.items())
        self.proxy = None
        self.skip_thres = 0.0
        self._cdf = None

    # ---- parameters
    @classmethod
    def synthetic(cls, seed: int = 0) -> "DMCI":
        m = cls()
        m.load_state_dict(synth_state_dict(m._spec, seed))
        return m

    def state_dict(self):
        return OrderedDict(self._sd)

    def load_state_dict(self, sd, strict: bool = True):
        missing = [k for k in self._spec if k not in sd]
        if strict and missing:
            raise KeyError(f"missing keys: {missing[:4]}...")
        for k, shape in self._spec.items():
            if k in sd:
                if tuple(sd[k].shape) != tuple(shape):
                    raise ValueError(f"shape mismatch for {k}: {tuple(sd[k].shape)} vs {shape}")
                self._sd[k] = sd[k].detach().clone()
        self.proxy = None   # stale cached params must not survive a reload (common_model.py:205-210)
        self._cdf = None

    def half(self):
        self._sd = OrderedDict((k, v.half()) for k, v in self._sd.items())
        self.proxy = None
        return self

    def to(self, device=None, memory_format=None):
        if device is not None:
            self._sd = OrderedDict((k, v.to(device)) for k, v in self._sd.items())
            self.proxy = None
        return self

    def eval(self):
        return self

    @staticmethod
    def qp_num():
        return QP_NUM

    @staticmethod
    def get_padding_size(height, width, p=64):
        new_h = (height + p - 1) // p * p
        new_w = (width + p - 1) // p * p
        return new_w - width, new_h - height   # (padding_right, padding_bottom) common_model.py:102-108

    # ---- entropy tables
    def update(self, skip_thres):
        """CompressionModel.update (common_model.py:152-155): build the quantised CDF tables."""
        self.skip_thres = float(skip_thres)
        zc, zl = entropy.bit_estimator_cdf_tables(self._sd["bit_estimator_z.h"], self._sd["bit_estimator_z.b"],
                                                  self._sd["bit_estimator_z.a"])
        yc, yl = entropy.gaussian_cdf_tables()
        self._cdf = (zc, zl, yc, yl)

    def add_cdf_to_state_dict(self, state_dict):
        if self._cdf is None:
            raise RuntimeError("call update(skip_thres) first")
        zc, zl, yc, yl = self._cdf
        state_dict["gaussian_encoder.quantized_cdf"] = torch.from_numpy(np.ascontiguousarray(yc))
        state_dict["gaussian_encoder.cdf_length"] = torch.from_numpy(np.ascontiguousarray(yl))
        state_dict["bit_estimator_z.quantized_cdf"] = torch.from_numpy(np.ascontiguousarray(zc))
        state_dict["bit_estimator_z.cdf_length"] = torch.from_numpy(np.ascontiguousarray(zl))
        return state_dict

    # ---- inference (image_model.py:194-217)
    def _ensure_proxy(self):
        if self.proxy is None:
            from inference_extensions_cuda import DMCIProxy  # no fallback: raises if unavailable
            sd = self.add_cdf_to_state_dict(self.state_dict())
            self.proxy = DMCIProxy()
            self.proxy.set_param(sd, self.skip_thres)

    def compress(self, x, qp, padding_b, padding_r):
        self._ensure_proxy()
        bit_stream, x_hat, ec_parallel = self.proxy.compress(x, qp, padding_b, padding_r)
        return {"bit_stream": bit_stream.tobytes(), "x_hat": x_hat, "ec_parallel": ec_parallel}

    def estimate_bits(self, x, qps, padding_b, padding_r):
        """compress()'s size at each QP of `qps` without coding: one dict per QP (bits_y, bits_z, ec_parallel, bytes, ...)"""
        self._ensure_proxy()
        return self.proxy.estimate_bits(x, qps, padding_b, padding_r)

    def decompress(self, bit_stream, sps, qp, ec_part):
        self._ensure_proxy()   # the reference needs a prior compress(); we tolerate decode-first use
        x_hat = self.proxy.decompress(np.frombuffer(bit_stream, dtype=np.uint8), qp, sps["height"], sps["width"],
                                      ec_part)
        return {"x_hat": x_hat}


class DMC(DMCI):
    """Host-side mirror of the reference's HT-S video model API (src/models/video_model_ht.py:320-450):
    clear_dpb / add_ref_feature_from_frame / compress / decompress, chunk = 8 frames stacked on the channel axis."""

    def __init__(self):
        from .spec import hts_spec
        self._spec = hts_spec()
        self._sd = OrderedDict((k, torch.zeros(v)) for k, v in self._spec.items())
        self.proxy = None
        self.skip_thres = 0.0
        self._cdf = None

    @classmethod
    def synthetic(cls, seed: int = 1) -> "DMC":
        m = cls()
        m.load_state_dict(synth_state_dict(m._spec, seed))
        return m

    def clear_dpb(self):
        # the reference forgets ref_feature / memory / ctx (video_model_ht.py:364-367); the proxy's state is rebuilt by the next
        # add_ref_feature_from_frame.  Coding a P unit in between would silently use the previous GOP's state: refuse it.
        self._dpb_cleared = True

    def _ensure_proxy(self):
        if self.proxy is None:
            from inference_extensions_cuda import DMCHTSProxy
            sd = self.add_cdf_to_state_dict(self.state_dict())
            self.proxy = DMCHTSProxy()
            self.proxy.set_param(sd, self.skip_thres)

    def add_ref_feature_from_frame(self, frame, apply_feature_adaptor=True):
        self._ensure_proxy()
        self._dpb_cleared = False
        return self.proxy.add_ref_feature_from_frame(frame, apply_feature_adaptor)

    def _check_dpb(self):
        if getattr(self, "_dpb_cleared", True):
            raise RuntimeError("no reference feature: call add_ref_feature_from_frame after clear_dpb / before the first P unit")

    def compress(self, x, qp, reset_feature_memory, padding_b, padding_r):
        self._ensure_proxy()
        self._check_dpb()
        bit_stream, ec_parallel = self.proxy.compress(x, qp, reset_feature_memory, padding_b, padding_r)
        return {"bit_stream": bit_stream.tobytes(), "ec_parallel": ec_parallel}

    def estimate_bits(self, x, qps, reset_feature_memory, padding_b, padding_r):
        """compress()'s size at each QP of `qps` without coding (see DMCI.estimate_bits); needs the same reference as
        compress()"""
        self._ensure_proxy()
        self._check_dpb()
        return self.proxy.estimate_bits(x, qps, reset_feature_memory, padding_b, padding_r)

    def decompress(self, bit_stream, sps, qp, ec_part, reset_feature_memory):
        self._ensure_proxy()
        self._check_dpb()
        x_hat = self.proxy.decompress(np.frombuffer(bit_stream, dtype=np.uint8), qp, sps["height"], sps["width"],
                                      ec_part, reset_feature_memory)
        return {"x_hat": x_hat}


class DMCLD(DMC):
    """Host-side mirror of the reference's low-delay video model API (src/models/video_model_ld.py:191-306): the class
    there is also called DMC; one frame per compress / decompress, `x_hat` is a single tensor."""

    def __init__(self):
        from .spec import ld_spec
        self._spec = ld_spec()
        self._sd = OrderedDict((k, torch.zeros(v)) for k, v in self._spec.items())
        self.proxy = None
        self.skip_thres = 0.0
        self._cdf = None

    @classmethod
    def synthetic(cls, seed: int = 2) -> "DMCLD":
        m = cls()
        m.load_state_dict(synth_state_dict(m._spec, seed))
        return m

    def _ensure_proxy(self):
        if self.proxy is None:
            from inference_extensions_cuda import DMCLDProxy
            sd = self.add_cdf_to_state_dict(self.state_dict())
            self.proxy = DMCLDProxy()
            self.proxy.set_param(sd, self.skip_thres)


class DMCHTL(DMC):
    """DMC(ModelStructure.HTL) of src/models/video_model_ht.py:320-450 (same API as the HT-S model)."""

    def __init__(self):
        from .spec import htl_spec
        self._spec = htl_spec()
        self._sd = OrderedDict((k, torch.zeros(v)) for k, v in self._spec.items())
        self.proxy = None
        self.skip_thres = 0.0
        self._cdf = None

    @classmethod
    def synthetic(cls, seed: int = 3) -> "DMCHTL":
        m = cls()
        m.load_state_dict(synth_state_dict(m._spec, seed))
        return m

    def _ensure_proxy(self):
        if self.proxy is None:
            from inference_extensions_cuda import DMCHTLProxy
            sd = self.add_cdf_to_state_dict(self.state_dict())
            self.proxy = DMCHTLProxy()
            self.proxy.set_param(sd, self.skip_thres)
