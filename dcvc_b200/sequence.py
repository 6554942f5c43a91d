"""Sequence-level driver: the loop the reference's `test_video.py` runs around the codec proxies — which pictures are intra,
how P pictures are grouped into chunks, when the feature memory is reset, and how every coded unit is framed in the
bitstream container (reference: test_video.py:204-266 encoder loop, :281-372 decoder loop; SURVEY.md §8 f2 "callers
either side of the path").  Frames enter and leave as 8-bit YUV 4:2:0 planes (src_type "yuv420") or 8-bit planar RGB
[3,H,W] (src_type "png", BT.709 as test_cfg/all_RGB.json); the conversion to and from the model tensor is the device
frame IO of dcvc_b200.frame_io unless other converters are injected (the CPU tests inject the oracle's).  `run_job`
is one job of test_video.py end to end: encode, decode, distortion, and the per-job JSON record.

    enc = SequenceEncoder(i_net, p_net, height, width, qp_i, qp_p, frame_delay=8)
    data = enc.encode(frames)                       # frames: iterable of (y, u, v) uint8 planes
    for y, u, v in SequenceDecoder(i_net, p_net, frame_delay=8).decode(data, len(frames)): ...

`i_net` / `p_net` are the model mirrors of dcvc_b200.model (or the reference's own models: same API).
"""
from __future__ import annotations

import io
from dataclasses import dataclass
from typing import Callable, Iterable, List, Optional, Sequence, Tuple

from .stream import NalType, SPSHelper, read_header, read_ip_remaining, read_sps_remaining, write_ip, write_sps


@dataclass(frozen=True)
class Unit:
    """one coded unit of the sequence: an intra picture or a chunk of `count` P pictures starting at `first`"""
    first: int
    count: int
    is_intra: bool
    reset_feature_memory: int


def frame_schedule(frame_num: int, frame_delay: int, intra_period: int = -1, reset_interval: int = 32,
                   force_intra: bool = False) -> List[Unit]:
    """The reference's picture-type decisions (test_video.py:204-236), as a list.

    Picture 0 is intra; with intra_period > 1 every picture whose index is 1 modulo the period (except picture 1) is
    intra too (the period must be a multiple of the frame delay); intra_period == 1 or force_intra codes everything
    intra.  P pictures are coded `frame_delay` at a time (the tail chunk is shorter; the caller pads it by repeating
    the last picture, test_video.py:101-107).  A chunk starting at picture f resets the feature memory when
    (f + frame_delay) % reset_interval == 1."""
    if frame_delay < 1 or frame_num < 0:
        raise ValueError("bad frame_delay / frame_num")
    if intra_period > 1 and intra_period % frame_delay != 0:
        raise ValueError("intra_period must be a multiple of the frame delay")
    units, f = [], 0
    while f < frame_num:
        intra = force_intra or f == 0 or intra_period == 1
        if intra_period > 1 and f != 1 and f % intra_period == 1:
            intra = True
        if intra:
            units.append(Unit(f, 1, True, 0))
            f += 1
            continue
        count = min(frame_delay, frame_num - f)
        reset = 1 if (reset_interval > 0 and (f + frame_delay) % reset_interval == 1) else 0
        units.append(Unit(f, count, False, reset))
        f += count
    return units


Planes = Tuple["object", "object", "object"]      # (y [H,W], u [H/2,W/2], v [H/2,W/2]) uint8 tensors


class UnitTimer:
    """The reference driver's timing of one coded unit (test_video.py:219-221 + 263-267, 284-285 + 321-325): device
    synchronise, start event, the unit's work (model call + container framing on the host), end event, synchronise."""

    def __init__(self, device=None):
        import torch
        self.torch, self.device = torch, device
        self.e0 = torch.cuda.Event(enable_timing=True)
        self.e1 = torch.cuda.Event(enable_timing=True)

    def start(self):
        self.torch.cuda.synchronize(self.device)
        self.e0.record()

    def stop(self) -> float:
        self.e1.record()
        self.torch.cuda.synchronize(self.device)
        return self.e0.elapsed_time(self.e1)


def _device_to_model(planes: Sequence[Planes], frame_delay: int):
    """8-bit planes of 1 .. frame_delay pictures -> fp16 [1, 3*n, H, W] channels_last on the device of the planes"""
    import torch

    from .frame_io import yuv420_to_frame
    y0 = planes[0][0]
    H, W = y0.shape
    x = torch.empty((1, 3 * len(planes), H, W), dtype=torch.float16, device=y0.device).contiguous(memory_format=torch.channels_last)
    for i, (y, u, v) in enumerate(planes):
        yuv420_to_frame(y, u, v, out=x, channel=3 * i)
    return x


def _device_from_model(x_hat, height: int, width: int) -> Planes:
    from .frame_io import frame_to_yuv420
    return frame_to_yuv420(x_hat, height, width)


def _device_rgb_to_model(frames: Sequence["object"], frame_delay: int):
    """uint8 [3,H,W] RGB pictures (1 .. frame_delay) -> fp16 [1, 3*n, H, W] channels_last (test_video.py:88-122)"""
    import torch

    from .frame_io import rgb_to_frame
    H, W = frames[0].shape[1:]
    x = torch.empty((1, 3 * len(frames), H, W), dtype=torch.float16, device=frames[0].device).contiguous(memory_format=torch.channels_last)
    for i, rgb in enumerate(frames):
        rgb_to_frame(rgb, out=x, channel=3 * i)
    return x


def _device_rgb_from_model(x_hat, height: int, width: int):
    from .frame_io import frame_to_rgb
    return frame_to_rgb(x_hat, height, width)


_CONVERTERS = {"yuv420": (_device_to_model, _device_from_model), "png": (_device_rgb_to_model, _device_rgb_from_model)}


def _converters(src_type: str):
    if src_type not in _CONVERTERS:
        raise ValueError(f"src_type must be 'yuv420' or 'png', got {src_type!r}")
    return _CONVERTERS[src_type]


class SequenceEncoder:
    def __init__(self, i_net, p_net, height: int, width: int, qp_i: int, qp_p: int, frame_delay: int = 8,
                 intra_period: int = -1, reset_interval: int = 32, force_intra: bool = False,
                 to_model: Optional[Callable] = None, src_type: str = "yuv420", rate_control=None):
        self.i_net, self.p_net = i_net, p_net
        self.src_type = src_type
        # rate_control: a dcvc_b200.rate_control.RateController; each unit's QP then comes from it (qp_i / qp_p unused)
        self.rate_control = rate_control
        self.height, self.width = height, width
        self.qp_i, self.qp_p = qp_i, qp_p
        self.frame_delay, self.intra_period, self.reset_interval = frame_delay, intra_period, reset_interval
        self.force_intra = force_intra
        self.to_model = to_model or _converters(src_type)[0]
        self.padding_r, self.padding_b = i_net.get_padding_size(height, width, 16)     # test_video.py:189
        self.bits: List[int] = []          # per picture, like the reference's `bits` list (chunk bits on its first picture)
        self.timer = None                  # UnitTimer: the reference's per-unit timing protocol (test_video.py:219-267)
        self.unit_ms: List[float] = []

    def encode(self, frames: Iterable[Planes]) -> bytes:
        frames = list(frames)
        out = io.BytesIO()
        sps_helper = SPSHelper()
        self.bits = []
        for unit in frame_schedule(len(frames), self.frame_delay, self.intra_period, self.reset_interval, self.force_intra):
            group = list(frames[unit.first:unit.first + unit.count])
            if not unit.is_intra:
                group += [group[-1]] * (self.frame_delay - len(group))      # tail chunk: repeat the last picture
            x = self.to_model(group, self.frame_delay)
            if self.timer:
                self.timer.start()
            rc = self.rate_control
            if unit.is_intra:
                qp = self.qp_i
                if rc is not None:
                    qp = rc.choose(unit.first, unit.count, True, lambda qps: [
                        r["bytes"] for r in self.i_net.estimate_bits(x, qps, self.padding_b, self.padding_r)])
                encoded = self.i_net.compress(x, qp, self.padding_b, self.padding_r)
                if not self.force_intra:
                    self.p_net.clear_dpb()
                    self.p_net.add_ref_feature_from_frame(encoded["x_hat"])
            else:
                qp = self.qp_p
                if rc is not None:
                    qp = rc.choose(unit.first, unit.count, False, lambda qps: [
                        r["bytes"] for r in self.p_net.estimate_bits(x, qps, unit.reset_feature_memory, self.padding_b,
                                                                     self.padding_r)])
                encoded = self.p_net.compress(x, qp, unit.reset_feature_memory, self.padding_b, self.padding_r)
            sps = {"sps_id": -1, "height": self.height, "width": self.width}
            sps_id, is_new = sps_helper.get_sps_id(sps)
            sps["sps_id"] = sps_id
            n = write_sps(out, sps) if is_new else 0
            n += write_ip(out, unit.is_intra, sps_id, qp, encoded["ec_parallel"], unit.reset_feature_memory,
                          encoded["bit_stream"])
            self.bits += [n * 8] + [0] * (unit.count - 1)
            if rc is not None:
                rc.update(n)
            if self.timer:
                self.unit_ms.append(self.timer.stop())
        return out.getvalue()


class SequenceDecoder:
    def __init__(self, i_net, p_net, frame_delay: int = 8, force_intra: bool = False,
                 from_model: Optional[Callable] = None, src_type: str = "yuv420"):
        self.i_net, self.p_net = i_net, p_net
        self.frame_delay, self.force_intra = frame_delay, force_intra
        self.src_type = src_type
        self.from_model = from_model or _converters(src_type)[1]
        self.timer = None
        self.unit_ms: List[float] = []

    def decode(self, data: bytes, frame_num: int):
        """yields `frame_num` pictures in display order: (y, u, v) uint8 planes, or [3,H,W] uint8 RGB for png"""
        f = io.BytesIO(data)
        sps_helper = SPSHelper()
        done = 0
        while done < frame_num:
            if self.timer:
                self.timer.start()
            header = read_header(f)
            while header["nal_type"] == NalType.NAL_SPS:
                sps_helper.add_sps_by_id(read_sps_remaining(f, header["sps_id"]))
                header = read_header(f)
            sps = sps_helper.get_sps_by_id(header["sps_id"])
            if sps is None:
                raise ValueError("coded unit refers to an unknown sequence parameter set")
            qp, ec_part, reset, bit_stream = read_ip_remaining(f)
            if header["nal_type"] == NalType.NAL_I:
                decoded = self.i_net.decompress(bit_stream, sps, qp, ec_part)
                if not self.force_intra:
                    self.p_net.clear_dpb()
                    self.p_net.add_ref_feature_from_frame(decoded["x_hat"], False)
                count = 1
            elif header["nal_type"] == NalType.NAL_P:
                decoded = self.p_net.decompress(bit_stream, sps, qp, ec_part, reset)
                count = min(self.frame_delay, frame_num - done)
            else:
                raise ValueError("unexpected unit type in a DCVC-UF stream")
            x_hat = decoded["x_hat"]
            if self.timer:
                self.unit_ms.append(self.timer.stop())
            for i in range(count):
                yield self.from_model(x_hat[i] if isinstance(x_hat, (list, tuple)) else x_hat, sps["height"], sps["width"])
            done += count


TIME_BYPASS_UNITS = 4      # test_video.py:376-377: the first 4 coded units are warm-up for the average unit times


def run_job(i_net, p_net, frames: Sequence, height: int, width: int, qp_i: int, qp_p: int, frame_delay: int = 8,
            intra_period: int = -1, reset_interval: int = 32, src_type: str = "yuv420", calc_ssim: bool = False,
            verbose_json: bool = False, verbose: int = 0, to_model: Optional[Callable] = None,
            metrics: Optional[Callable] = None, timer: Optional[Callable] = None, rate_control=None):
    """One job of test_video.py (run_one_point_with_stream, test_video.py:166-398): encode `frames`, decode the
    stream, measure every decoded picture against its source, and build the per-job record.

    Returns (bitstream, log): the bytes test_video.py writes to <seq>_q<qp_i>.bin and the dict it writes to the JSON
    beside it (generate_log_json's schema, see dcvc_b200.metrics.log_json).  `bits` of a unit include the SPS bytes
    in front of it and sit on the unit's first picture; `frame_types` is 0 per intra picture and 1 per P picture of a
    chunk (the padded tail of the last chunk not counted).  Unit times come from `timer` (default UnitTimer: the
    reference's synchronise + events protocol); with verbose >= 1 and more than 4 units the averages without the first
    4 units are reported in seconds, as the reference does.  Distortion is computed outside the timed regions.

    Injection points for tests: `to_model` (source frames -> model tensor), `metrics` (a factory with Distortion's
    signature and .add / .results), `timer` (a factory of objects with .start() / .stop() -> ms).

    `rate_control` (a dcvc_b200.rate_control.RateController) chooses every unit's QP instead of qp_i / qp_p; its size
    trials run inside the unit's timed region, as encoding time."""
    import time

    if metrics is None:
        from .metrics import Distortion as metrics
    from .metrics import log_json
    frames = list(frames)
    frame_num = len(frames)
    timer = timer or UnitTimer
    start_time = time.time()
    enc = SequenceEncoder(i_net, p_net, height, width, qp_i, qp_p, frame_delay, intra_period, reset_interval,
                          to_model=to_model, src_type=src_type, rate_control=rate_control)
    enc.timer = timer()
    data = enc.encode(frames)
    frame_types: List[int] = []
    for unit in frame_schedule(frame_num, frame_delay, intra_period, reset_interval):
        frame_types += [0] if unit.is_intra else [1] * unit.count

    dist = metrics(src_type, height, width, calc_ssim, frame_num)
    dec = SequenceDecoder(i_net, p_net, frame_delay, from_model=lambda x_hat, h, w: x_hat, src_type=src_type)
    dec.timer = timer()
    for f, x_hat in enumerate(dec.decode(data, frame_num)):
        dist.add(x_hat, frames[f])          # cropped to height x width inside, as test_video.py:340
    psnrs, ssims = dist.results()
    test_time = time.time() - start_time

    enc_s = [ms / 1000.0 for ms in enc.unit_ms]
    dec_s = [ms / 1000.0 for ms in dec.unit_ms]
    avg_enc = avg_dec = None
    if verbose >= 1 and len(enc_s) > TIME_BYPASS_UNITS:
        enc_s, dec_s = enc_s[TIME_BYPASS_UNITS:], dec_s[TIME_BYPASS_UNITS:]
        avg_enc, avg_dec = sum(enc_s) / len(enc_s), sum(dec_s) / len(dec_s)
    log = log_json(frame_num, height * width, test_time, frame_types, enc.bits, psnrs, ssims, verbose=verbose_json,
                   avg_encoding_time=avg_enc, avg_decoding_time=avg_dec)
    return data, log
