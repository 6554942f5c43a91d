"""Rate control for the sequence encoder: a QP per coded unit, chosen from on-device size estimates.

DCVC-UF codes 64 quality levels with one model; the QP index selects the level and a larger index spends more bits.
`RateController` keeps a virtual buffer (bits spent minus the target's share of the units coded so far) and gives
every unit a budget that pays the buffer back over about `window_s` seconds.  It then searches the QP whose estimated
size fits that budget, asking an injected estimator (the models' `estimate_bits`, one analysis pass per QP, no entropy
coding) for the sizes of a few candidate QPs:

* the first unit of a type (intra / P) bisects [qp_min, qp_max] for the largest QP that fits (6 trials cover 64);
* later units start from the QP the previous unit of their type was coded at and take secant steps on log(bytes)
  against QP, with the slope learnt from the trials so far.

Intra and P units keep separate models.  No strict monotonicity is assumed: the choice is the largest tried QP whose
estimate fits the budget, or the tried QP with the fewest bytes when none fits.  Everything is integer or float
arithmetic on the estimates, so equal estimates give equal choices.

    rc = RateController(target_kbps=2000, fps=30)
    enc = SequenceEncoder(i_net, p_net, H, W, qp_i, qp_p, rate_control=rc)
"""
from __future__ import annotations

import math
from typing import Callable, Dict, List, Sequence

Estimator = Callable[[Sequence[int]], Sequence[int]]     # QPs -> estimated bytes, one per QP

# log(bytes) per QP step to start the secant from before two trials of a type have measured it: the intra streams of
# DESIGN.md §5 grow from about 150 KB to 440 KB over q 0 .. 63 at 1080p
_DEFAULT_SLOPE = math.log(440.0 / 150.0) / 63.0


class RateController:
    def __init__(self, target_kbps: float, fps: float = 30.0, qp_min: int = 0, qp_max: int = 63, max_trials: int = 6,
                 window_s: float = 1.0, tolerance: float = 0.03):
        if target_kbps <= 0 or fps <= 0 or window_s <= 0:
            raise ValueError("target_kbps, fps and window_s must be positive")
        if not (0 <= qp_min <= qp_max <= 63):
            raise ValueError("need 0 <= qp_min <= qp_max <= 63")
        if max_trials < 1:
            raise ValueError("max_trials must be at least 1")
        self.target_kbps, self.fps = float(target_kbps), float(fps)
        self.qp_min, self.qp_max, self.max_trials = int(qp_min), int(qp_max), int(max_trials)
        self.window_s, self.tolerance = float(window_s), float(tolerance)
        self.bits_per_frame = self.target_kbps * 1000.0 / self.fps
        self.buffer_bits = 0.0                     # bits spent - bits_per_frame * frames coded
        self.history: List[Dict] = []
        self._last_qp: Dict[bool, int] = {}         # per type: QP of the previous unit
        self._slope: Dict[bool, float] = {}         # per type: d log(bytes) / d QP

    def budget_bytes(self, count: int) -> float:
        """the next unit's budget: its frames' share of the target, minus the buffer's share over the window.  An intra
        picture gets one frame's share like any other; what it spends above that, the following units pay back."""
        frames_in_window = self.fps * self.window_s
        bits = count * self.bits_per_frame - self.buffer_bits * min(1.0, count / frames_in_window)
        return max(bits, 0.1 * count * self.bits_per_frame) / 8.0

    def choose(self, first: int, count: int, is_intra: bool, estimate: Estimator) -> int:
        """the QP of the unit of `count` pictures starting at `first`; `estimate(qps)` returns its size at each QP"""
        budget = self.budget_bytes(count)
        tried: Dict[int, int] = {}

        def probe(qp: int) -> int:
            if qp not in tried:
                tried[qp] = int(estimate([qp])[0])
            return tried[qp]

        if is_intra not in self._last_qp:
            qp = self._bisect(budget, probe, tried)
        else:
            qp = self._secant(budget, probe, tried, is_intra)
        self._learn_slope(is_intra, tried)
        self._last_qp[is_intra] = qp
        self.history.append({"first": first, "count": count, "is_intra": is_intra, "budget": budget,
                             "tried": sorted(tried.items()), "qp": qp, "bytes": None})
        return qp

    def update(self, actual_bytes: int) -> None:
        """the size the last chosen unit was coded at (the bytes written for it)"""
        h = self.history[-1]
        h["bytes"] = int(actual_bytes)
        self.buffer_bits += 8.0 * actual_bytes - h["count"] * self.bits_per_frame

    # ---------------------------------------------------------------- search
    def _bisect(self, budget, probe, tried) -> int:
        lo, hi = self.qp_min, self.qp_max      # invariant: every tried QP above hi is over budget
        while lo < hi and len(tried) < self.max_trials:
            mid = (lo + hi + 1) // 2
            if probe(mid) <= budget:
                lo = mid
            else:
                hi = mid - 1
        return lo       # a tried QP that fits, or qp_min when nothing tried did (saturated at the lower bound)

    def _secant(self, budget, probe, tried, is_intra) -> int:
        slope = self._slope.get(is_intra, _DEFAULT_SLOPE)
        qp = self._last_qp[is_intra]
        target = math.log(max(budget, 1.0))
        while len(tried) < self.max_trials:
            b = probe(qp)
            if budget * (1.0 - self.tolerance) <= b <= budget:
                break
            step = (target - math.log(max(b, 1))) / slope
            nxt = min(self.qp_max, max(self.qp_min, qp + int(round(step))))
            if nxt == qp:
                nxt = min(self.qp_max, max(self.qp_min, qp + (1 if b < budget else -1)))
            if nxt in tried:
                break                           # the neighbourhood is bracketed
            qp = nxt
        return self._pick(budget, tried)

    def _pick(self, budget, tried) -> int:
        fits = [q for q, b in tried.items() if b <= budget]
        if fits:
            return max(fits)
        return min(tried, key=lambda q: (tried[q], q))

    def _learn_slope(self, is_intra, tried) -> None:
        pts = sorted((q, b) for q, b in tried.items() if b > 0)
        if len(pts) < 2:
            return
        (q0, b0), (q1, b1) = pts[0], pts[-1]
        s = (math.log(b1) - math.log(b0)) / (q1 - q0)
        if s > 1e-4:
            self._slope[is_intra] = s
