"""Roofline denominators: the driver-written MEASURED_PEAKS.json (or the profiling recipe's fallback)."""
from __future__ import annotations

import json
import os

_FALLBACK = dict(hbm_gbs=6650.0, bf16_tflops=1590.0, bf16_tflops_sustained=1400.0, source="fallback")
NVLINK_PEER_GBS = 770.0  # measured peer-copy bandwidth per direction on this pool (B200_PROFILING.md)


def measured_peaks() -> dict:
    here = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    try:
        with open(os.path.join(here, "MEASURED_PEAKS.json")) as f:
            d = json.load(f)
        return dict(hbm_gbs=float(d["hbm_gbs"]), bf16_tflops=float(d["bf16_tflops"]),
                    bf16_tflops_sustained=float(d.get("bf16_tflops_sustained", d["bf16_tflops"])), source="measured")
    except Exception:
        return dict(_FALLBACK)
