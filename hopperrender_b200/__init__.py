"""hopperrender_b200 — HopperRender's optical-flow frame-interpolation hot path, B200-native.

The product is the CUDA library `libhrb.so` (C ABI in include/hrb.h).  This package is the thin
host-side mirror of the reference's calculator classes used by tests and bench.py.  Importing it
loads the CUDA library and fails loudly when it is missing — there is no CPU fallback.
"""
from . import _lib
from .ofc import (BlendedFrame, Delivery, FlowBatch, GreyFlow, HSVFlow, OpticalFlowCalc, OpticalFlowCalcHDR, OpticalFlowCalcSDR, SideBySide1,
                  SideBySide2, SplitSearch, WarpedFrame12, WarpedFrame21, kernel_launch_count, microbench_sad_peak, split_plan)

_lib.load()

__all__ = ["OpticalFlowCalc", "OpticalFlowCalcSDR", "OpticalFlowCalcHDR", "WarpedFrame12", "WarpedFrame21", "BlendedFrame",
           "HSVFlow", "GreyFlow", "SideBySide1", "SideBySide2", "SplitSearch", "split_plan", "FlowBatch", "Delivery", "kernel_launch_count", "microbench_sad_peak"]
