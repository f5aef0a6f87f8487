#!/usr/bin/env python
"""CTAs per SM of the tile search passes of one flow calculation, measured from the per-CTA debug timeline (needs a GPU).

For every pass the tile kernel (sadTileKernel, kernels_search_slide.cu) runs: window size, step, warps per CTA (NWV), the
grid, the most CTAs that were resident on one SM at the same time (from the CTAs' start / end times and SM ids), the
rounds the grid needs on that many slots per SM, and the kernel time.  The slot count is what the runtime places: the
launch's registers, shared memory and carve-out decide it, not the cost model that picked NWV.
usage: python tools/tile_occupancy.py [W H] [R]"""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

import hopperrender_b200 as hr
from hopperrender_b200 import synth

W, H = (int(sys.argv[1]), int(sys.argv[2])) if len(sys.argv) > 2 else (3840, 2160)
R = int(sys.argv[3]) if len(sys.argv) > 3 else 16
sms = torch.cuda.get_device_properties(0).multi_processor_count
g = hr.OpticalFlowCalcHDR(H, W, 0, 0, 8, 6, 0.0, 255.0, H)
g.m_opticalFlowSearchRadius = R
g.setTapMode(True)  # launches the passes one by one: a replayed ladder graph would not carry the timeline
fr = [synth.make_frame(W, H, t, synth.SEED_BASE + 2, True) for t in range(4)]
for f in fr[:3]:
    g.updateFrame(f)
g.calculateOpticalFlow()
lh, lw = g.m_opticalFlowFrameHeight, g.m_opticalFlowFrameWidth
WPP = 16 * max(-(-lw // 128) * -(-lh // 64), -(-lh // 128) * -(-lw // 64))  # every tile CTA of a pass (NWV >= 2)
g.debugTimeline(WPP)
g.updateFrame(fr[3])
g.calculateOpticalFlow()
tl = g.readDebugTimeline(WPP)
print(f"{torch.cuda.get_device_name(0)}, {sms} SMs, {W}x{H} R {R}")
for p in range(g.numPasses()):
    t = tl[p]
    t = t[t[:, 0] > 0]
    if not len(t):
        continue
    info = g.passInfo(p)
    st, en = t[:, 0].astype(np.int64), t[:, 3].astype(np.int64)
    sm = t[:, 4].astype(np.int64)
    resident = 0
    for s in np.unique(sm):
        a, b = st[sm == s], en[sm == s]
        # the most intervals [start, end) of this SM that overlap at one time: sweep over the start / end events
        ev = np.concatenate([np.stack([a, np.ones_like(a)], 1), np.stack([b, -np.ones_like(b)], 1)])
        ev = ev[np.lexsort((ev[:, 1], ev[:, 0]))]
        resident = max(resident, int(np.cumsum(ev[:, 1]).max()))
    n = len(t)
    print(f"pass {p:2d} ws {info['windowSize']:4d} step {info['step']}: NWV {int(t[0, 8])} grid {int(t[:, 5].max()) + 1} x {int(t[:, 6].max()) + 1} = {n:4d} CTAs, "
          f"resident per SM {resident}, rounds {-(-n // (sms * resident))}, kernel {(en.max() - st.min()) / 1e3:6.1f} us")
g.close()
