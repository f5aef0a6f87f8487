#!/usr/bin/env python
"""Per-CTA timeline of the tile search kernels of one 4K flow calculation (debug aid, needs a GPU):
for every pass, the spread of CTA start / boxes-landed / runs-done / end times and the slowest CTAs.
usage: python tools/cta_timeline.py [W H] [R]"""
import sys, os
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import hopperrender_b200 as hr
from hopperrender_b200 import synth

W, H = (int(sys.argv[1]), int(sys.argv[2])) if len(sys.argv) > 2 else (3840, 2160)
R = int(sys.argv[3]) if len(sys.argv) > 3 else 16
g = hr.OpticalFlowCalcHDR(H, W, 0, 0, 8, 6, 0.0, 255.0, H)
g.m_opticalFlowSearchRadius = R
fr = [synth.make_frame(W, H, t, synth.SEED_BASE + 2, True) for t in range(5)]
for f in fr[:3]:
    g.updateFrame(f)
g.calculateOpticalFlow()
g.updateFrame(fr[3]); g.calculateOpticalFlow()
# 16 words per CTA.  A tile CTA covers 128 flow pixels along u and 32 * NWV >= 64 along v (u = x for Y steps, u = y for X
# steps), so no pass launches more CTAs than the bound below; a CTA whose record does not fit the slice records nothing.
lh, lw = g.m_opticalFlowFrameHeight, g.m_opticalFlowFrameWidth
WPP = 16 * max(-(-lw // 128) * -(-lh // 64), -(-lh // 128) * -(-lw // 64))
g.debugTimeline(WPP)
g.updateFrame(fr[4]); g.calculateOpticalFlow()
tl = g.readDebugTimeline(WPP)
for p in range(32):
    t = tl[p]
    t = t[t[:, 0] > 0]
    if not len(t):
        continue
    t0 = t[:, 0].min()
    st, bx, rn, en = [(t[:, k].astype(np.int64) - int(t0)) / 1e3 for k in range(4)]
    dur = en - st
    rounds = t[:, 7] % 100
    border = t[:, 7] >= 100
    print(f"pass {p:2d}: {len(t):4d} CTAs  kernel {en.max():7.1f} us | start max {st.max():6.1f} | boxes-landed-start med {np.median(bx-st):6.1f} max {(bx-st).max():6.1f} | "
          f"runs med {np.median(rn-bx):6.1f} max {(rn-bx).max():6.1f} | tail med {np.median(en-rn):5.1f} max {(en-rn).max():5.1f} | CTA dur med {np.median(dur):6.1f} max {dur.max():6.1f} | "
          f"rounds max {rounds.max()} mean {rounds.mean():.2f} border {border.sum()}")
    worst = np.argsort(-en)[:4]
    for i in worst:
        print("          dbg:", [round((int(t[i, k]) - int(t0)) / 1e3, 1) if t[i, k] else 0 for k in (0, 1, 2, 3)], int(t[i,5]), int(t[i,6]), f"nwv{int(t[i,8])}")
    print("          slowest:", [(int(t[i, 5]), int(t[i, 6]), f"sm{int(t[i,4])}", f"st{st[i]:.1f}", f"bx{bx[i]-st[i]:.1f}", f"run{rn[i]-bx[i]:.1f}", f"end{en[i]:.1f}", int(t[i, 7])) for i in worst])
    # CTAs per SM and per-SM busy time
    sm = t[:, 4].astype(int)
    per = np.bincount(sm, minlength=148)
    print(f"          CTAs per SM: min {per.min()} max {per.max()}; SMs used {np.count_nonzero(per)}")
