// kernels_delivery.cu — the delivery loop's scene-change decision (hrb_delivery, include/hrb.h): one thread evaluates
// HopperRender.cpp:1126-1176 on the frame-delta history, as soon as pass 0 of the step's flow has written its raw delta.
#include "hrb_internal.cuh"

namespace hrb {

namespace {

__global__ void deliveryDecisionKernel(const DeliveryDecision d) {
    if (threadIdx.x != 0) return;
    unsigned delta = 0;
    if (d.append) {
        // m_totalFrameDelta (opticalFlowCalcSDR.cpp:92-93 / HDR): the raw window sum over the flow size and the divisor
        delta = *d.rawDelta / d.divisor;
        d.ring[d.slot] = delta;
    }
    long long d1 = 0, d2 = 0;
    bool scene = false;
    if (d.n >= 3) {
        // entry n-1 (nxt) is at ring[slot], entry n-2-i at ring[slot - 1 - i]
        long long total = 0;
        for (int i = 0; i < d.count; ++i) total += d.ring[(d.slot - 1 - i) & 15];
        const long long average = total / d.count;  // non-negative: floor division
        const long long nxt = d.ring[d.slot];
        const long long cur = d.ring[(d.slot - 1) & 15];
        d1 = cur - average;
        d2 = cur - nxt;
        scene = d1 >= d.threshold && d1 > 0 && d2 >= d.threshold && d2 > 0;
    }
    *d.gate = scene ? 1u : 0u;
    DeliveryRecord r;
    r.warped = !d.copy && !scene;
    r.sceneChange = scene;
    r.d1 = d1;
    r.d2 = d2;
    r.frameDelta = delta;
    *d.out = r;
}

}  // namespace

int launchDeliveryDecision(hrb_ofc* h, const DeliveryDecision& d) {
    deliveryDecisionKernel<<<1, 32, 0, h->stream>>>(d);
    HRB_LAUNCH_CHECK();
    return HRB_OK;
}

}  // namespace hrb
