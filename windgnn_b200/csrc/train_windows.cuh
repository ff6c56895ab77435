// Training on windows over one table: the windows' first GI rows, and the gate gradients of every (window, step)
// summed per table row.
//
// The GCN, the input projection and the backward of both depend only on a table row, and the backward is linear in
// the input-gate gradient dGI.  So when the windows table[starts[n] : starts[n] + L] overlap, the forward runs those
// stages once per row of the span the windows cover (abi.cu, train_forward), and the backward sums, per span row t,
// the dGI rows of every (n, l) that read it (starts[n] + l = t), then runs dW_ih, dU and the GCN backward once per
// span row instead of once per (window, step).  A materialised batch x [B][T] is such a table, x.view(B*T), with
// windows that tile it (starts[n] = n*T): every row has one contributor, and the backward reads dGI in place.
#pragma once

#include "wg_common.cuh"

namespace wg {

// row0[n] = n * L: the first GI rows of N windows that tile the table (a materialised batch)
__global__ void tiled_row0_kernel(long long* __restrict__ row0, long long N, int L) {
    const long long n = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (n < N) row0[n] = n * L;
}

constexpr int kDgiWarps = 8;   // rows per CTA (one warp each)
constexpr int kDgiVec = 3;     // float4 columns per lane: 3H <= 384, i.e. H <= 128 (training serves H <= 106)

// DG    [N*L][ld]  the BPTT kernel's gate gradients, window-major; columns [0, G4) summed (G4: 3H rounded up to 4)
// ssort [N]        the windows' starts relative to the span's first row, ascending
// wsort [N]        the windows in that order (ties by window index)
// dgi   [span][ld] dgi[t] = sum of DG[wsort[k] * L + t - ssort[k]] over the k with t - L < ssort[k] <= t, in ascending
//                  k, the first term as is (no 0 + x: a row with one contributor is an exact copy); rows no window
//                  covers are zero, and so are the columns [G4, ld) (gemm_kb_kernel reads them and discards the result)
// The windows covering row t are the contiguous range of the sorted list found by two binary searches.  The order of
// the sum is fixed, so the result is reproducible bit for bit.  Every DG element is read once: HBM-bound.
__global__ void __launch_bounds__(kDgiWarps * 32)
    dgi_rows_kernel(const float* __restrict__ DG, const long long* __restrict__ ssort,
                    const long long* __restrict__ wsort, long long N, int L, long long span, int ld, int G4,
                    float* __restrict__ dgi) {
    const int lane = threadIdx.x & 31;
    const long long t = (long long)blockIdx.x * kDgiWarps + (threadIdx.x >> 5);
    if (t >= span) return;
    auto lower = [&](long long v) {   // first k with ssort[k] >= v
        long long a = 0, b = N;
        while (a < b) {
            const long long m = (a + b) >> 1;
            if (__ldg(ssort + m) < v) a = m + 1;
            else b = m;
        }
        return a;
    };
    const long long k0 = lower(t - L + 1), k1 = lower(t + 1);
    const int nv = G4 >> 2;
    float4 acc[kDgiVec];
#pragma unroll
    for (int i = 0; i < kDgiVec; ++i) acc[i] = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
    if (k0 < k1) {
        {   // the first contributor initialises the sum
            const float* src = DG + ((size_t)__ldg(wsort + k0) * L + (size_t)(t - __ldg(ssort + k0))) * ld;
#pragma unroll
            for (int i = 0; i < kDgiVec; ++i) {
                const int c = lane + 32 * i;
                if (c < nv) acc[i] = __ldg(reinterpret_cast<const float4*>(src) + c);
            }
        }
#pragma unroll 2
        for (long long k = k0 + 1; k < k1; ++k) {
            const float* src = DG + ((size_t)__ldg(wsort + k) * L + (size_t)(t - __ldg(ssort + k))) * ld;
#pragma unroll
            for (int i = 0; i < kDgiVec; ++i) {
                const int c = lane + 32 * i;
                if (c < nv) {
                    const float4 v = __ldg(reinterpret_cast<const float4*>(src) + c);
                    acc[i].x += v.x;
                    acc[i].y += v.y;
                    acc[i].z += v.z;
                    acc[i].w += v.w;
                }
            }
        }
    }
    float4* dst = reinterpret_cast<float4*>(dgi + (size_t)t * ld);
#pragma unroll
    for (int i = 0; i < kDgiVec; ++i) {
        const int c = lane + 32 * i;
        if (c < nv) dst[c] = acc[i];
    }
    for (int c = nv + lane; c < (ld >> 2); c += 32) dst[c] = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
}

}  // namespace wg
