// Row-resident CSR GCN, second generation (BASELINE.json configs[3]: 4096 stations, kNN(k=8), hidden 128).
//
// Reference arithmetic as in gcn_sparse.cuh (src/step5_gcn_layer_model.py:13-23 twice, via
// src/step6_gcn_gru_combined_model.py:17,20), layer 2 evaluated as relu(A.(G1.W2) + b2).
//
// ncu on the first-generation row-resident kernel (profiles/r01_sparse_ncu_summary.md) showed the shared-memory
// pipe as the bound, not the FMA pipe: 1.59 G wavefronts per launch, half of them the warp-uniform LDS.128 weight
// reads of the dense phase (2 wavefronts each) and half the neighbour gathers (2.7 wavefronts per LDS: the 32 lanes
// of a warp read 32 random slab rows).  This kernel removes both:
//   * W1, W2, b1, b2 live in CONSTANT memory and reach FFMA2 as uniform-register operands (LDCU): the dense
//     phase issues no shared-memory instruction at all and a thread covers FOUR stations (two FFMA2 pairs),
//     68 TFLOP/s in isolation (scripts/probes/dense_probe.cu) against 52 with LDS.128 weights;
//   * the gathers follow a per-graph PLAN (csr_plan_kernel, a few tens of microseconds per call): for every
//     block of 32 consecutive stations the neighbour lists are re-ordered into steps in which the 32 lanes
//     read 32 DIFFERENT bank classes (col mod 32) — a greedy edge colouring of the lanes x classes bipartite
//     graph, longest list first.  Every gather LDS is one wavefront; idle slots are predicated off.  The plan
//     entry (col, val) of a step is one coalesced 8-byte load per lane.  Blocks the plan cannot hold
//     (a station with more than 64 neighbours, or more than kSqPlanCap steps) keep the CSR order.
// The order in which a station's neighbours are added is the plan's (a pure function of the graph), so results
// are deterministic and independent of batch size / chunking; they differ from the CSR-order sums of
// gcn_sparse_l1_kernel / gcn_sparse_l2_kernel by rounding only.
// Both passes write f-major rows ([F][S], coalesced from the thread = station mapping); fmajor_to_tiles_kernel
// re-lays U into the projection GEMM's K-major 128-row tiles.
#pragma once

#include "gcn_sparse.cuh"

namespace wg {

constexpr int kSqThreads = 512;
constexpr int kSqWarps = kSqThreads / 32;
constexpr int kSqStations = 4;     // stations per thread per sweep of pass 1 (two FFMA2 pairs)
constexpr int kSqPlanCap = 64;     // gather steps per block of 32 stations the plan can hold
constexpr int kSqMaxDeg = 64;      // neighbours per station the planner tracks (one bit each)
constexpr int kSqMaxFh = 256;      // hidden width the constant bank holds

struct SqWeights {
    float4 w1[kSqMaxFh * (kSpF / 4)];   // [fh][16]: W1[f][fh]
    float4 w2[kSqMaxFh * (kSpF / 4)];   // [fh][16]: W2[fh][fo]
    float b1[kSqMaxFh];
    float b2[kSpF];
};
__constant__ SqWeights c_sq;

// stage the weights in the constant-bank layout (plain global memory; copied to c_sq by the host)
__global__ void sq_pack_weights_kernel(const float* __restrict__ W1, const float* __restrict__ b1,
                                       const float* __restrict__ W2, const float* __restrict__ b2,
                                       SqWeights* __restrict__ dst, int Fi, int Fh, int Fo) {
    float* w1 = reinterpret_cast<float*>(dst->w1);
    float* w2 = reinterpret_cast<float*>(dst->w2);
    for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < kSqMaxFh * kSpF; e += gridDim.x * blockDim.x) {
        const int fh = e / kSpF, f = e % kSpF;
        w1[e] = (fh < Fh && f < Fi) ? W1[(size_t)f * Fh + fh] : 0.0f;
        w2[e] = (fh < Fh && f < Fo) ? W2[(size_t)fh * Fo + f] : 0.0f;
        if (f == 0) dst->b1[fh] = fh < Fh ? b1[fh] : 0.0f;
        if (e < kSpF) dst->b2[e] = e < Fo ? b2[e] : 0.0f;
    }
}

__host__ __device__ inline size_t sq_plan_bytes(int S) {
    const size_t wb = (size_t)ceil_div(S, 32);
    return round_up((int)wb, 4) * sizeof(int) + wb * kSqPlanCap * 32 * sizeof(int2);
}
__host__ __device__ inline size_t gcn_sparse_plan_smem_bytes(int S, int Fi, int Fo) {
    const int FS = Fi > Fo ? Fi : Fo;
    return (size_t)round_up(S * FS, 4) * 4 + 16;
}

// One warp per block of 32 stations.  steps[wb] = number of gather steps, or -1 when the block stays in CSR
// order; entries[(wb * cap + step) * 32 + lane] = (column, value bits) or (-1, 0) for an idle slot.
__global__ void __launch_bounds__(128) csr_plan_kernel(const int* __restrict__ rowptr, const int* __restrict__ colidx,
                                                       const float* __restrict__ vals, int S,
                                                       int* __restrict__ steps, int2* __restrict__ entries) {
    const int lane = threadIdx.x & 31;
    const int wb = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (wb * 32 >= S) return;
    const unsigned full = 0xffffffffu;
    const int s = wb * 32 + lane;
    const int e0 = s < S ? __ldg(rowptr + s) : 0;
    const int deg = s < S ? __ldg(rowptr + s + 1) - e0 : 0;
    if (__any_sync(full, deg > kSqMaxDeg)) {
        if (lane == 0) steps[wb] = -1;
        return;
    }
    unsigned long long done = 0;   // bit j: neighbour j of this lane's station is scheduled
    int rem = deg, nsteps = 0;
    int2* out = entries + (size_t)wb * kSqPlanCap * 32 + lane;
    while (__any_sync(full, rem > 0)) {
        if (nsteps == kSqPlanCap) {
            if (lane == 0) steps[wb] = -1;
            return;
        }
        unsigned taken = 0;   // bank classes used in this step (warp-uniform)
        int pick = -1;
        const int maxrem = __reduce_max_sync(full, rem);
        // round 0: only the lanes with the longest remaining list propose (they bound the step count)
        for (int round = 0; round < 2; ++round) {
            for (;;) {
                int cand = -1, c = 0;
                if (pick < 0 && rem > 0 && (round == 1 || rem == maxrem)) {
                    for (int j = 0; j < deg; ++j) {
                        if ((done >> j) & 1ull) continue;
                        const int cj = __ldg(colidx + e0 + j) & 31;
                        if (!((taken >> cj) & 1u)) { cand = j; c = cj; break; }
                    }
                }
                const unsigned act = __ballot_sync(full, cand >= 0);
                if (act == 0) break;
                bool won = false;
                if (cand >= 0) {
                    const unsigned peers = __match_any_sync(act, c);
                    won = lane == __ffs(peers) - 1;
                    if (won) pick = cand;
                }
                taken |= __reduce_or_sync(full, won ? (1u << c) : 0u);
            }
        }
        int2 e = make_int2(-1, 0);
        if (pick >= 0) {
            e.x = __ldg(colidx + e0 + pick);
            e.y = __float_as_int(__ldg(vals + e0 + pick));
            done |= 1ull << pick;
            --rem;
        }
        out[(size_t)nsteps * 32] = e;
        ++nsteps;
    }
    if (lane == 0) steps[wb] = nsteps;
}

// acc[f] = sum over the neighbours c of station (wb * 32 + lane) of a(s, c) * slab[c * cs + f * fs]
template <int FW, bool EXACT>
__device__ __forceinline__ void sq_gather(const float* __restrict__ slab, int cs, int fs, int F, int wb, int lane,
                                          int S, const int* __restrict__ steps, const int2* __restrict__ plan,
                                          const int* __restrict__ rowptr, const int* __restrict__ colidx,
                                          const float* __restrict__ vals, float (&acc)[FW]) {
#pragma unroll
    for (int f = 0; f < FW; ++f) acc[f] = 0.0f;
    const int n = __ldg(steps + wb);   // warp-uniform
    if (n >= 0) {
        const int2* pe = plan + (size_t)wb * kSqPlanCap * 32 + lane;
        constexpr int U = 4;           // steps in flight (the entries come from L2)
        int2 cur[U];
#pragma unroll
        for (int u = 0; u < U; ++u) cur[u] = u < n ? __ldg(pe + u * 32) : make_int2(-1, 0);
        for (int j0 = 0; j0 < n; j0 += U) {
            int2 nxt[U];
#pragma unroll
            for (int u = 0; u < U; ++u) nxt[u] = j0 + U + u < n ? __ldg(pe + (j0 + U + u) * 32) : make_int2(-1, 0);
#pragma unroll
            for (int u = 0; u < U; ++u) {
                if (cur[u].x >= 0) {
                    const float a = __int_as_float(cur[u].y);
                    const float* xs = slab + (size_t)cur[u].x * cs;
#pragma unroll
                    for (int f = 0; f < FW; ++f)
                        if (EXACT || f < F) acc[f] = fmaf(a, xs[(size_t)f * fs], acc[f]);
                }
            }
#pragma unroll
            for (int u = 0; u < U; ++u) cur[u] = nxt[u];
        }
    } else {
        const int s = wb * 32 + lane;
        if (s < S) {
            const int e1 = __ldg(rowptr + s + 1);
            for (int e = __ldg(rowptr + s); e < e1; ++e) {
                const float a = __ldg(vals + e);
                const float* xs = slab + (size_t)__ldg(colidx + e) * cs;
#pragma unroll
                for (int f = 0; f < FW; ++f)
                    if (EXACT || f < F) acc[f] = fmaf(a, xs[(size_t)f * fs], acc[f]);
            }
        }
    }
}

// FW: compile-time bound on F_in and F_out; EXACT: F_in == F_out == FW (no per-feature predicates)
template <int FW, bool EXACT>
__global__ void __launch_bounds__(kSqThreads, 1)
    gcn_sparse_plan_kernel(const float* __restrict__ X, const int* __restrict__ rowptr,
                           const int* __restrict__ colidx, const float* __restrict__ vals,
                           const int* __restrict__ steps, const int2* __restrict__ plan, float* __restrict__ Zscr,
                           float* __restrict__ U, long long R, int S, int Fi, int Fh, int Fo) {
    extern __shared__ __align__(16) float smem[];
    const int FS = Fi > Fo ? Fi : Fo;
    float* slab = smem;                                    // X row [S][Fi], then Z row [Fo][S]
    uint64_t* bar = reinterpret_cast<uint64_t*>(slab + round_up(S * FS, 4));
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (tid == 0) {
        mbar_init(bar, 1);
        fence_mbar_init();
    }
    __syncthreads();
    const int WB = ceil_div(S, 32);
    float* zrow = Zscr + (size_t)blockIdx.x * Fo * S;      // this CTA's scratch row, [Fo][S]
    const unsigned xbytes = (unsigned)((size_t)S * Fi * 4), zbytes = (unsigned)((size_t)S * Fo * 4);
    const bool z_bulk = (zbytes & 15) == 0 && (reinterpret_cast<uintptr_t>(zrow) & 15) == 0;
    unsigned phase = 0;

    for (long long r = blockIdx.x; r < R; r += gridDim.x) {
        // ---- the row's X slab: one bulk copy ----
        const float* xr = X + (size_t)r * S * Fi;
        if ((xbytes & 15) == 0 && (reinterpret_cast<uintptr_t>(xr) & 15) == 0) {
            if (tid == 0) {
                mbar_expect_tx(bar, xbytes);
                bulk_g2s(slab, xr, xbytes, bar);
            }
            mbar_wait(bar, phase);
            phase ^= 1;
        } else {
            for (int e = tid; e < S * Fi; e += kSqThreads) slab[e] = __ldg(xr + e);
            __syncthreads();
        }
        // ---- pass 1: Z = relu((A.X).W1 + b1).W2, four stations per thread ----
        for (int wb0 = warp; wb0 < WB; wb0 += kSqWarps * kSqStations) {
            float2 ag[FW][2];
#pragma unroll
            for (int i = 0; i < kSqStations; ++i) {
                const int wb = wb0 + i * kSqWarps;
                float acc[FW];
                if (wb < WB) {
                    sq_gather<FW, EXACT>(slab, Fi, 1, Fi, wb, lane, S, steps, plan, rowptr, colidx, vals, acc);
                } else {
#pragma unroll
                    for (int f = 0; f < FW; ++f) acc[f] = 0.0f;
                }
#pragma unroll
                for (int f = 0; f < FW; ++f) {
                    if (i & 1) ag[f][i >> 1].y = acc[f];
                    else ag[f][i >> 1].x = acc[f];
                }
            }
            float2 z[FW][2];
#pragma unroll
            for (int f = 0; f < FW; ++f) z[f][0] = z[f][1] = make_float2(0.0f, 0.0f);
#pragma unroll 2
            for (int fh = 0; fh < Fh; ++fh) {
                const float bb = c_sq.b1[fh];
                float2 h[2] = {make_float2(bb, bb), make_float2(bb, bb)};
#pragma unroll
                for (int v = 0; v < kSpF / 4; ++v) {
                    const float4 w = c_sq.w1[fh * (kSpF / 4) + v];
                    const float wv[4] = {w.x, w.y, w.z, w.w};
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        if (4 * v + j < FW) {
                            h[0] = __ffma2_rn(make_float2(wv[j], wv[j]), ag[4 * v + j][0], h[0]);
                            h[1] = __ffma2_rn(make_float2(wv[j], wv[j]), ag[4 * v + j][1], h[1]);
                        }
                    }
                }
#pragma unroll
                for (int q = 0; q < 2; ++q) {   // ReLU of layer 1
                    h[q].x = h[q].x < 0.0f ? 0.0f : h[q].x;
                    h[q].y = h[q].y < 0.0f ? 0.0f : h[q].y;
                }
#pragma unroll
                for (int v = 0; v < kSpF / 4; ++v) {
                    const float4 w = c_sq.w2[fh * (kSpF / 4) + v];
                    const float wv[4] = {w.x, w.y, w.z, w.w};
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        if (4 * v + j < FW) {
                            z[4 * v + j][0] = __ffma2_rn(make_float2(wv[j], wv[j]), h[0], z[4 * v + j][0]);
                            z[4 * v + j][1] = __ffma2_rn(make_float2(wv[j], wv[j]), h[1], z[4 * v + j][1]);
                        }
                    }
                }
            }
#pragma unroll
            for (int i = 0; i < kSqStations; ++i) {
                const int s = (wb0 + i * kSqWarps) * 32 + lane;
                if (s < S) {
#pragma unroll
                    for (int f = 0; f < FW; ++f)
                        if (EXACT || f < Fo) zrow[(size_t)f * S + s] = (i & 1) ? z[f][i >> 1].y : z[f][i >> 1].x;
                }
            }
        }
        // ---- Z row back over the slab (every thread is done with X; the scratch row is L2-hot) ----
        __threadfence();
        asm volatile("fence.proxy.async;\n" ::: "memory");   // generic-proxy stores -> visible to the bulk copy
        __syncthreads();
        if (z_bulk) {
            if (tid == 0) {
                mbar_expect_tx(bar, zbytes);
                bulk_g2s(slab, zrow, zbytes, bar);
            }
            mbar_wait(bar, phase);
            phase ^= 1;
        } else {
            for (int e = tid; e < S * Fo; e += kSqThreads) slab[e] = zrow[e];
            __syncthreads();
        }
        // ---- pass 2: U[f][s] = relu((A.Z)[s][f] + b2[f]) ----
        float* urow = U + (size_t)r * S * Fo;   // f-major [Fo][S]; fmajor_to_tiles_kernel re-lays it
        for (int wb = warp; wb < WB; wb += kSqWarps) {
            float acc[FW];
            sq_gather<FW, EXACT>(slab, 1, S, Fo, wb, lane, S, steps, plan, rowptr, colidx, vals, acc);
            const int s = wb * 32 + lane;
            if (s < S) {
#pragma unroll
                for (int f = 0; f < FW; ++f) {
                    if (EXACT || f < Fo) {
                        float v = acc[f] + c_sq.b2[f];
                        v = v < 0.0f ? 0.0f : v;
                        urow[(size_t)f * S + s] = v;
                    }
                }
            }
        }
        __syncthreads();   // the slab is free for the next row's bulk copy
    }
}

// Urow [R][F][S] (f-major rows) -> U tiles [ceil(R/128)][ldo][128] with column k = s * F + f (the flatten of
// src/step6_gcn_gru_combined_model.py:20), columns S*F .. ldo and rows beyond R zeroed.
// A CTA moves 32 rows x 32 stations: coalesced 128-byte reads along s, a [32][32 F + 1] shared-memory
// transpose, 128-byte writes along the rows.  grid = (ceil(S / 32), ceil(R_tiled / 32)), 256 threads.
__host__ __device__ inline size_t fmajor_to_tiles_smem_bytes(int F) { return (size_t)32 * (32 * F + 1) * 4; }

__global__ void __launch_bounds__(256) fmajor_to_tiles_kernel(const float* __restrict__ Urow, float* __restrict__ U,
                                                              long long R, int S, int F, int ldo) {
    extern __shared__ float t[];   // [32 rows][32 * F + 1]
    const int ld = 32 * F + 1;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;   // 8 warps
    const long long r0 = (long long)blockIdx.y * 32;
    const int s0 = blockIdx.x * 32;
    const int s = s0 + lane;
    for (int i = warp; i < 32; i += 8) {
        const long long r = r0 + i;
        const float* src = Urow + (size_t)r * S * F + s;
        for (int f = 0; f < F; ++f) t[i * ld + lane * F + f] = (r < R && s < S) ? __ldg(src + (size_t)f * S) : 0.0f;
    }
    __syncthreads();
    float* dst = U + (size_t)(r0 / kSpThreads) * ldo * kSpThreads + (r0 % kSpThreads) + lane;
    const int ncol = (S - s0 < 32 ? S - s0 : 32) * F;
    for (int c = warp; c < ncol; c += 8) dst[(size_t)(s0 * F + c) * kSpThreads] = t[lane * ld + c];
    if (blockIdx.x == gridDim.x - 1)   // K padding
        for (int k = S * F + warp; k < ldo; k += 8) dst[(size_t)k * kSpThreads] = 0.0f;
}

}  // namespace wg
