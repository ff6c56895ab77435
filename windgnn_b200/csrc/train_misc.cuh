// Loss and optimiser kernels of the training step.
//
// Reference: `lossFunction = nn.MSELoss()` (src/main.py:49), `loss = lossFunction(outputs, batch_y)`
// (:72), `torch.optim.Adam(model.parameters(), lr=learning_rate)` (:52), `optimizer.step()` (:77).
#pragma once

#include "wg_common.cuh"

namespace wg {

constexpr int kMseThreads = 256;

// Where the targets y[e] of mse_grad_kernel come from: a buffer laid out as out ...
struct LabelBuffer {
    const float* __restrict__ y;
    __device__ float operator()(long long e) const { return y[e]; }
};

// ... or the table itself, for out [N][L][K*S] over the windows table[starts[n] : starts[n] + L]: the target of
// (n, l, k*S + s) is the label feature k + 1 rows after the window's row l, as wg_make_windows_f32 builds y:
// y[n][l][k*S + s] = table[starts[n] + l + 1 + k][s][label_f].
struct LabelTable {
    const float* __restrict__ table;
    const long long* __restrict__ starts;   // device, [N]
    int L, S, F, label_f, KS;               // KS = K * S: the width of out
    __device__ float operator()(long long e) const {
        const long long row = e / KS;        // n * L + l
        const int c = (int)(e - row * KS);
        const long long n = row / L;
        const int l = (int)(row - n * L);
        const int k = c / S, s = c - k * S;
        return table[((starts[n] + l + 1 + k) * S + s) * F + label_f];
    }
};

// d_out = 2 (out - y) / n ; partial[cta] = sum of (out - y)^2 over the CTA's grid-stride slice.
template <typename Labels>
__global__ void __launch_bounds__(kMseThreads)
    mse_grad_kernel(const float* __restrict__ out, Labels y, float* __restrict__ d_out,
                    double* __restrict__ partial, long long n, float scale) {
    __shared__ double red[kMseThreads / 32];
    double s = 0.0;
    for (long long e = (long long)blockIdx.x * kMseThreads + threadIdx.x; e < n;
         e += (long long)gridDim.x * kMseThreads) {
        const float d = out[e] - y(e);
        if (d_out) d_out[e] = d * scale;
        s += (double)d * (double)d;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x == 0) {
        double t = 0.0;
        for (int w = 0; w < kMseThreads / 32; ++w) t += red[w];
        partial[blockIdx.x] = t;
    }
}

__global__ void mse_finish_kernel(const double* __restrict__ partial, int nparts, long long n,
                                  float* __restrict__ loss) {
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        double t = 0.0;
        for (int i = 0; i < nparts; ++i) t += partial[i];
        *loss = (float)(t / (double)n);
    }
}

// torch.optim.Adam (no weight decay, no amsgrad), one fused pass over a flat parameter buffer:
//   g = grad * grad_scale ; m = b1 m + (1 - b1) g ; v = b2 v + (1 - b2) g^2
//   p -= (lr / bc1) * m / (sqrt(v) / sqrt(bc2) + eps)          bc = 1 - beta^step (host, fp64)
__global__ void adam_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m,
                            float* __restrict__ v, long long n, float grad_scale, float beta1, float beta2,
                            float omb1, float omb2, float step_size, float sqrt_bc2, float eps) {
    for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < n;
         e += (long long)gridDim.x * blockDim.x) {
        const float gg = g[e] * grad_scale;
        const float mm = beta1 * m[e] + omb1 * gg;   // omb = 1 - beta, rounded once from fp64 like torch
        const float vv = beta2 * v[e] + omb2 * gg * gg;
        m[e] = mm;
        v[e] = vv;
        const float denom = sqrtf(vv) / sqrt_bc2 + eps;
        p[e] -= step_size * (mm / denom);
    }
}

}  // namespace wg
