// C-ABI of the WindGNN B200 forward path (see include/windgnn_b200.h).
// Host side: argument validation, workspace planning, kernel dispatch.  No torch, no state.

#include "../../include/windgnn_b200.h"

#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <vector>

#include "gcn.cuh"
#include "gcn_bwd.cuh"
#include "gcn_bwd_rows.cuh"
#include "gcn_rows.cuh"
#include "gcn_sparse.cuh"
#include "gcn_sparse_plan.cuh"
#include "gemm_kb.cuh"
#include "gru_bwd.cuh"
#include "inproj.cuh"
#include "inproj_tc2.cuh"
#include "recur.cuh"
#include "recur_tc.cuh"
#include "recur_unit.cuh"
#include "sgemm.cuh"
#include "train_misc.cuh"
#include "wg_common.cuh"

namespace {

thread_local char g_err[512] = "";

int fail(int code, const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return code;
}

#define WG_CUDA(expr)                                                                          \
    do {                                                                                       \
        cudaError_t e_ = (expr);                                                               \
        if (e_ != cudaSuccess)                                                                 \
            return fail(WG_ERR_CUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(e_),   \
                        __FILE__, __LINE__);                                                   \
    } while (0)

// RAII device switch (the caller's current device is restored on return).
struct DeviceGuard {
    int prev = -1;
    cudaError_t err = cudaSuccess;
    explicit DeviceGuard(int dev) {
        err = cudaGetDevice(&prev);
        if (err == cudaSuccess && prev != dev) err = cudaSetDevice(dev);
    }
    ~DeviceGuard() {
        int cur = -1;
        if (prev >= 0 && cudaGetDevice(&cur) == cudaSuccess && cur != prev) cudaSetDevice(prev);
    }
};

constexpr size_t kAlign = 256;
size_t align_up(size_t v) { return (v + kAlign - 1) / kAlign * kAlign; }

enum GcnKind { kGcnRows, kGcn13x7, kGcn13x4, kGcn16x4, kGcnSparsePlan, kGcnSparseLanes };
enum RecurKind { kRecurTc, kRecurUnit, kRecurWide };

// Everything the stages need to agree on: shapes, workspace layout, the kernel of every stage and the launch geometry
// that depends only on the shape.
struct Plan {
    int T, S, Fi, Fh, Fo, H;
    long long chunk;
    int I, G;      // S*Fo, 3H
    int IP;        // K of the projection GEMM: I rounded up to 16
    int NPB;       // rows of packed w_ih: G rounded up to 64
    int GP;        // leading dim of GI: G rounded up to 8
    int KP;        // K of the recurrent GEMM: H rounded up to 4
    int NPR;       // columns of packed w_hh^T: G rounded up to 80 (one warp's column block)
    int n_bias;    // packed bias entries: one per packed w_ih row of either projection, at least 512
    bool sparse;   // CSR graph path: adds the Z scratch of the sparse GCN kernels
    GcnKind gcn;
    size_t gcn_smem;   // dynamic shared memory of the GCN kernel (the lane kernels: of gcn_sparse_l1_kernel)
    int gcn_rb;        // gcn_kernel: rows per block
    int gcn_threads;   // gcn_rows_kernel: block size
    size_t off_sqw, off_sqsteps, off_sqpairs;   // gcn_sparse_plan_kernel: constant-bank weights, gather plan (steps, pairs)
    bool tc;       // tensor-core input projection (inproj_tc2.cuh): w_ih packed as fp16 hi + lo
    wg::Tc2Shape tc2;
    RecurKind recur;   // small chunks may run gru_recur_regw_kernel instead (launch_recur)
    bool regw;         // the contraction length fits gru_recur_regw_kernel, which then takes small chunks
    bool whu;          // W_hh^T packed for gru_recur_unit_kernel: whenever that kernel serves H, on every path
    int ru_wpg, ru_ht; // gru_recur_unit_kernel: warps per group, compile-time H (102 or 21) or 0
    int ru_rmax;       // gru_recur_unit_kernel: the largest R (sequences per group) whose shared memory fits
    int rc_ts;         // gru_recur_kernel: steps of h staged per bulk store (0: every step stored directly)
    size_t rc_smem;    //                   its dynamic shared memory
    size_t off_wp, off_bias, off_wht, off_whu, off_bhn, off_u, off_gi, off_z, total;
    size_t off_whh_hi, off_whh_lo;   // kRecurTc: W_hh packed as fp16 hi + lo
    // tensor path: the inverse power-of-two scales of the split operands (tc_scale_exp), per packed W_ih row (tc2.NP)
    // then per packed W_hh row ([3][128], h's scale folded in); the largest element of every U row (float bits)
    size_t off_tcs, off_umax;
};

long long default_chunk(long long B, size_t bytes_per_seq) {
    long long c = (long long)wg::kNumSMs * wg::kRcBT;  // 4736 sequences: one wave of the recurrence
    // keep the per-chunk scratch under ~6 GB for the scaled shapes (whole 32-sequence CTAs)
    const size_t cap = (size_t)6 << 30;
    if ((size_t)c * bytes_per_seq > cap) {
        c = (long long)(cap / bytes_per_seq) / wg::kRcBT * wg::kRcBT;
        if (c < wg::kRcBT) c = wg::kRcBT;
    }
    return B < c ? (B < 1 ? 1 : B) : c;
}

// gcn_kernel instantiation for the feature widths (the single layer passes F_out as F_hid): the exact 13-wide one
// with 7 or 4 stations per thread, whichever pads S less (ties: 7), else the generic 16-wide one, which
// dense_gcn_geometry rejects for widths above 16
GcnKind dense_gcn_kind(int S, int Fi, int Fh, int Fo) {
    if (Fi == 13 && Fh == 13 && Fo == 13) return wg::ceil_div(S, 7) * 7 <= wg::ceil_div(S, 4) * 4 ? kGcn13x7 : kGcn13x4;
    return kGcn16x4;
}

// Rows per block and dynamic shared memory of gcn_kernel instantiation k, or the reason why it cannot serve the shape
// (the single layer passes F_out as F_hid).
int dense_gcn_geometry(GcnKind k, int S, int Fi, int Fh, int Fo, int& RB, size_t& smem) {
    const int Fmax = Fi > Fh ? (Fi > Fo ? Fi : Fo) : (Fh > Fo ? Fh : Fo);
    if (Fmax > 16) return fail(WG_ERR_UNSUPPORTED, "GCN feature width %d > 16 is not built into the dense kernel", Fmax);
    const int NSG = wg::ceil_div(S, k == kGcn13x7 ? 7 : 4);
    if (NSG > wg::kGcnThreads)
        return fail(WG_ERR_UNSUPPORTED, "S=%d too large for the dense GCN kernel", S);
    auto smem_of = [&](int rb) {
        const size_t floats = k == kGcn13x7   ? wg::gcn_smem_floats<13, 7>(S, Fmax, rb)
                              : k == kGcn13x4 ? wg::gcn_smem_floats<13, 4>(S, Fmax, rb)
                                              : wg::gcn_smem_floats<16, 4>(S, Fmax, rb);
        return floats * 4;
    };
    // rows per block: as many as the 128 threads cover, rounded down so that whole blocks are
    // 16-byte multiples (bulk-copyable): RB * S * Fi % 4 == 0
    RB = wg::kGcnThreads / NSG;
    const int in_cols = S * Fi;
    const int need = (in_cols % 4 == 0) ? 1 : (in_cols % 2 == 0 ? 2 : 4);
    if (RB > need) RB -= RB % need;
    smem = smem_of(RB);
    // aim for >= 3 resident CTAs per SM when the slabs allow it
    while (smem > (size_t)wg::kMaxSmemOptin / 3 && RB > 2 * need && RB > 8) {
        RB -= need > (RB + 7) / 8 ? need : (RB + 7) / 8 / need * need;
        smem = smem_of(RB);
    }
    while (smem > (size_t)wg::kMaxSmemOptin && RB > 1) {
        RB = RB / 2;
        smem = smem_of(RB);
    }
    if (smem > (size_t)wg::kMaxSmemOptin)
        return fail(WG_ERR_UNSUPPORTED, "dense GCN needs %zu B of shared memory (S=%d); use the sparse path", smem, S);
    return WG_OK;
}

// Testing knob: WG_FORCE_LEGACY=1 runs the fused two-layer GCN on gcn_kernel where gcn_rows_kernel would run, so
// that the tests can compare the two (they are bit-identical).  It selects nothing else.
bool force_legacy() {
    const char* e = getenv("WG_FORCE_LEGACY");
    return e && e[0] == '1';
}

// Table rows per GCN + projection piece of a forecast: a chunk of windows' worth, at most the table.
long long forecast_piece_rows(const Plan& p, long long Ttot) {
    const long long r = p.chunk * p.T;
    return r < Ttot ? r : Ttot;
}

// The shapes, the kernel of every stage and the workspace layout (plan_launch completes the plan).
// table_rows > 0 (the forecast): GI holds that many rows, and the GCN / projection scratch (U, Z) pieces of
// forecast_piece_rows rows instead of a chunk's.
int plan_layout(Plan& p, long long B, int T, int S, int Fi, int Fh, int Fo, int H, long long chunk, bool sparse,
                int flags, long long table_rows = 0) {
    if (B < 0 || T <= 0 || S <= 0 || Fi <= 0 || Fh <= 0 || Fo <= 0 || H <= 0 || chunk < 0)
        return fail(WG_ERR_BAD_ARG, "non-positive dimension (B=%lld T=%d S=%d F=%d/%d/%d H=%d chunk=%lld)",
                    B, T, S, Fi, Fh, Fo, H, chunk);
    if ((long long)S * Fo > (1 << 20) || H > (1 << 15))
        return fail(WG_ERR_UNSUPPORTED, "dimension too large (S*F_out=%lld, H=%d)", (long long)S * Fo, H);
    p.T = T; p.S = S; p.Fi = Fi; p.Fh = Fh; p.Fo = Fo; p.H = H;
    p.sparse = sparse;
    if (flags & ~WG_FLAG_TENSOR_CORES) return fail(WG_ERR_BAD_ARG, "unknown flags 0x%x", flags);
    p.I = S * Fo;
    p.G = 3 * H;
    // tensor-core projection (inproj_tc2.cuh): when two accumulators of the gate slice fit TMEM; it consumes the
    // same fp32 U tiles (dense or CSR graph path alike), K padded to its 32-k stage
    p.tc2 = wg::tc2_shape(p.G, p.I);
    p.tc = (flags & WG_FLAG_TENSOR_CORES) != 0;
    if (p.tc && !p.tc2.ok)
        return fail(WG_ERR_UNSUPPORTED, "tensor-core projection: unsupported gate width 3H = %d", p.G);
    p.IP = p.tc ? p.tc2.KP : wg::round_up(p.I, wg::kIpBK);
    p.NPB = wg::round_up(p.G, wg::kIpBN);
    p.GP = wg::round_up(p.G, 8);   // GI rows 32-byte aligned (256-bit stores in the tensor-path projection)
    p.KP = wg::round_up(H, 4);
    p.NPR = wg::recur_np(p.G);
    {
        const size_t per_seq = (size_t)T * ((size_t)p.IP + p.GP + (sparse ? (size_t)S * Fo : 0)) * 4;
        p.chunk = chunk > 0 ? chunk : default_chunk(B, per_seq);
        if (p.chunk > B && B > 0) p.chunk = B;
    }
    // GCN: the CSR graph on the second-generation kernel when its weights fit the constant bank and its slab fits
    // shared memory; the dense graph on gcn_rows_kernel when that kernel serves the shape
    if (sparse)
        p.gcn = Fi <= wg::kSpF && Fo <= wg::kSpF && Fh <= wg::kSqMaxFh &&
                        wg::gcn_sparse_plan_smem_bytes(S, Fi, Fo) <= (size_t)wg::kMaxSmemOptin
                    ? kGcnSparsePlan : kGcnSparseLanes;
    else if (wg::gcn_rows_applies(S, Fi, Fh, Fo) && wg::gcn_rows_smem_floats(S) * 4 <= (size_t)wg::kMaxSmemOptin &&
             !force_legacy())
        p.gcn = kGcnRows;
    else
        p.gcn = dense_gcn_kind(S, Fi, Fh, Fo);
    p.whu = wg::recur_u_applies(H);
    if (p.tc && wg::recur_tc_applies(H) && wg::recur_tc_smem_bytes(H) <= (size_t)wg::kMaxSmemOptin)
        p.recur = kRecurTc;
    else if (p.whu && wg::recur_u_smem_floats(H, wg::kRuMinR) * 4 <= (size_t)wg::kMaxSmemOptin)
        p.recur = kRecurUnit;
    else
        p.recur = kRecurWide;
    // small chunks (the reference's batch-1 calls, small shards) of the shipped models: W_hh in registers for their
    // contraction lengths (H = 102 -> 104, H = 21 -> 24), 4 sequences per CTA, bit-identical results
    p.regw = (p.KP == 104 || p.KP == 24) && p.NPR <= wg::kRwThreads &&
             wg::recur_regw_smem_floats(p.KP, p.NPR, p.GP) * 4 <= (size_t)wg::kMaxSmemOptin;
    // H = 102 and H = 21 (the shipped 34- and 7-station models, 3 x S) have their own instantiations with
    // compile-time strides; for the odd H = 21 this also folds the alignment branches of the gate phase
    // (ncu: 55 % of the generic kernel's samples sat in that branchy code at H = 21)
    p.ru_wpg = wg::recur_u_wpg(H);
    p.ru_ht = H == 102 || H == 21 ? H : 0;
    size_t o = 0;
    const int wrows = p.tc && p.tc2.NP > p.NPB ? p.tc2.NP : p.NPB;
    p.n_bias = wrows > 512 ? wrows : 512;
    // packed w_ih: fp32 [N/64][K][64] for the FFMA GEMM, or fp16 hi + lo stage blocks for the tensor cores
    p.off_wp = o;   o = align_up(o + (p.tc ? wg::tc2_w_halves(p.tc2) * 2 : (size_t)p.NPB * p.IP * 4));
    p.off_bias = o; o = align_up(o + (size_t)p.n_bias * 4);
    p.off_tcs = o;  if (p.tc) o = align_up(o + ((size_t)p.tc2.NP + 3 * 128) * 4);
    p.off_wht = o;  o = align_up(o + (size_t)p.KP * p.NPR * 4);
    p.off_whu = o;  // [k][gate][unit] (recur_unit.cuh)
    if (p.whu) o = align_up(o + (size_t)p.KP * 3 * wg::recur_u_hp2(H) * 4);
    p.off_bhn = o;  o = align_up(o + (size_t)p.KP * 4);
    const bool tc_recur = p.recur == kRecurTc;
    p.off_whh_hi = o; if (tc_recur) o = align_up(o + wg::recur_tc_w_halves(H) * 2);
    p.off_whh_lo = o; if (tc_recur) o = align_up(o + wg::recur_tc_w_halves(H) * 2);
    const size_t rows = table_rows > 0 ? (size_t)forecast_piece_rows(p, table_rows) : (size_t)p.chunk * T;
    const size_t rows_tiled = (rows + wg::kUTileRows - 1) / wg::kUTileRows * wg::kUTileRows;
    p.off_u = o;    o = align_up(o + rows_tiled * p.IP * 4);  // K-major 128-row tiles
    p.off_umax = o; if (p.tc) o = align_up(o + rows_tiled * 4);
    // GI: the tensor-core recurrence reads whole groups of kRtSeqs sequences (rows past the batch are scratch)
    const size_t rows_gi =
        table_rows > 0 ? (size_t)table_rows : (size_t)((p.chunk + wg::kRtSeqs - 1) / wg::kRtSeqs * wg::kRtSeqs) * T;
    p.off_gi = o;   o = align_up(o + rows_gi * p.GP * 4);
    // sparse path scratch: row-major U (rows x S*Fo) + one [Fo][S] row per resident CTA
    p.off_z = o;    if (sparse) o = align_up(o + (rows + wg::kNumSMs) * (size_t)S * Fo * 4);
    // second-generation CSR kernel: weights staged for the constant bank + the gather plan (one step count per
    // 32-station block, padded to 4, then the gather pairs)
    const bool sq = p.gcn == kGcnSparsePlan;
    p.off_sqw = o;     if (sq) o = align_up(o + sizeof(wg::SqWeights));
    p.off_sqsteps = o;
    p.off_sqpairs = o + (size_t)wg::round_up(wg::ceil_div(S, 32), 4) * sizeof(int);
    if (sq) o = align_up(o + wg::sq_plan_bytes(S));
    p.total = o;
    return WG_OK;
}

// The launch geometry of the plan's kernels that depends only on the shape, and their limits, checked in stage order
// (GCN, projection, recurrence).  A shape that passes runs every chunk: the checks that grow with the rows take the
// plan's full chunk, the largest a call runs.
int plan_launch(Plan& p) {
    const long long rows = p.chunk * p.T;
    switch (p.gcn) {
    case kGcnRows:
        p.gcn_smem = wg::gcn_rows_smem_floats(p.S) * 4;
        p.gcn_threads = wg::gcn_rows_warps(p.S) * 32;
        break;
    case kGcnSparsePlan: {
        p.gcn_smem = wg::gcn_sparse_plan_smem_bytes(p.S, p.Fi, p.Fo);
        // fmajor_to_tiles_kernel: one grid row per 32 rows of whole tiles
        const long long rt = (rows + wg::kSpThreads - 1) / wg::kSpThreads * wg::kSpThreads;
        if (rt / 32 > 65535) return fail(WG_ERR_UNSUPPORTED, "sparse GCN: chunk of %lld rows too large", rows);
        break;
    }
    case kGcnSparseLanes:
        if (p.Fi > wg::kSpF || p.Fo > wg::kSpF)
            return fail(WG_ERR_UNSUPPORTED, "sparse GCN: F_in / F_out must be <= %d (got %d / %d)", wg::kSpF, p.Fi, p.Fo);
        p.gcn_smem = ((size_t)2 * p.Fh * wg::kSpF + p.Fh) * 4;
        if (p.gcn_smem > (size_t)wg::kMaxSmemOptin)
            return fail(WG_ERR_UNSUPPORTED, "sparse GCN: hidden width %d too large", p.Fh);
        break;
    default: {
        const int rc = dense_gcn_geometry(p.gcn, p.S, p.Fi, p.Fh, p.Fo, p.gcn_rb, p.gcn_smem);
        if (rc) return rc;
    }
    }
    if (!p.tc && (rows + wg::kIpBM - 1) / wg::kIpBM * (p.NPB / wg::kIpBN) > 0x7fffffffLL)
        return fail(WG_ERR_UNSUPPORTED, "projection grid too large");
    if (p.recur == kRecurUnit) {
        p.ru_rmax = wg::kRuMaxR;
        while (p.ru_rmax > wg::kRuMinR && wg::recur_u_smem_floats(p.H, p.ru_rmax) * 4 > (size_t)wg::kMaxSmemOptin)
            --p.ru_rmax;
    } else if (p.recur == kRecurWide) {
        // stage h in shared memory for bulk stores when it fits, else store every step directly
        p.rc_ts = wg::recur_stage_steps(p.H);
        p.rc_smem = wg::recur_smem_floats(p.KP, p.GP, p.H, p.rc_ts) * 4;
        if (p.rc_smem > (size_t)wg::kMaxSmemOptin) {
            p.rc_ts = 0;
            p.rc_smem = wg::recur_smem_floats(p.KP, p.GP) * 4;
        }
        if (p.rc_smem > (size_t)wg::kMaxSmemOptin)
            return fail(WG_ERR_UNSUPPORTED, "GRU hidden size %d: state does not fit shared memory", p.H);
    }
    return WG_OK;
}

// The whole plan of a forward: every shape it rejects is rejected here, before any launch.
int make_plan(Plan& p, long long B, int T, int S, int Fi, int Fh, int Fo, int H, long long chunk,
              bool sparse = false, int flags = 0) {
    const int rc = plan_layout(p, B, T, S, Fi, Fh, Fo, H, chunk, sparse, flags);
    return rc ? rc : plan_launch(p);
}

int check_ws(const void* ws, size_t bytes, size_t need) {
    if (!ws) return fail(WG_ERR_WORKSPACE, "workspace is NULL (need %zu bytes)", need);
    if (reinterpret_cast<uintptr_t>(ws) % kAlign)
        return fail(WG_ERR_WORKSPACE, "workspace must be %zu-byte aligned", kAlign);
    if (bytes < need)
        return fail(WG_ERR_WORKSPACE, "workspace too small: %zu bytes given, %zu needed", bytes, need);
    return WG_OK;
}

template <typename T>
T* ws_ptr(void* ws, size_t off) { return reinterpret_cast<T*>(static_cast<char*>(ws) + off); }

// ---------------------------------------------------------------------------------------------
// parameter packing (tiny; runs every call so the library stays stateless)
// ---------------------------------------------------------------------------------------------
// pack_wih: 0 when the tensor path packs w_ih itself (pack_wih_tc2_kernel)
__global__ void pack_params_kernel(const float* __restrict__ w_ih, const float* __restrict__ w_hh,
                                   const float* __restrict__ b_ih, const float* __restrict__ b_hh,
                                   float* __restrict__ wp, float* __restrict__ bias,
                                   float* __restrict__ wht, float* __restrict__ whu, float* __restrict__ bhn, int I,
                                   int H, int IP, int NPB, int KP, int NPR, int pack_wih, int n_bias) {
    const int G = 3 * H;
    const long long n_wp = pack_wih ? (long long)NPB * IP : 0;
    const long long n_wht = (long long)KP * NPR;
    const long long stride = (long long)gridDim.x * blockDim.x;
    const long long t0 = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    for (long long e = t0; e < n_wp; e += stride) {
        // destination layout [n / 64][k][n % 64] (K-major 64-column tiles, see inproj.cuh)
        const int nl = (int)(e % wg::kIpBN);
        const long long r = e / wg::kIpBN;
        const int k = (int)(r % IP), n = (int)(r / IP) * wg::kIpBN + nl;
        wp[e] = (n < G && k < I) ? w_ih[(size_t)n * I + k] : 0.0f;
    }
    for (long long e = t0; e < n_wht; e += stride) {
        const int k = (int)(e / NPR), n = (int)(e % NPR);
        wht[e] = (k < H && n < G) ? w_hh[(size_t)n * H + k] : 0.0f;
    }
    if (whu != nullptr) {   // W_hh^T for the unit-tiled recurrence: whu[k][g][j] = w_hh[g*H + j][k]
        const int HP2 = wg::recur_u_hp2(H);
        const long long n_whu = (long long)KP * 3 * HP2;
        for (long long e = t0; e < n_whu; e += stride) {
            const int j = (int)(e % HP2);
            const long long r = e / HP2;
            const int g = (int)(r % 3), k = (int)(r / 3);
            whu[e] = (k < H && j < H) ? w_hh[((size_t)g * H + j) * H + k] : 0.0f;
        }
    }
    for (long long e = t0; e < n_bias; e += stride) {
        float v = 0.0f;
        if (e < G) v = b_ih[e] + (e < 2 * H ? b_hh[e] : 0.0f);  // r,z: both biases; n: b_in only
        bias[e] = v;
    }
    for (long long e = t0; e < KP; e += stride) bhn[e] = e < H ? b_hh[2 * H + e] : 0.0f;
}

// ---------------------------------------------------------------------------------------------
// stage launchers
// ---------------------------------------------------------------------------------------------
// RB, smem: from dense_gcn_geometry
template <int FP, int SG, bool EXACT, int LAYERS, bool TILED>
int launch_gcn_t(const float* X, const float* adj, const float* W1, const float* b1, const float* W2,
                 const float* b2, float* out, long long R, int S, int Fi, int Fh, int Fo, int ldo, int RB, size_t smem,
                 cudaStream_t st) {
    auto kern = wg::gcn_kernel<FP, SG, EXACT, LAYERS, TILED>;
    WG_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int per_sm = 0;
    WG_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, wg::kGcnThreads, smem));
    if (per_sm < 1) per_sm = 1;
    const long long nblocks = (R + RB - 1) / RB;
    long long grid = (long long)wg::kNumSMs * per_sm;
    if (grid > nblocks) grid = nblocks;
    if (grid < 1) return WG_OK;
    kern<<<(unsigned)grid, wg::kGcnThreads, smem, st>>>(X, adj, W1, b1, W2, b2, out, R, S, Fi, Fh, Fo, ldo, RB);
    WG_CUDA(cudaGetLastError());
    return WG_OK;
}

template <int LAYERS, bool TILED>
int launch_gcn_dense(GcnKind k, int RB, size_t smem, const float* X, const float* adj, const float* W1,
                     const float* b1, const float* W2, const float* b2, float* out, long long R, int S, int Fi, int Fh,
                     int Fo, int ldo, cudaStream_t st) {
#define WG_GCN(FP, SG, EX) \
    launch_gcn_t<FP, SG, EX, LAYERS, TILED>(X, adj, W1, b1, W2, b2, out, R, S, Fi, Fh, Fo, ldo, RB, smem, st)
    if (k == kGcn13x7) return WG_GCN(13, 7, true);
    if (k == kGcn13x4) return WG_GCN(13, 4, true);
    return WG_GCN(16, 4, false);
#undef WG_GCN
}

// second-generation fused two-layer kernel (gcn_rows.cuh): lane = row, output straight into the tiles
// (the tensor path's instantiation also records the U row maxima in umax, cleared here)
int launch_gcn_rows(const Plan& p, const float* X, const float* adj, const float* W1, const float* b1,
                    const float* W2, const float* b2, float* out, int* umax, long long R, cudaStream_t st) {
    auto kern = p.tc ? wg::gcn_rows_kernel<true> : wg::gcn_rows_kernel<false>;
    if (p.tc) WG_CUDA(cudaMemsetAsync(umax, 0, (size_t)(R + wg::kT2BM - 1) / wg::kT2BM * wg::kT2BM * 4, st));
    WG_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)p.gcn_smem));
    int per_sm = 0;
    WG_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, p.gcn_threads, p.gcn_smem));
    if (per_sm < 1) per_sm = 1;
    const long long nblocks = (R + wg::kGrRows - 1) / wg::kGrRows;
    long long grid = (long long)wg::kNumSMs * per_sm;
    if (grid > nblocks) grid = nblocks;
    if (grid < 1) return WG_OK;
    kern<<<(unsigned)grid, p.gcn_threads, p.gcn_smem, st>>>(X, adj, W1, b1, W2, b2, out, R, p.S, p.IP, umax);
    WG_CUDA(cudaGetLastError());
    return WG_OK;
}

// The graph of a forward: the dense adjacency, or the CSR arrays when Plan::sparse.
struct Graph {
    const float* adj;
    const int* rowptr;
    const int* colidx;
    const float* vals;
};

int launch_gcn_sparse(const Plan& p, void* ws, const Graph& g, const float* x, const float* w1, const float* b1,
                      const float* w2, const float* b2, long long rows, cudaStream_t st) {
    if (rows < 1) return WG_OK;
    if (p.gcn == kGcnSparsePlan) {   // constant-bank weights + gather plan (prepare_sparse ran)
        const bool narrow = p.Fi <= 13 && p.Fo <= 13, exact = p.Fi == 13 && p.Fo == 13;
        auto kern = exact ? wg::gcn_sparse_plan_kernel<13, true>
                          : narrow ? wg::gcn_sparse_plan_kernel<13, false> : wg::gcn_sparse_plan_kernel<16, false>;
        WG_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)p.gcn_smem));
        const unsigned grid = (unsigned)(rows < wg::kNumSMs ? rows : wg::kNumSMs);
        float* urow = ws_ptr<float>(ws, p.off_z);   // [rows][Fo][S] f-major U, then gridDim per-CTA Z rows
        float* zscr = urow + (size_t)rows * p.S * p.Fo;
        kern<<<grid, wg::kSqThreads, p.gcn_smem, st>>>(x, g.rowptr, g.colidx, g.vals, ws_ptr<int>(ws, p.off_sqsteps),
                                                       ws_ptr<int2>(ws, p.off_sqpairs), zscr, urow, rows, p.S, p.Fi,
                                                       p.Fh, p.Fo);
        WG_CUDA(cudaGetLastError());
        const long long rt = (rows + wg::kSpThreads - 1) / wg::kSpThreads * wg::kSpThreads;  // whole tiles (zero rows)
        const dim3 tg((unsigned)((p.S + 31) / 32), (unsigned)(rt / 32));
        const size_t tsmem = wg::fmajor_to_tiles_smem_bytes(p.Fo);
        WG_CUDA(cudaFuncSetAttribute(wg::fmajor_to_tiles_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tsmem));
        wg::fmajor_to_tiles_kernel<<<tg, 256, tsmem, st>>>(urow, ws_ptr<float>(ws, p.off_u), rows, p.S, p.Fo, p.IP);
        WG_CUDA(cudaGetLastError());
        return WG_OK;
    }
    // gcn_sparse_plan_kernel does not apply (hidden width above its constant bank, or a slab too large for
    // shared memory): the two lane = row kernels
    const long long tiles = (rows + wg::kSpThreads - 1) / wg::kSpThreads;
    // split the stations so that the grid fills the machine a few times over
    int chunks = (int)((4LL * wg::kNumSMs * 4 + tiles - 1) / tiles);
    if (chunks < 1) chunks = 1;
    if (chunks > p.S) chunks = p.S;
    const int s_chunk = (p.S + chunks - 1) / chunks;
    const dim3 grid((unsigned)tiles, (unsigned)((p.S + s_chunk - 1) / s_chunk));
    WG_CUDA(cudaFuncSetAttribute(wg::gcn_sparse_l1_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                 (int)p.gcn_smem));
    wg::gcn_sparse_l1_kernel<<<grid, wg::kSpThreads, p.gcn_smem, st>>>(x, g.rowptr, g.colidx, g.vals, w1, b1, w2,
                                                                       ws_ptr<float>(ws, p.off_z), rows, p.S, p.Fi,
                                                                       p.Fh, p.Fo, s_chunk);
    WG_CUDA(cudaGetLastError());
    wg::gcn_sparse_l2_kernel<<<grid, wg::kSpThreads, 0, st>>>(ws_ptr<float>(ws, p.off_z), g.rowptr, g.colidx, g.vals,
                                                             b2, ws_ptr<float>(ws, p.off_u), rows, p.S, p.Fo, p.IP,
                                                             s_chunk);
    WG_CUDA(cudaGetLastError());
    return WG_OK;
}

// The plan's two-layer GCN over `rows` = sequences x steps, into the projection's U tiles; on the tensor path also
// the largest element of every U row, which sets the row's scale in the projection (gcn_rows_kernel records it while
// it writes U, u_rowmax_kernel reads it back after the other GCN kernels).
int launch_gcn(const Plan& p, void* ws, const Graph& g, const float* x, const float* w1, const float* b1,
               const float* w2, const float* b2, long long rows, cudaStream_t st) {
    float* u = ws_ptr<float>(ws, p.off_u);
    int* umax = ws_ptr<int>(ws, p.off_umax);
    if (p.gcn == kGcnRows) return launch_gcn_rows(p, x, g.adj, w1, b1, w2, b2, u, umax, rows, st);
    const int rc = p.sparse ? launch_gcn_sparse(p, ws, g, x, w1, b1, w2, b2, rows, st)
                            : launch_gcn_dense<2, true>(p.gcn, p.gcn_rb, p.gcn_smem, x, g.adj, w1, b1, w2, b2, u, rows,
                                                        p.S, p.Fi, p.Fh, p.Fo, p.IP, st);
    if (rc || !p.tc || rows < 1) return rc;
    const long long rt = (rows + wg::kT2BM - 1) / wg::kT2BM * wg::kT2BM;
    wg::u_rowmax_kernel<<<(unsigned)((rt + 255) / 256), 256, 0, st>>>(u, umax, rows, p.IP);
    WG_CUDA(cudaGetLastError());
    return WG_OK;
}

// The projection of the `rows` U rows into GI rows gi[0 .. rows) (row stride p.GP).
int launch_inproj_tc(const Plan& p, void* ws, long long rows, cudaStream_t st, float* gi) {
    const long long m_tiles = (rows + wg::kT2BM - 1) / wg::kT2BM;
    if (m_tiles < 1) return WG_OK;
    const wg::Tc2Shape& t = p.tc2;
    WG_CUDA(cudaFuncSetAttribute(wg::inproj_tc2_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                 (int)t.smem_bytes));
    const long long tiles = m_tiles * t.n_nt;
    const unsigned grid = (unsigned)(tiles < wg::kNumSMs ? tiles : wg::kNumSMs);
    wg::inproj_tc2_kernel<<<grid, wg::kT2Threads, t.smem_bytes, st>>>(
        ws_ptr<float>(ws, p.off_u), ws_ptr<int>(ws, p.off_umax), ws_ptr<__half>(ws, p.off_wp),
        ws_ptr<float>(ws, p.off_tcs), ws_ptr<float>(ws, p.off_bias), gi, rows, p.IP, t.KP, p.GP, t.n_nt, t.N_each,
        t.stages);
    WG_CUDA(cudaGetLastError());
    return WG_OK;
}

int launch_inproj(const Plan& p, void* ws, long long rows, cudaStream_t st, float* gi) {
    if (p.tc) return launch_inproj_tc(p, ws, rows, st, gi);
    const long long m_tiles = (rows + wg::kIpBM - 1) / wg::kIpBM;
    const int n_tiles = p.NPB / wg::kIpBN;
    const long long grid = m_tiles * n_tiles;
    if (grid < 1) return WG_OK;
    WG_CUDA(cudaFuncSetAttribute(wg::inproj_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                 wg::kIpSmemBytes));
    wg::inproj_kernel<<<(unsigned)grid, wg::kIpThreads, wg::kIpSmemBytes, st>>>(
        ws_ptr<float>(ws, p.off_u), ws_ptr<float>(ws, p.off_wp), ws_ptr<float>(ws, p.off_bias), gi, rows, p.IP, p.GP,
        n_tiles);
    WG_CUDA(cudaGetLastError());
    return WG_OK;
}

// The recurrence launchers take row0 = NULL for a chunk of sequences laid out one after another in GI (the
// forward), or the device array of each window's first GI row (the forecast: the windowed instantiations, which
// store only h at the last step, out [Bc][H]).

// FP32 recurrence of the hidden sizes gru_recur_unit_kernel cannot fit (H = 125 .. 360): W_hh^T read through L1 / L2
int launch_recur_wide(const Plan& p, void* ws, float* out, long long Bc, cudaStream_t st, const long long* row0) {
    auto kern = row0 ? wg::gru_recur_kernel<true> : wg::gru_recur_kernel<false>;
    WG_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)p.rc_smem));
    const long long grid = (Bc + wg::kRcBT - 1) / wg::kRcBT;
    if (grid < 1) return WG_OK;
    kern<<<(unsigned)grid, wg::kRcWarps * 32, p.rc_smem, st>>>(ws_ptr<float>(ws, p.off_gi), ws_ptr<float>(ws, p.off_wht),
                                                              ws_ptr<float>(ws, p.off_bhn), out, Bc, p.T, p.H, p.GP,
                                                              p.KP, p.NPR, row0 ? 0 : p.rc_ts, row0);
    WG_CUDA(cudaGetLastError());
    return WG_OK;
}

// ---- second-generation throughput recurrence (recur_unit.cuh) ----
// sequences per group: the R in [4, 8] that needs the fewest (waves x R) for this batch
int recur_u_pick_r(long long Bc, int ngrp) {
    int best = wg::kRuMaxR;
    long long best_cost = -1;
    for (int r = wg::kRuMaxR; r >= wg::kRuMinR; --r) {
        const long long ctas = (Bc + (long long)ngrp * r - 1) / ((long long)ngrp * r);
        const long long waves = (ctas + wg::kNumSMs - 1) / wg::kNumSMs;
        const long long cost = waves * (r + 1);   // +1: the per-step work that does not shrink with R
        if (best_cost < 0 || cost < best_cost) { best_cost = cost; best = r; }
    }
    return best;
}

using RegwKernel = decltype(&wg::gru_recur_regw_kernel<false, 1, 24>);
template <bool SAVE, int KPT, bool WIN = false>
RegwKernel regw_kernel(int nb) {
    const RegwKernel k[4] = {wg::gru_recur_regw_kernel<SAVE, 1, KPT, WIN>, wg::gru_recur_regw_kernel<SAVE, 2, KPT, WIN>,
                             wg::gru_recur_regw_kernel<SAVE, 3, KPT, WIN>, wg::gru_recur_regw_kernel<SAVE, 4, KPT, WIN>};
    return k[nb - 1];
}
int launch_recur_regw(const Plan& p, void* ws, float* out, long long Bc, int nb, cudaStream_t st, float* gsave,
                      int ldsave, const long long* row0) {
    if (Bc < 1) return WG_OK;
    const RegwKernel kern =
        row0    ? (p.KP == 104 ? regw_kernel<false, 104, true>(nb) : regw_kernel<false, 24, true>(nb))
        : gsave ? (p.KP == 104 ? regw_kernel<true, 104>(nb) : regw_kernel<true, 24>(nb))
                : (p.KP == 104 ? regw_kernel<false, 104>(nb) : regw_kernel<false, 24>(nb));
    const size_t smem = wg::recur_regw_smem_floats(p.KP, p.NPR, p.GP) * 4;
    WG_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const long long grid = (Bc + wg::kRsBT - 1) / wg::kRsBT;
    kern<<<(unsigned)grid, wg::kRwThreads, smem, st>>>(ws_ptr<float>(ws, p.off_gi), ws_ptr<float>(ws, p.off_wht),
                                                      ws_ptr<float>(ws, p.off_bhn), out, Bc, p.T, p.H, p.GP, p.NPR,
                                                      gsave, ldsave, row0);
    WG_CUDA(cudaGetLastError());
    return WG_OK;
}

using UnitKernel = decltype(&wg::gru_recur_unit_kernel<4, 1, false, 0>);
template <int WPG, bool SAVE, int HT, bool WIN>
UnitKernel unit_kernel(int r) {
    const UnitKernel k[5] = {
        wg::gru_recur_unit_kernel<4, WPG, SAVE, HT, WIN>, wg::gru_recur_unit_kernel<5, WPG, SAVE, HT, WIN>,
        wg::gru_recur_unit_kernel<6, WPG, SAVE, HT, WIN>, wg::gru_recur_unit_kernel<7, WPG, SAVE, HT, WIN>,
        wg::gru_recur_unit_kernel<8, WPG, SAVE, HT, WIN>};
    return k[r - wg::kRuMinR];
}
template <bool SAVE, bool WIN = false>
UnitKernel unit_kernel(const Plan& p, int r) {
    if (p.ru_ht == 102) return unit_kernel<2, SAVE, 102, WIN>(r);
    if (p.ru_ht == 21) return unit_kernel<1, SAVE, 21, WIN>(r);
    return p.ru_wpg == 1 ? unit_kernel<1, SAVE, 0, WIN>(r) : unit_kernel<2, SAVE, 0, WIN>(r);
}
int launch_recur_unit(const Plan& p, void* ws, float* out, long long Bc, int r, cudaStream_t st, float* gsave,
                      int ldsave, const long long* row0) {
    const UnitKernel kern =
        row0 ? unit_kernel<false, true>(p, r) : gsave ? unit_kernel<true>(p, r) : unit_kernel<false>(p, r);
    const size_t smem = wg::recur_u_smem_floats(p.H, r) * 4;
    WG_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const int per_cta = (wg::kRuWarps / p.ru_wpg) * r;
    const long long grid = (Bc + per_cta - 1) / per_cta;
    if (grid < 1) return WG_OK;
    // FMA-pipe hand-over between the two one-warp groups of a scheduler (profiles/r02_handover_ab.json: H = 21, 4096
    // sequences: 0.395 -> 0.358 ms, identical results).  Two-warp groups (H = 102) own their scheduler and need none.
    const int handover = p.ru_wpg == 1 ? 1 : 0;
    kern<<<(unsigned)grid, wg::kRuThreads, smem, st>>>(ws_ptr<float>(ws, p.off_gi), ws_ptr<float>(ws, p.off_whu),
                                                      ws_ptr<float>(ws, p.off_bhn), out, Bc, p.T, p.H, gsave, ldsave,
                                                      handover, row0);
    WG_CUDA(cudaGetLastError());
    return WG_OK;
}

int launch_recur_tc(const Plan& p, void* ws, float* out, long long Bc, cudaStream_t st, const long long* row0) {
    auto kern = row0 ? wg::gru_recur_tc_kernel<true> : wg::gru_recur_tc_kernel<false>;
    const size_t smem = wg::recur_tc_smem_bytes(p.H);
    WG_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const long long grid = (Bc + wg::kRtSeqs - 1) / wg::kRtSeqs;
    if (grid < 1) return WG_OK;
    kern<<<(unsigned)grid, wg::kRtThreads, smem, st>>>(ws_ptr<float>(ws, p.off_gi), ws_ptr<__half>(ws, p.off_whh_hi),
                                                      ws_ptr<__half>(ws, p.off_whh_lo),
                                                      ws_ptr<float>(ws, p.off_tcs) + p.tc2.NP,
                                                      ws_ptr<float>(ws, p.off_bhn), out, Bc, p.T, p.H, p.GP, row0);
    WG_CUDA(cudaGetLastError());
    return WG_OK;
}

// whether a chunk of Bc sequences runs gru_recur_regw_kernel (launch_recur)
bool regw_serves(const Plan& p, long long Bc) {
    return p.recur != kRecurTc && p.regw && Bc <= 2LL * wg::kRsBT * wg::kNumSMs;
}

// The recurrence of one chunk: the plan's kernel, except that up to two waves of 4-sequence CTAs run
// gru_recur_regw_kernel where it serves the contraction length (FMA chains per thread = sequences per CTA that can
// exist: the reference's batch-1 calls run one).  gsave: the training forward, which also saves [r | z | n | hn] per
// (sequence, step), row stride ldsave; only the regw and unit kernels save gates, and make_train_plan accepts only the
// shapes that reach one of them.  row0: the forecast's windows (see launch_recur_wide), which save no gates.
int launch_recur(const Plan& p, void* ws, float* out, long long Bc, cudaStream_t st, float* gsave, int ldsave,
                 const long long* row0 = nullptr) {
    if (regw_serves(p, Bc)) return launch_recur_regw(p, ws, out, Bc, Bc >= 4 ? 4 : (int)Bc, st, gsave, ldsave, row0);
    if (p.recur == kRecurUnit) {
        const int r = recur_u_pick_r(Bc, wg::kRuWarps / p.ru_wpg);
        return launch_recur_unit(p, ws, out, Bc, r < p.ru_rmax ? r : p.ru_rmax, st, gsave, ldsave, row0);
    }
    if (p.recur == kRecurTc) return launch_recur_tc(p, ws, out, Bc, st, row0);   // the tensor path: every batch size
    return launch_recur_wide(p, ws, out, Bc, st, row0);
}

int launch_pack(const Plan& p, void* ws, const float* w_ih, const float* w_hh, const float* b_ih,
                const float* b_hh, cudaStream_t st) {
    pack_params_kernel<<<wg::kNumSMs * 2, 256, 0, st>>>(
        w_ih, w_hh, b_ih, b_hh, ws_ptr<float>(ws, p.off_wp), ws_ptr<float>(ws, p.off_bias),
        ws_ptr<float>(ws, p.off_wht), p.whu ? ws_ptr<float>(ws, p.off_whu) : nullptr, ws_ptr<float>(ws, p.off_bhn),
        p.I, p.H, p.IP, p.NPB, p.KP, p.NPR, p.tc ? 0 : 1, p.n_bias);
    WG_CUDA(cudaGetLastError());
    if (p.tc) {
        wg::pack_wih_tc2_kernel<<<wg::kNumSMs, 256, 0, st>>>(w_ih, ws_ptr<__half>(ws, p.off_wp),
                                                            ws_ptr<float>(ws, p.off_tcs), p.G, p.I, p.tc2.KP,
                                                            p.tc2.n_nt, p.tc2.N_each);
        WG_CUDA(cudaGetLastError());
    }
    if (p.recur == kRecurTc) {
        wg::pack_whh_tc_kernel<<<48, 256, 0, st>>>(w_hh, ws_ptr<__half>(ws, p.off_whh_hi),
                                                  ws_ptr<__half>(ws, p.off_whh_lo),
                                                  ws_ptr<float>(ws, p.off_tcs) + p.tc2.NP, p.H);
        WG_CUDA(cudaGetLastError());
    }
    return WG_OK;
}

// One chunk (Bc <= plan.chunk sequences) through the three stages; gsave / ldsave: see launch_recur.
int run_chunk(const Plan& p, void* ws, const Graph& g, const float* x, const float* w1, const float* b1,
              const float* w2, const float* b2, float* out, long long Bc, cudaStream_t st, float* gsave = nullptr,
              int ldsave = 0) {
    const long long rows = Bc * p.T;
    int rc = launch_gcn(p, ws, g, x, w1, b1, w2, b2, rows, st);
    if (rc) return rc;
    rc = launch_inproj(p, ws, rows, st, ws_ptr<float>(ws, p.off_gi));
    if (rc) return rc;
    return launch_recur(p, ws, out, Bc, st, gsave, ldsave);
}

// Per-device tables (constant-bank ordering below, host-path streams): DeviceGuard has rejected a negative index.
constexpr int kMaxDevices = 64;

// Per-call setup of the second-generation CSR kernel: weights into the constant bank, gather plan.
// The constant bank is one per device: forwards on different streams are ordered through an event (a later
// call's upload waits for the earlier call's last GCN kernel), the host side is serialised by a mutex that
// the caller holds from prepare_sparse to finish_sparse.
std::mutex g_sq_mu;
struct SqDeviceState { cudaEvent_t ev = nullptr; cudaStream_t last = nullptr; bool recorded = false; };
SqDeviceState g_sq_dev[kMaxDevices];

int prepare_sparse(const Plan& p, void* ws, const Graph& g, const float* w1, const float* b1, const float* w2,
                   const float* b2, int device, cudaStream_t st) {
    if (device >= kMaxDevices) return fail(WG_ERR_BAD_ARG, "device index %d out of range", device);
    wg::SqWeights* stage = ws_ptr<wg::SqWeights>(ws, p.off_sqw);
    wg::sq_pack_weights_kernel<<<32, 256, 0, st>>>(w1, b1, w2, b2, stage, p.Fi, p.Fh, p.Fo);
    WG_CUDA(cudaGetLastError());
    const int wbs = wg::ceil_div(p.S, 32);
    wg::csr_plan_kernel<<<wg::ceil_div(wbs, 4), 128, 0, st>>>(g.rowptr, g.colidx, g.vals, p.S,
                                                             ws_ptr<int>(ws, p.off_sqsteps),
                                                             ws_ptr<int2>(ws, p.off_sqpairs));
    WG_CUDA(cudaGetLastError());
    SqDeviceState& d = g_sq_dev[device];
    cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
    cudaStreamIsCapturing(st, &cap);
    if (cap == cudaStreamCaptureStatusNone && d.recorded && d.last != st) WG_CUDA(cudaStreamWaitEvent(st, d.ev, 0));
    WG_CUDA(cudaMemcpyToSymbolAsync(wg::c_sq, stage, sizeof(wg::SqWeights), 0, cudaMemcpyDeviceToDevice, st));
    return WG_OK;
}
int finish_sparse(int device, cudaStream_t st) {
    SqDeviceState& d = g_sq_dev[device];
    cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
    cudaStreamIsCapturing(st, &cap);
    if (cap != cudaStreamCaptureStatusNone) return WG_OK;
    if (!d.ev) WG_CUDA(cudaEventCreateWithFlags(&d.ev, cudaEventDisableTiming));
    WG_CUDA(cudaEventRecord(d.ev, st));
    d.last = st;
    d.recorded = true;
    return WG_OK;
}

bool any_null(std::initializer_list<const void*> ps) {
    for (const void* q : ps)
        if (!q) return true;
    return false;
}

// The frame of a device-buffer forward or forecast, on either graph form: check the pointers (x: the input windows or
// the table) and the workspace (need bytes), switch to the device, pack the parameters, then run `stages` on the
// stream.  On gcn_sparse_plan_kernel the CSR graph also holds the constant bank from prepare_sparse to finish_sparse.
template <typename Stages>
int run_packed(const Plan& p, size_t need, const Graph& g, const float* x, const float* w1, const float* b1,
               const float* w2, const float* b2, const float* w_ih, const float* w_hh, const float* b_ih,
               const float* b_hh, const float* out, void* ws, size_t ws_bytes, int device, void* stream,
               Stages stages) {
    const bool no_graph = p.sparse ? any_null({g.rowptr, g.colidx, g.vals}) : !g.adj;
    if (no_graph || any_null({x, w1, b1, w2, b2, w_ih, w_hh, b_ih, b_hh, out}))
        return fail(WG_ERR_BAD_ARG, "null pointer argument");
    int rc = check_ws(ws, ws_bytes, need);
    if (rc) return rc;
    DeviceGuard dg(device);
    WG_CUDA(dg.err);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if ((rc = launch_pack(p, ws, w_ih, w_hh, b_ih, b_hh, st))) return rc;
    const bool sq = p.gcn == kGcnSparsePlan;
    std::unique_lock<std::mutex> sq_lock(g_sq_mu, std::defer_lock);
    if (sq) {
        sq_lock.lock();
        if ((rc = prepare_sparse(p, ws, g, w1, b1, w2, b2, device, st))) return rc;
    }
    if ((rc = stages(st))) return rc;
    return sq ? finish_sparse(device, st) : WG_OK;
}

// The device-buffer forward of a finished plan: every chunk through the three stages.  need: the workspace bytes to
// check (the training plan adds its regions to the forward's); gsave / ldsave: see launch_recur.
int forward(const Plan& p, size_t need, const Graph& g, const float* x, const float* w1, const float* b1,
            const float* w2, const float* b2, const float* w_ih, const float* w_hh, const float* b_ih,
            const float* b_hh, float* out, long long B, void* ws, size_t ws_bytes, int device, void* stream,
            float* gsave = nullptr, int ldsave = 0) {
    if (B == 0) return WG_OK;
    auto stages = [&](cudaStream_t st) {
        const size_t x_seq = (size_t)p.T * p.S * p.Fi, o_seq = (size_t)p.T * p.H;
        for (long long b0 = 0; b0 < B; b0 += p.chunk) {
            const long long Bc = (B - b0) < p.chunk ? (B - b0) : p.chunk;
            const int rc = run_chunk(p, ws, g, x + (size_t)b0 * x_seq, w1, b1, w2, b2, out + (size_t)b0 * o_seq, Bc,
                                     st, gsave ? gsave + (size_t)b0 * p.T * ldsave : nullptr, ldsave);
            if (rc) return rc;
        }
        return (int)WG_OK;
    };
    return run_packed(p, need, g, x, w1, b1, w2, b2, w_ih, w_hh, b_ih, b_hh, out, ws, ws_bytes, device, stream,
                      stages);
}

// ---- rolling forecasts: windows over one table --------------------------------------------------
// GCN and input projection depend only on a table row, the recurrence on the window (h0 = 0 at its first row): the
// rows the windows cover run the first two stages once, each into a GI row of its own, and every window's recurrence
// reads its L rows in place.  The plan is the forward's for N windows of L steps, with a GI region of Ttot rows and
// the windows' first GI rows (int64, relative to the first row covered) after it.
struct ForecastPlan {
    Plan p;
    size_t off_row0, total;
};

int make_forecast_plan(ForecastPlan& f, long long N, long long Ttot, int L, int S, int Fi, int Fh, int Fo, int H,
                       long long chunk, bool sparse, int flags) {
    if (N < 0 || L < 1 || Ttot < L)
        return fail(WG_ERR_BAD_ARG, "forecast: need N >= 0 and 1 <= L <= Ttot (N=%lld L=%d Ttot=%lld)", N, L, Ttot);
    int rc = plan_layout(f.p, N, L, S, Fi, Fh, Fo, H, chunk, sparse, flags, Ttot);
    if (rc || (rc = plan_launch(f.p))) return rc;
    f.off_row0 = f.p.total;
    f.total = align_up(f.off_row0 + (size_t)N * sizeof(long long));
    return WG_OK;
}

// starts: HOST [N], validated before anything else is looked at; out [N][H] = h at the last step of each window.
int forecast(const ForecastPlan& f, const Graph& g, const float* table, const int64_t* starts, const float* w1,
             const float* b1, const float* w2, const float* b2, const float* w_ih, const float* w_hh,
             const float* b_ih, const float* b_hh, float* out, long long N, long long Ttot, void* ws,
             size_t ws_bytes, int device, void* stream) {
    const Plan& p = f.p;
    if (N == 0) return WG_OK;
    if (!starts) return fail(WG_ERR_BAD_ARG, "starts is NULL (N=%lld)", N);
    const long long last = Ttot - p.T;
    long long lo = 0, hi = 0;
    for (long long n = 0; n < N; ++n) {
        const long long s = starts[n];
        if (s < 0 || s > last)
            return fail(WG_ERR_BAD_ARG, "starts[%lld] = %lld outside [0, Ttot - L] = [0, %lld]", n, s, last);
        if (n == 0 || s < lo) lo = s;
        if (n == 0 || s > hi) hi = s;
    }
    auto stages = [&](cudaStream_t st) {
        // first GI rows relative to the span; a pageable source is staged before cudaMemcpyAsync returns
        std::vector<long long> row0((size_t)N);
        for (long long n = 0; n < N; ++n) row0[(size_t)n] = starts[n] - lo;
        long long* row0_dev = ws_ptr<long long>(ws, f.off_row0);
        WG_CUDA(cudaMemcpyAsync(row0_dev, row0.data(), (size_t)N * sizeof(long long), cudaMemcpyHostToDevice, st));
        // GCN + projection over table rows [lo, hi + L), in pieces of the U scratch's rows
        float* gi = ws_ptr<float>(ws, p.off_gi);
        const size_t x_row = (size_t)p.S * p.Fi;
        const long long span = hi + p.T - lo, piece = forecast_piece_rows(p, Ttot);
        for (long long r0 = 0; r0 < span; r0 += piece) {
            const long long rows = span - r0 < piece ? span - r0 : piece;
            int rc = launch_gcn(p, ws, g, table + (size_t)(lo + r0) * x_row, w1, b1, w2, b2, rows, st);
            if (rc || (rc = launch_inproj(p, ws, rows, st, gi + (size_t)r0 * p.GP))) return rc;
        }
        // the recurrence in the forward's chunks, so that every chunk runs the kernel the forward would
        for (long long b0 = 0; b0 < N; b0 += p.chunk) {
            const long long Bc = (N - b0) < p.chunk ? (N - b0) : p.chunk;
            const int rc = launch_recur(p, ws, out + (size_t)b0 * p.H, Bc, st, nullptr, 0, row0_dev + b0);
            if (rc) return rc;
        }
        return (int)WG_OK;
    };
    return run_packed(p, f.total, g, table, w1, b1, w2, b2, w_ih, w_hh, b_ih, b_hh, out, ws, ws_bytes, device, stream,
                      stages);
}

// The wg_stage_* entry points: plan one chunk, check Bc, the workspace and the device, then run `launch`.
template <typename Launch>
int run_stage(long long Bc, int T, int S, int Fi, int Fh, int Fo, int H, long long chunk, int flags, void* ws,
              size_t ws_bytes, int device, void* stream, Launch launch) {
    Plan p;
    int rc = make_plan(p, chunk, T, S, Fi, Fh, Fo, H, chunk, false, flags);
    if (rc) return rc;
    if (Bc < 0 || Bc > p.chunk) return fail(WG_ERR_BAD_ARG, "Bc=%lld outside [0, chunk=%lld]", Bc, p.chunk);
    if ((rc = check_ws(ws, ws_bytes, p.total))) return rc;
    DeviceGuard g(device);
    WG_CUDA(g.err);
    return launch(p, static_cast<cudaStream_t>(stream));
}


// w_ih [G][I] -> [NP/64][KP][64] with element (n, k) = w_ih[k][n] (the B operand of dU = dGI . w_ih in
// inproj_kernel's layout), zero padded; zb: NP zeros (that kernel always adds a bias)
__global__ void pack_wih_bwd_kernel(const float* __restrict__ w_ih, float* __restrict__ wp, float* __restrict__ zb,
                                    int G, int I, int KP, int NP) {
    const long long total = (long long)NP * KP;
    for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < total;
         e += (long long)gridDim.x * blockDim.x) {
        const int nl = (int)(e % wg::kIpBN);
        const long long r = e / wg::kIpBN;
        const int k = (int)(r % KP), n = (int)(r / KP) * wg::kIpBN + nl;
        wp[e] = (k < G && n < I) ? w_ih[(size_t)k * I + n] : 0.0f;
    }
    for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < NP; e += gridDim.x * blockDim.x) zb[e] = 0.0f;
}

// ---------------------------------------------------------------------------------------------
// training step: forward that saves the gate values, backward (BPTT + GEMMs + GCN backward)
// ---------------------------------------------------------------------------------------------
// BPTT kernels: gru_bwd_regw_kernel<BT, HPT> (W_hh in registers, HPT = 104 or 24) in the CTA sizes kGbRegwBT, else
// gru_bwd_kernel<BT> with 4 or kGbBT sequences per CTA
using GbRegwKernel = decltype(&wg::gru_bwd_regw_kernel<4, 24>);
using GbKernel = decltype(&wg::gru_bwd_kernel<4>);
constexpr int kGbRegwBT[4] = {4, 8, 16, 28};
template <int HPT>
GbRegwKernel gb_regw_kernel(int i) {
    const GbRegwKernel k[4] = {wg::gru_bwd_regw_kernel<4, HPT>, wg::gru_bwd_regw_kernel<8, HPT>,
                               wg::gru_bwd_regw_kernel<16, HPT>, wg::gru_bwd_regw_kernel<28, HPT>};
    return k[i];
}

// GCN backward kernel: gcn_bwd_rows_kernel (13 / 13 / 13 features, S <= 48), else gcn_bwd_kernel<13> (exactly 13
// features everywhere) or gcn_bwd_kernel<16>
enum GcnBwdKind { kGcnBwdRows, kGcnBwd13, kGcnBwd16 };

struct TrainPlan {
    Plan f;            // the forward's plan (chunk == B, FP32 path, dense graph)
    int LD4;           // row stride of the gate / DG buffers: 4H rounded up to 4
    long long rows;    // B * T
    // 1. BPTT: exactly one of gb_regw and gb is set
    GbRegwKernel gb_regw;
    GbKernel gb;
    int HP, GR;        // H rounded up to 4; gru_bwd_kernel: padded contraction length
    int gb_threads, gb_grid, gb_parts;   // gb_parts: bias partial sets the kernel writes (3 per CTA on gb_regw, else 2)
    size_t gb_smem;
    // 2. dW_hh on sgemm_kernel: K splits of the r / z and of the n product
    int splits_hh_a, splits_hh_b;
    // 3. dW_ih on gemm_kb_kernel: tiles over the input features / the gate columns, splits of the B*T rows
    int mt_ih, nt_ih, splits_ih;
    long long kt_per_ih;    // k-tiles (16 rows) per split
    // 4. dU on inproj_kernel
    int ldu, KPd, NPd;  // dU row stride (I rounded up to 4); K / N of the dU GEMM padded for inproj_kernel
    dim3 tg_du;         // rows_to_tiles_kernel: dGI into K-major 128-row tiles
    long long mt_du;    // inproj_kernel: row tiles
    int nt_du;          //                column tiles
    // 5. GCN backward
    GcnBwdKind gcn;
    int grid_gcn, rb_gcn, parts_gcn;   // parts_gcn: partial gradient sets the GCN backward writes
    size_t smem_gcn;
    size_t off_gates, off_dg, off_dgt, off_wpb, off_zb, off_du, off_biasp, off_gcnp, off_splitk, total;
};

int pick_splits(long long M, long long N, long long K) {
    const long long tiles = ((M + wg::kSgBM - 1) / wg::kSgBM) * ((N + wg::kSgBN - 1) / wg::kSgBN);
    long long s = (2LL * wg::kNumSMs) / tiles;  // whole grid resident at once (2 CTAs per SM): one wave
    const long long kmax = (K + 63) / 64;  // at least 64 k's per split
    if (s > kmax) s = kmax;
    return s < 1 ? 1 : (int)s;
}

size_t param_count(int S, int Fi, int Fh, int Fo, int H) {
    const size_t I = (size_t)S * Fo, G = 3 * (size_t)H;
    return (size_t)Fi * Fh + Fh + (size_t)Fh * Fo + Fo + G * I + G * H + G + G;
}

// Largest GRU hidden size training accepts: the bound of the recurrence it was built and tested with (W_hh^T resident
// in shared memory beside the state of 32 sequences).  The gate-saving recurrence that runs now
// (gru_recur_unit_kernel or gru_recur_regw_kernel) serves every H up to it.
constexpr int kTrainMaxH = 106;

int make_train_plan(TrainPlan& tp, long long B, int T, int S, int Fi, int Fh, int Fo, int H) {
    const long long Bn = B > 0 ? B : 1;   // B = 0 plans one sequence: the backward then only zeroes the gradients
    int rc = plan_layout(tp.f, B, T, S, Fi, Fh, Fo, H, Bn, false, 0);
    if (rc) return rc;
    const Plan& p = tp.f;
    if (Fi > 16 || Fh > 16 || Fo > 16)
        return fail(WG_ERR_UNSUPPORTED, "training: GCN feature widths must be <= 16 (got %d / %d / %d)", Fi, Fh, Fo);
    tp.LD4 = wg::round_up(4 * H, 4);
    tp.HP = wg::round_up(H, 4);
    int bt;   // sequences per BPTT CTA
    if (tp.HP == 104 || tp.HP == 24) {
        // W_hh in registers: the smallest CTA size that still makes the grid one wave (28 sequences fit)
        int i = 0;
        while (i < 3 && (Bn + kGbRegwBT[i] - 1) / kGbRegwBT[i] > wg::kNumSMs) ++i;
        bt = kGbRegwBT[i];
        tp.gb_regw = tp.HP == 104 ? gb_regw_kernel<104>(i) : gb_regw_kernel<24>(i);
        tp.gb = nullptr;
        tp.gb_threads = wg::kGrwThreads;
        tp.gb_smem = wg::gru_bwd_regw_smem_floats(tp.HP, bt) * 4;
    } else {
        // 16 sequences per CTA when that fills the machine, else 4 (the recurrence is latency-bound: with few
        // sequences per GPU — configs[4]: 512 — more, lighter CTAs shorten every one of the T serial steps)
        bt = Bn > 4LL * wg::kNumSMs ? wg::kGbBT : 4;
        tp.GR = wg::gru_bwd_gr(H, bt);
        tp.gb_smem = wg::gru_bwd_smem_floats(tp.HP, tp.GR, bt) * 4;
        if (tp.HP > 128 || (tp.HP / 4) * (bt / 4) * wg::gru_bwd_ksplit(bt) > wg::kGbThreads ||
            tp.gb_smem > (size_t)wg::kMaxSmemOptin)
            return fail(WG_ERR_UNSUPPORTED, "training: GRU hidden size %d too large for the shared-memory BPTT kernel", H);
        tp.gb_regw = nullptr;
        tp.gb = bt == 4 ? wg::gru_bwd_kernel<4> : wg::gru_bwd_kernel<wg::kGbBT>;
        tp.gb_threads = wg::kGbThreads;
    }
    tp.gb_grid = (int)((Bn + bt - 1) / bt);
    tp.gb_parts = tp.gb_grid * (tp.gb_regw ? 3 : 2);
    // the forward's recurrence saves the gates: only gru_recur_regw_kernel and gru_recur_unit_kernel do (launch_recur)
    if (H > kTrainMaxH || !(regw_serves(p, B) || p.recur == kRecurUnit))
        return fail(WG_ERR_UNSUPPORTED, "training: GRU hidden size %d does not fit the shared-memory recurrence", H);
    tp.rows = Bn * T;
    tp.ldu = wg::round_up(p.I, 4);
    tp.KPd = wg::round_up(p.G, wg::kIpBK);
    tp.NPd = wg::round_up(p.I, wg::kIpBN);
    // GCN backward geometry (same station grouping as the forward)
    if (wg::gcn_bwd_rows_applies(S, Fi, Fh, Fo) &&
        wg::gcn_bwd_rows_smem_floats(S, tp.ldu) * 4 <= (size_t)wg::kMaxSmemOptin) {
        tp.gcn = kGcnBwdRows;
        tp.rb_gcn = wg::kGb2Rows;
        tp.smem_gcn = wg::gcn_bwd_rows_smem_floats(S, tp.ldu) * 4;
        const long long nblk = (tp.rows + wg::kGb2Rows - 1) / wg::kGb2Rows;
        const int per_sm = tp.smem_gcn + 1024 <= (size_t)(228 * 1024) / 2 ? 2 : 1;   // 228 KB per SM, 1 KB reserved per CTA
        tp.grid_gcn = (int)(nblk < (long long)per_sm * wg::kNumSMs ? nblk : (long long)per_sm * wg::kNumSMs);
        tp.parts_gcn = tp.grid_gcn * wg::kGb2Slices;
    } else {
        tp.gcn = Fi == 13 && Fh == 13 && Fo == 13 ? kGcnBwd13 : kGcnBwd16;
        const int NSG = wg::ceil_div(S, wg::kGbwSG);
        if (NSG > wg::kGcnThreads) return fail(WG_ERR_UNSUPPORTED, "training: S=%d too large for the dense GCN kernels", S);
        int RB = wg::kGbwThreads / NSG;
        const int cols = S * Fi;
        const int need = (cols % 4 == 0) ? 1 : (cols % 2 == 0) ? 2 : 4;
        if (RB > need) RB -= RB % need;
        auto smem_of = [&](int rb) { return wg::gcn_bwd_smem_floats(S, tp.ldu, rb) * 4; };
        while (smem_of(RB) > (size_t)wg::kMaxSmemOptin && RB > 1) RB = (RB > need) ? RB - need : RB - 1;
        if (smem_of(RB) > (size_t)wg::kMaxSmemOptin)
            return fail(WG_ERR_UNSUPPORTED, "training: S=%d does not fit the shared-memory GCN backward", S);
        tp.rb_gcn = RB;
        tp.smem_gcn = smem_of(RB);
        const long long nblk = (tp.rows + RB - 1) / RB;
        tp.grid_gcn = (int)(nblk < wg::kNumSMs ? nblk : wg::kNumSMs);
        tp.parts_gcn = tp.grid_gcn * (wg::kGbwThreads / 16);
    }
    // dU stage: dGI re-laid into K-major 128-row tiles by one pass of 32-row blocks (at most 65535 of them)
    const long long rt = (tp.rows + wg::kUTileRows - 1) / wg::kUTileRows * wg::kUTileRows;
    if (rt / 32 > 65535) return fail(WG_ERR_UNSUPPORTED, "training: B*T = %lld rows exceed one pass", tp.rows);
    tp.tg_du = dim3((unsigned)((tp.KPd + 31) / 32), (unsigned)(rt / 32));
    tp.mt_du = rt / wg::kIpBM;
    tp.nt_du = tp.NPd / wg::kIpBN;
    tp.splits_hh_a = pick_splits(2 * H, H, tp.rows);
    tp.splits_hh_b = pick_splits(H, H, tp.rows);
    // dW_ih on gemm_kb_kernel<64, 160, 0>: tiles over (i, g), the B*T rows split so that the grid is one wave
    tp.mt_ih = (p.IP + wg::KbWih::kBM - 1) / wg::KbWih::kBM;
    tp.nt_ih = (p.G + wg::KbWih::kBN - 1) / wg::KbWih::kBN;
    {
        const long long ktall = (tp.rows + wg::kKbBK - 1) / wg::kKbBK;
        long long sp = (3LL * wg::kNumSMs) / ((long long)tp.mt_ih * tp.nt_ih);   // one wave at 3 CTAs per SM
        if (sp < 1) sp = 1;
        if (sp > ktall) sp = ktall;
        tp.kt_per_ih = (ktall + sp - 1) / sp;
        tp.splits_ih = (int)((ktall + tp.kt_per_ih - 1) / tp.kt_per_ih);
    }
    size_t o = p.total;
    tp.off_gates = o; o = align_up(o + (size_t)tp.rows * tp.LD4 * 4);
    tp.off_dg = o;    o = align_up(o + (size_t)tp.rows * tp.LD4 * 4);
    tp.off_dgt = o;   o = align_up(o + (size_t)rt * tp.KPd * 4);              // dGI in K-major 128-row tiles
    tp.off_wpb = o;   o = align_up(o + (size_t)tp.NPd * tp.KPd * 4);          // w_ih packed for dU = dGI . w_ih
    tp.off_zb = o;    o = align_up(o + (size_t)tp.NPd * 4);                   // zero bias (written by the pack kernel)
    tp.off_du = o;    o = align_up(o + (size_t)tp.rows * tp.ldu * 4);
    tp.off_biasp = o; o = align_up(o + (size_t)tp.gb_grid * 3 * tp.LD4 * 4);  // 3 partial sets per CTA (regw), else 2
    tp.off_gcnp = o;  o = align_up(o + (size_t)tp.parts_gcn * (2 * 256 + 32) * 4);
    size_t sk = (size_t)tp.splits_hh_a * 2 * H * H;
    if ((size_t)tp.splits_hh_b * H * H > sk) sk = (size_t)tp.splits_hh_b * H * H;
    if ((size_t)tp.splits_ih * p.I * tp.nt_ih * wg::KbWih::kBN > sk) sk = (size_t)tp.splits_ih * p.I * tp.nt_ih * wg::KbWih::kBN;
    tp.off_splitk = o; o = align_up(o + sk * 4);
    tp.total = o;
    return plan_launch(tp.f);   // last: a shape outside the training limits reports those
}

bool aligned16(const void* q) { return (reinterpret_cast<uintptr_t>(q) & 15) == 0; }

// C[M][N] (strided out[m * s_m + n * s_n]) = A . B with K split over `splits` CTAs per tile.
int splitk_gemm(const wg::SgOperand& A, const wg::SgOperand& Bo, long long M, int N, long long K, int splits,
                float* part, float* out, long long s_m, long long s_n, cudaStream_t st) {
    if (M < 1 || N < 1) return WG_OK;
    long long kper = (K + splits - 1) / splits;
    kper = (kper + wg::kSgBK - 1) / wg::kSgBK * wg::kSgBK;
    const dim3 grid((unsigned)((N + wg::kSgBN - 1) / wg::kSgBN), (unsigned)((M + wg::kSgBM - 1) / wg::kSgBM),
                    (unsigned)splits);
    WG_CUDA(cudaFuncSetAttribute(wg::sgemm_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, wg::kSgSmemBytes));
    // splits == 1 still goes through `part` (dense [M][N]) so that the strided write is in one place
    wg::sgemm_kernel<<<grid, wg::kSgThreads, wg::kSgSmemBytes, st>>>(A, Bo, part, N, M, N, K, kper);
    WG_CUDA(cudaGetLastError());
    const long long total = M * N;
    wg::sg_reduce_kernel<<<(unsigned)((total * 8 + 255) / 256), 256, 0, st>>>(part, splits, M, N, out, s_m, s_n, N);
    WG_CUDA(cudaGetLastError());
    return WG_OK;
}

// FFMA peak microbenchmark: 8 independent chains per thread, register resident.
__global__ void __launch_bounds__(256) ffma_peak_kernel(float* sink, int iters, float a, float b) {
    float v0 = threadIdx.x, v1 = v0 + 1, v2 = v0 + 2, v3 = v0 + 3, v4 = v0 + 4, v5 = v0 + 5, v6 = v0 + 6,
          v7 = v0 + 7;
    for (int i = 0; i < iters; ++i) {
#pragma unroll
        for (int u = 0; u < 16; ++u) {
            v0 = fmaf(v0, a, b); v1 = fmaf(v1, a, b); v2 = fmaf(v2, a, b); v3 = fmaf(v3, a, b);
            v4 = fmaf(v4, a, b); v5 = fmaf(v5, a, b); v6 = fmaf(v6, a, b); v7 = fmaf(v7, a, b);
        }
    }
    const float s = v0 + v1 + v2 + v3 + v4 + v5 + v6 + v7;
    if (s == 123.456f) sink[0] = s;  // never true in practice; keeps the chains alive
}

}  // namespace

// =============================================================================================
extern "C" {

int wg_abi_version(void) { return WG_ABI_VERSION; }
// used by graph.cu (separate translation unit, built with -fmad=false) to set the error text
int wg_internal_fail(int code, const char* msg) { return fail(code, "%s", msg); }
const char* wg_last_error(void) { return g_err; }

size_t wg_gcn_gru_workspace_bytes(int64_t B, int T, int S, int F_in, int F_hid, int F_out, int H,
                                  int64_t chunk, int flags) {
    Plan p;
    if (make_plan(p, B, T, S, F_in, F_hid, F_out, H, chunk, false, flags)) return 0;
    return p.total;
}

int wg_stage_pack_f32(const float* w_ih, const float* w_hh, const float* b_ih, const float* b_hh, int T,
                      int S, int F_in, int F_hid, int F_out, int H, int64_t chunk, int flags, void* workspace,
                      size_t workspace_bytes, int device, void* stream) {
    if (any_null({w_ih, w_hh, b_ih, b_hh})) return fail(WG_ERR_BAD_ARG, "null parameter pointer");
    auto launch = [&](const Plan& p, cudaStream_t st) { return launch_pack(p, workspace, w_ih, w_hh, b_ih, b_hh, st); };
    return run_stage(0, T, S, F_in, F_hid, F_out, H, chunk, flags, workspace, workspace_bytes, device, stream, launch);
}

int wg_stage_gcn_f32(const float* adj, const float* x, const float* w1, const float* b1, const float* w2,
                     const float* b2, int64_t Bc, int T, int S, int F_in, int F_hid, int F_out, int H,
                     int64_t chunk, int flags, void* workspace, size_t workspace_bytes, int device, void* stream) {
    if (any_null({adj, x, w1, b1, w2, b2})) return fail(WG_ERR_BAD_ARG, "null pointer");
    auto launch = [&](const Plan& p, cudaStream_t st) {
        return launch_gcn(p, workspace, Graph{adj}, x, w1, b1, w2, b2, Bc * T, st);
    };
    return run_stage(Bc, T, S, F_in, F_hid, F_out, H, chunk, flags, workspace, workspace_bytes, device, stream, launch);
}

int wg_stage_inproj_f32(int64_t Bc, int T, int S, int F_in, int F_hid, int F_out, int H, int64_t chunk,
                        int flags, void* workspace, size_t workspace_bytes, int device, void* stream) {
    auto launch = [&](const Plan& p, cudaStream_t st) {
        return launch_inproj(p, workspace, Bc * T, st, ws_ptr<float>(workspace, p.off_gi));
    };
    return run_stage(Bc, T, S, F_in, F_hid, F_out, H, chunk, flags, workspace, workspace_bytes, device, stream, launch);
}

int wg_stage_recur_f32(float* out, int64_t Bc, int T, int S, int F_in, int F_hid, int F_out, int H,
                       int64_t chunk, int flags, void* workspace, size_t workspace_bytes, int device, void* stream) {
    if (!out) return fail(WG_ERR_BAD_ARG, "null output pointer");
    auto launch = [&](const Plan& p, cudaStream_t st) { return launch_recur(p, workspace, out, Bc, st, nullptr, 0); };
    return run_stage(Bc, T, S, F_in, F_hid, F_out, H, chunk, flags, workspace, workspace_bytes, device, stream, launch);
}

int wg_gcn_gru_forward_f32(const float* adj, const float* x, const float* w1, const float* b1,
                           const float* w2, const float* b2, const float* w_ih, const float* w_hh,
                           const float* b_ih, const float* b_hh, float* out, int64_t B, int T, int S,
                           int F_in, int F_hid, int F_out, int H, int64_t chunk, int flags, void* workspace,
                           size_t workspace_bytes, int device, void* stream) {
    Plan p;
    const int rc = make_plan(p, B, T, S, F_in, F_hid, F_out, H, chunk, false, flags);
    return rc ? rc : forward(p, p.total, Graph{adj}, x, w1, b1, w2, b2, w_ih, w_hh, b_ih, b_hh, out, B, workspace,
                             workspace_bytes, device, stream);
}

size_t wg_gcn_gru_csr_workspace_bytes(int64_t B, int T, int S, int F_in, int F_hid, int F_out, int H,
                                      int64_t chunk, int flags) {
    Plan p;
    if (make_plan(p, B, T, S, F_in, F_hid, F_out, H, chunk, true, flags)) return 0;
    return p.total;
}

int wg_gcn_gru_forward_csr_f32(const int32_t* rowptr, const int32_t* colidx, const float* vals, const float* x,
                               const float* w1, const float* b1, const float* w2, const float* b2,
                               const float* w_ih, const float* w_hh, const float* b_ih, const float* b_hh,
                               float* out, int64_t B, int T, int S, int F_in, int F_hid, int F_out, int H,
                               int64_t chunk, int flags, void* workspace, size_t workspace_bytes, int device,
                               void* stream) {
    Plan p;
    const int rc = make_plan(p, B, T, S, F_in, F_hid, F_out, H, chunk, true, flags);
    return rc ? rc : forward(p, p.total, Graph{nullptr, rowptr, colidx, vals}, x, w1, b1, w2, b2, w_ih, w_hh, b_ih,
                             b_hh, out, B, workspace, workspace_bytes, device, stream);
}

size_t wg_gcn_gru_forecast_workspace_bytes(int64_t N, int64_t Ttot, int L, int S, int F_in, int F_hid, int F_out,
                                           int H, int64_t chunk, int flags) {
    ForecastPlan f;
    if (make_forecast_plan(f, N, Ttot, L, S, F_in, F_hid, F_out, H, chunk, false, flags)) return 0;
    return f.total;
}

int wg_gcn_gru_forecast_f32(const float* adj, const float* table, const int64_t* starts, const float* w1,
                            const float* b1, const float* w2, const float* b2, const float* w_ih, const float* w_hh,
                            const float* b_ih, const float* b_hh, float* out, int64_t N, int64_t Ttot, int L, int S,
                            int F_in, int F_hid, int F_out, int H, int64_t chunk, int flags, void* workspace,
                            size_t workspace_bytes, int device, void* stream) {
    ForecastPlan f;
    const int rc = make_forecast_plan(f, N, Ttot, L, S, F_in, F_hid, F_out, H, chunk, false, flags);
    return rc ? rc : forecast(f, Graph{adj}, table, starts, w1, b1, w2, b2, w_ih, w_hh, b_ih, b_hh, out, N, Ttot,
                              workspace, workspace_bytes, device, stream);
}

size_t wg_gcn_gru_forecast_csr_workspace_bytes(int64_t N, int64_t Ttot, int L, int S, int F_in, int F_hid, int F_out,
                                               int H, int64_t chunk, int flags) {
    ForecastPlan f;
    if (make_forecast_plan(f, N, Ttot, L, S, F_in, F_hid, F_out, H, chunk, true, flags)) return 0;
    return f.total;
}

int wg_gcn_gru_forecast_csr_f32(const int32_t* rowptr, const int32_t* colidx, const float* vals, const float* table,
                                const int64_t* starts, const float* w1, const float* b1, const float* w2,
                                const float* b2, const float* w_ih, const float* w_hh, const float* b_ih,
                                const float* b_hh, float* out, int64_t N, int64_t Ttot, int L, int S, int F_in,
                                int F_hid, int F_out, int H, int64_t chunk, int flags, void* workspace,
                                size_t workspace_bytes, int device, void* stream) {
    ForecastPlan f;
    const int rc = make_forecast_plan(f, N, Ttot, L, S, F_in, F_hid, F_out, H, chunk, true, flags);
    return rc ? rc : forecast(f, Graph{nullptr, rowptr, colidx, vals}, table, starts, w1, b1, w2, b2, w_ih, w_hh,
                              b_ih, b_hh, out, N, Ttot, workspace, workspace_bytes, device, stream);
}

}  // extern "C"

namespace {

// ---- host-buffer variant: H2D / compute / D2H of consecutive chunks overlapped ----------------
// Two compute lanes (streams, each with its own scratch) so that the latency-bound recurrence of chunk c
// overlaps the GCN / projection of chunk c+1; three staging slots each for x, out and pred.
constexpr int kHostLanes = 2;
constexpr int kHostSlots = 3;
constexpr long long kHostDefaultChunk = 256;   // measured best piece size for the 34-station model (DESIGN.md, section 5)

// workspace = [ compute workspace 0 | compute workspace 1 | x staging 0..2 | out staging 0..2 | pred staging 0..2 ]
struct HostLayout {
    size_t lane, xs, os, ps;   // bytes of one compute workspace and of one x / out / pred staging slot
    size_t total;
};
int host_plan(Plan& p, HostLayout& L, long long B, int T, int S, int Fi, int Fh, int Fo, int H, long long chunk,
              int flags) {
    if (chunk == 0) chunk = kHostDefaultChunk;   // the host path pipelines: a piece small enough to overlap copies
    int rc = make_plan(p, B, T, S, Fi, Fh, Fo, H, chunk, false, flags);
    if (rc) return rc;
    L.lane = align_up(p.total);
    L.xs = align_up((size_t)p.chunk * T * S * Fi * 4);
    L.os = align_up((size_t)p.chunk * T * H * 4);
    L.ps = align_up((size_t)p.chunk * H * 4);   // de-normalised last step (wg_gcn_gru_predict_host_f32)
    L.total = kHostLanes * L.lane + kHostSlots * (L.xs + L.os + L.ps);
    return WG_OK;
}

// Internal streams and events of the host-buffer entry points: created once per (host thread, device) and
// reused by every later call of that thread (creating 4 streams + 9 events per call cost ~0.1 ms).
struct HostCtx {
    bool ready = false;
    cudaStream_t s_in = nullptr, s_out = nullptr, s_cmp[kHostLanes] = {};
    cudaEvent_t ev_in[kHostSlots] = {}, ev_cmp[kHostSlots] = {}, ev_out[kHostSlots] = {};
};
thread_local HostCtx g_host_ctx[kMaxDevices];

int host_ctx(int device, HostCtx** out) {
    if (device >= kMaxDevices) return fail(WG_ERR_BAD_ARG, "device index %d out of range", device);
    HostCtx& c = g_host_ctx[device];
    if (!c.ready) {
        WG_CUDA(cudaStreamCreateWithFlags(&c.s_in, cudaStreamNonBlocking));
        WG_CUDA(cudaStreamCreateWithFlags(&c.s_out, cudaStreamNonBlocking));
        for (int l = 0; l < kHostLanes; ++l) WG_CUDA(cudaStreamCreateWithFlags(&c.s_cmp[l], cudaStreamNonBlocking));
        for (int i = 0; i < kHostSlots; ++i) {
            WG_CUDA(cudaEventCreateWithFlags(&c.ev_in[i], cudaEventDisableTiming));
            WG_CUDA(cudaEventCreateWithFlags(&c.ev_cmp[i], cudaEventDisableTiming));
            WG_CUDA(cudaEventCreateWithFlags(&c.ev_out[i], cudaEventDisableTiming));
        }
        c.ready = true;
    }
    *out = &c;
    return WG_OK;
}

// last_only: instead of out [B,T,H], `dst_host` receives pred [B,H] = out[:, T-1, :] * (vmax - vmin) + vmin
int host_pipeline(const float* adj, const float* x_host, const float* w1, const float* b1, const float* w2,
                  const float* b2, const float* w_ih, const float* w_hh, const float* b_ih, const float* b_hh,
                  float* dst_host, int64_t B, int T, int S, int F_in, int F_hid, int F_out, int H, int64_t chunk,
                  int flags, void* workspace, size_t workspace_bytes, int device, bool last_only, double vmin,
                  double vmax) {
    Plan p;
    HostLayout L;
    int rc = host_plan(p, L, B, T, S, F_in, F_hid, F_out, H, chunk, flags);
    if (rc) return rc;
    if (B == 0) return WG_OK;
    if (any_null({adj, x_host, w1, b1, w2, b2, w_ih, w_hh, b_ih, b_hh, dst_host}))
        return fail(WG_ERR_BAD_ARG, "null pointer argument");
    if ((rc = check_ws(workspace, workspace_bytes, L.total))) return rc;
    DeviceGuard g(device);
    WG_CUDA(g.err);
    HostCtx* cx = nullptr;
    if ((rc = host_ctx(device, &cx))) return rc;

    char* base = static_cast<char*>(workspace);
    void* lane_ws[kHostLanes];
    for (int l = 0; l < kHostLanes; ++l) lane_ws[l] = base + l * L.lane;
    char* slots = base + kHostLanes * L.lane;
    float* xdev[kHostSlots];
    float* odev[kHostSlots];
    float* pdev[kHostSlots];
    for (int i = 0; i < kHostSlots; ++i) {
        xdev[i] = reinterpret_cast<float*>(slots + i * L.xs);
        odev[i] = reinterpret_cast<float*>(slots + kHostSlots * L.xs + i * L.os);
        pdev[i] = reinterpret_cast<float*>(slots + kHostSlots * (L.xs + L.os) + i * L.ps);
    }
    int result = WG_OK;
#define WG_CUDA_H(expr)                                                                         \
    do {                                                                                        \
        cudaError_t e_ = (expr);                                                                \
        if (e_ != cudaSuccess) {                                                                \
            result = fail(WG_ERR_CUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(e_),  \
                          __FILE__, __LINE__);                                                  \
            cudaDeviceSynchronize();                                                            \
            return result;                                                                      \
        }                                                                                       \
    } while (0)

    auto synced = [](int code) { cudaDeviceSynchronize(); return code; };   // an error leaves no copy in flight
    const long long n_chunks = (B + p.chunk - 1) / p.chunk;
    for (int l = 0; l < kHostLanes && l < n_chunks; ++l)   // each lane packs the parameters into its own scratch
        if ((rc = launch_pack(p, lane_ws[l], w_ih, w_hh, b_ih, b_hh, cx->s_cmp[l]))) return synced(rc);
    const Graph graph{adj};
    const size_t x_seq = (size_t)T * S * F_in, o_seq = (size_t)T * H;
    for (long long c = 0; c < n_chunks; ++c) {
        const int sl = (int)(c % kHostSlots), lane = (int)(c % kHostLanes);
        const long long b0 = c * p.chunk;
        const long long Bc = (B - b0) < p.chunk ? (B - b0) : p.chunk;
        // x staging slot is free once the compute that read it (chunk c - slots) is done
        if (c >= kHostSlots) WG_CUDA_H(cudaStreamWaitEvent(cx->s_in, cx->ev_cmp[sl], 0));
        WG_CUDA_H(cudaMemcpyAsync(xdev[sl], x_host + (size_t)b0 * x_seq, (size_t)Bc * x_seq * 4,
                                  cudaMemcpyHostToDevice, cx->s_in));
        WG_CUDA_H(cudaEventRecord(cx->ev_in[sl], cx->s_in));
        // compute waits for its input and for the D2H that last used this out slot (chunk c - slots);
        // the lane's scratch is free because chunk c - lanes ran on the same stream
        WG_CUDA_H(cudaStreamWaitEvent(cx->s_cmp[lane], cx->ev_in[sl], 0));
        if (c >= kHostSlots) WG_CUDA_H(cudaStreamWaitEvent(cx->s_cmp[lane], cx->ev_out[sl], 0));
        if ((rc = run_chunk(p, lane_ws[lane], graph, xdev[sl], w1, b1, w2, b2, odev[sl], Bc, cx->s_cmp[lane])))
            return synced(rc);
        if (last_only &&   // only 3S floats per window leave the GPU (src/main.py:103,116)
            (rc = wg_denorm_last_step_f32(odev[sl], pdev[sl], Bc, T, H, vmin, vmax, device, cx->s_cmp[lane])))
            return synced(rc);
        WG_CUDA_H(cudaEventRecord(cx->ev_cmp[sl], cx->s_cmp[lane]));
        WG_CUDA_H(cudaStreamWaitEvent(cx->s_out, cx->ev_cmp[sl], 0));
        if (last_only)
            WG_CUDA_H(cudaMemcpyAsync(dst_host + (size_t)b0 * H, pdev[sl], (size_t)Bc * H * 4, cudaMemcpyDeviceToHost,
                                      cx->s_out));
        else
            WG_CUDA_H(cudaMemcpyAsync(dst_host + (size_t)b0 * o_seq, odev[sl], (size_t)Bc * o_seq * 4,
                                      cudaMemcpyDeviceToHost, cx->s_out));
        WG_CUDA_H(cudaEventRecord(cx->ev_out[sl], cx->s_out));
    }
    WG_CUDA_H(cudaStreamSynchronize(cx->s_out));
    for (int l = 0; l < kHostLanes; ++l) WG_CUDA_H(cudaStreamSynchronize(cx->s_cmp[l]));
    WG_CUDA_H(cudaStreamSynchronize(cx->s_in));
#undef WG_CUDA_H
    return WG_OK;
}

}  // namespace

extern "C" {

size_t wg_gcn_gru_host_workspace_bytes(int64_t B, int T, int S, int F_in, int F_hid, int F_out, int H,
                                       int64_t chunk, int flags) {
    Plan p;
    HostLayout L;
    if (host_plan(p, L, B, T, S, F_in, F_hid, F_out, H, chunk, flags)) return 0;
    return L.total;
}

int wg_gcn_gru_forward_host_f32(const float* adj, const float* x_host, const float* w1, const float* b1,
                                const float* w2, const float* b2, const float* w_ih, const float* w_hh,
                                const float* b_ih, const float* b_hh, float* out_host, int64_t B, int T,
                                int S, int F_in, int F_hid, int F_out, int H, int64_t chunk, int flags,
                                void* workspace, size_t workspace_bytes, int device) {
    return host_pipeline(adj, x_host, w1, b1, w2, b2, w_ih, w_hh, b_ih, b_hh, out_host, B, T, S, F_in, F_hid, F_out, H,
                         chunk, flags, workspace, workspace_bytes, device, false, 0.0, 1.0);
}

int wg_gcn_gru_predict_host_f32(const float* adj, const float* x_host, const float* w1, const float* b1,
                                const float* w2, const float* b2, const float* w_ih, const float* w_hh,
                                const float* b_ih, const float* b_hh, float* pred_host, int64_t B, int T,
                                int S, int F_in, int F_hid, int F_out, int H, int64_t chunk, int flags, double vmin,
                                double vmax, void* workspace, size_t workspace_bytes, int device) {
    return host_pipeline(adj, x_host, w1, b1, w2, b2, w_ih, w_hh, b_ih, b_hh, pred_host, B, T, S, F_in, F_hid, F_out,
                         H, chunk, flags, workspace, workspace_bytes, device, true, vmin, vmax);
}

int wg_gcn_layer_f32(const float* adj, const float* attr, const float* weight, const float* bias,
                     float* out, int64_t R, int S, int F_in, int F_out, int device, void* stream) {
    if (R < 0 || S <= 0 || F_in <= 0 || F_out <= 0)
        return fail(WG_ERR_BAD_ARG, "non-positive dimension (R=%lld S=%d F=%d/%d)", (long long)R, S, F_in, F_out);
    if (R == 0) return WG_OK;
    if (any_null({adj, attr, weight, bias, out})) return fail(WG_ERR_BAD_ARG, "null pointer argument");
    DeviceGuard g(device);
    WG_CUDA(g.err);
    // single layer: "hidden" plays the role of the output width
    const GcnKind k = dense_gcn_kind(S, F_in, F_out, F_out);
    int RB = 0;
    size_t smem = 0;
    const int rc = dense_gcn_geometry(k, S, F_in, F_out, F_out, RB, smem);
    if (rc) return rc;
    return launch_gcn_dense<1, false>(k, RB, smem, attr, adj, weight, bias, nullptr, nullptr, out, R, S, F_in, F_out,
                                      F_out, S * F_out, static_cast<cudaStream_t>(stream));
}


// ---- training step --------------------------------------------------------------------------
size_t wg_gcn_gru_param_count(int S, int F_in, int F_hid, int F_out, int H) {
    if (S <= 0 || F_in <= 0 || F_hid <= 0 || F_out <= 0 || H <= 0) return 0;
    return param_count(S, F_in, F_hid, F_out, H);
}

size_t wg_gcn_gru_train_workspace_bytes(int64_t B, int T, int S, int F_in, int F_hid, int F_out, int H) {
    TrainPlan tp;
    if (make_train_plan(tp, B, T, S, F_in, F_hid, F_out, H)) return 0;
    return tp.total;
}

int wg_gcn_gru_forward_train_f32(const float* adj, const float* x, const float* w1, const float* b1,
                                 const float* w2, const float* b2, const float* w_ih, const float* w_hh,
                                 const float* b_ih, const float* b_hh, float* out, int64_t B, int T, int S,
                                 int F_in, int F_hid, int F_out, int H, void* workspace, size_t workspace_bytes,
                                 int device, void* stream) {
    TrainPlan tp;
    const int rc = make_train_plan(tp, B, T, S, F_in, F_hid, F_out, H);
    if (rc) return rc;
    float* gates = workspace ? ws_ptr<float>(workspace, tp.off_gates) : nullptr;   // forward() rejects a NULL workspace
    return forward(tp.f, tp.total, Graph{adj}, x, w1, b1, w2, b2, w_ih, w_hh, b_ih, b_hh, out, B, workspace,
                   workspace_bytes, device, stream, gates, tp.LD4);
}

int wg_gcn_gru_backward_f32(const float* adj, const float* x, const float* w1, const float* b1, const float* w2,
                            const float* b2, const float* w_ih, const float* w_hh, const float* out,
                            const float* d_out, float* grads, int64_t B, int T, int S, int F_in, int F_hid,
                            int F_out, int H, void* workspace, size_t workspace_bytes, int device, void* stream) {
    TrainPlan tp;
    int rc = make_train_plan(tp, B, T, S, F_in, F_hid, F_out, H);
    if (rc) return rc;
    if (any_null({adj, x, w1, b1, w2, b2, w_ih, w_hh, out, d_out, grads}))
        return fail(WG_ERR_BAD_ARG, "null pointer argument");
    DeviceGuard g(device);
    WG_CUDA(g.err);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const Plan& p = tp.f;
    const size_t n_params = param_count(S, F_in, F_hid, F_out, H);
    if (B == 0) {
        WG_CUDA(cudaMemsetAsync(grads, 0, n_params * 4, st));
        return WG_OK;
    }
    if ((rc = check_ws(workspace, workspace_bytes, tp.total))) return rc;
    // flat gradient layout = state_dict order
    float* d_w1 = grads;
    float* d_b1 = d_w1 + (size_t)F_in * F_hid;
    float* d_w2 = d_b1 + F_hid;
    float* d_b2 = d_w2 + (size_t)F_hid * F_out;
    float* d_wih = d_b2 + F_out;
    float* d_whh = d_wih + (size_t)p.G * p.I;
    float* d_bih = d_whh + (size_t)p.G * H;
    float* d_bhh = d_bih + p.G;

    float* gates = ws_ptr<float>(workspace, tp.off_gates);
    float* DG = ws_ptr<float>(workspace, tp.off_dg);
    float* dU = ws_ptr<float>(workspace, tp.off_du);
    float* biasp = ws_ptr<float>(workspace, tp.off_biasp);
    float* skp = ws_ptr<float>(workspace, tp.off_splitk);
    const long long rows = tp.rows;

    // 1. BPTT through the recurrence: DG = [da_r | da_z | da_n | da_n r], bias partials
    if (tp.gb_regw) {
        WG_CUDA(cudaFuncSetAttribute(tp.gb_regw, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tp.gb_smem));
        tp.gb_regw<<<tp.gb_grid, tp.gb_threads, tp.gb_smem, st>>>(gates, out, d_out, w_hh, DG, biasp, B, T, H, tp.LD4);
    } else {
        WG_CUDA(cudaFuncSetAttribute(tp.gb, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tp.gb_smem));
        tp.gb<<<tp.gb_grid, tp.gb_threads, tp.gb_smem, st>>>(gates, out, d_out, w_hh, DG, biasp, B, T, H, tp.LD4, tp.HP,
                                                              tp.GR);
    }
    WG_CUDA(cudaGetLastError());
    wg::gru_bias_grad_kernel<<<(4 * H + 127) / 128, 128, 0, st>>>(biasp, tp.gb_parts, H, tp.LD4, d_bih, d_bhh);
    WG_CUDA(cudaGetLastError());
    const int dg_vec = (tp.LD4 % 4 == 0) && aligned16(DG);
    // 2. dW_hh = dGH^T . H_prev   (H_prev[b, t] = out[b, t-1], 0 at t = 0)
    {
        const wg::SgOperand hprev{out, H, 0, 0, (H % 4 == 0) && aligned16(out), T};
        const wg::SgOperand a_rz{DG, tp.LD4, 0, 0, dg_vec, 0};
        if ((rc = splitk_gemm(a_rz, hprev, 2 * H, H, rows, tp.splits_hh_a, skp, d_whh, H, 1, st))) return rc;
        const wg::SgOperand a_n{DG + 3 * (size_t)H, tp.LD4, 0, 0, dg_vec && ((3 * H) % 4 == 0), 0};
        if ((rc = splitk_gemm(a_n, hprev, H, H, rows, tp.splits_hh_b, skp, d_whh + 2 * (size_t)H * H, H, 1, st)))
            return rc;
    }
    // 3. dW_ih [3H x I] = dGI^T . U: gemm_kb_kernel reads dGI (row-major, as the BPTT kernel wrote it) and U (the
    //    forward's K-major tiles) in place; one wave of CTAs over (tile, row split), fixed-order reduction
    {
        using Cfg = wg::KbWih;
        auto kern = wg::gemm_kb_kernel<Cfg::kBM, Cfg::kBN, Cfg::kTN>;
        WG_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::kSmemBytes));
        wg::KbArgs a{};
        a.a = ws_ptr<float>(workspace, p.off_u);
        a.b = DG;
        a.c = skp;
        a.R = rows;
        a.I = p.I;
        a.IP = p.IP;
        a.ld_dg = tp.LD4;
        a.ldc = tp.nt_ih * Cfg::kBN;
        a.m_tiles = tp.mt_ih;
        a.n_tiles = tp.nt_ih;
        a.kt_per_split = tp.kt_per_ih;
        const dim3 grid((unsigned)(tp.mt_ih * tp.nt_ih), (unsigned)tp.splits_ih);
        kern<<<grid, Cfg::kThreads, Cfg::kSmemBytes, st>>>(a);
        WG_CUDA(cudaGetLastError());
        // d_wih[g][i] = sum_z part[z][i][g]
        const long long total = (long long)p.G * p.I;
        wg::sg_reduce_kernel<<<(unsigned)((total * 8 + 255) / 256), 256, 0, st>>>(skp, tp.splits_ih, p.I, p.G, d_wih, 1, p.I,
                                                                             a.ldc);
        WG_CUDA(cudaGetLastError());
    }
    // 4. dU [BT x I] = dGI . W_ih on the forward's projection kernel (bulk-copy pipeline, 87 % of the FMA
    //    peak): dGI re-laid into K-major 128-row tiles, w_ih packed as [N/64][K][64], zero bias.  (A variant
    //    of gemm_kb_kernel that reads dGI in place ran this product in 3.60 ms against 0.32 + 3.01 ms here.)
    {
        float* DGt = ws_ptr<float>(workspace, tp.off_dgt);
        float* wpb = ws_ptr<float>(workspace, tp.off_wpb);
        float* zb = ws_ptr<float>(workspace, tp.off_zb);
        wg::rows_to_tiles_kernel<<<tp.tg_du, 256, 0, st>>>(DG, DGt, rows, p.G, tp.LD4, tp.KPd);
        WG_CUDA(cudaGetLastError());
        pack_wih_bwd_kernel<<<wg::kNumSMs, 256, 0, st>>>(w_ih, wpb, zb, p.G, p.I, tp.KPd, tp.NPd);
        WG_CUDA(cudaGetLastError());
        WG_CUDA(cudaFuncSetAttribute(wg::inproj_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, wg::kIpSmemBytes));
        wg::inproj_kernel<<<(unsigned)(tp.mt_du * tp.nt_du), wg::kIpThreads, wg::kIpSmemBytes, st>>>(
            DGt, wpb, zb, dU, rows, tp.KPd, tp.ldu, tp.nt_du);
        WG_CUDA(cudaGetLastError());
    }
    // 5. GCN backward: dW1, db1, dW2, db2
    float* gcnp = ws_ptr<float>(workspace, tp.off_gcnp);
    if (tp.gcn == kGcnBwdRows) {
        WG_CUDA(cudaFuncSetAttribute(wg::gcn_bwd_rows_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tp.smem_gcn));
        wg::gcn_bwd_rows_kernel<<<tp.grid_gcn, wg::kGb2Threads, tp.smem_gcn, st>>>(x, dU, adj, w1, b1, w2, b2, gcnp, rows,
                                                                                 p.S, tp.ldu);
    } else {
        auto kern = tp.gcn == kGcnBwd13 ? wg::gcn_bwd_kernel<13> : wg::gcn_bwd_kernel<16>;
        WG_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tp.smem_gcn));
        kern<<<tp.grid_gcn, wg::kGbwThreads, tp.smem_gcn, st>>>(x, dU, adj, w1, b1, w2, b2, gcnp, rows, p.S, p.Fi, p.Fh,
                                                               p.Fo, tp.rb_gcn, tp.ldu);
    }
    WG_CUDA(cudaGetLastError());
    wg::gcn_bwd_finish_kernel<<<(2 * 256 + 32 + 7) / 8, 256, 0, st>>>(
        gcnp, tp.parts_gcn, F_in, F_hid, F_out, d_w1, d_b1, d_w2, d_b2);
    WG_CUDA(cudaGetLastError());
    return WG_OK;
}

size_t wg_mse_workspace_bytes(void) { return (size_t)2 * wg::kNumSMs * sizeof(double); }

int wg_mse_loss_grad_f32(const float* out, const float* y, int64_t n, float* d_out, float* loss, void* workspace,
                         size_t workspace_bytes, int device, void* stream) {
    if (n <= 0) return fail(WG_ERR_BAD_ARG, "mse: n must be positive");
    if (any_null({out, y, loss})) return fail(WG_ERR_BAD_ARG, "null pointer argument");
    if (!workspace || workspace_bytes < wg_mse_workspace_bytes() || reinterpret_cast<uintptr_t>(workspace) % 8)
        return fail(WG_ERR_WORKSPACE, "mse: workspace of %zu bytes (8-byte aligned) needed", wg_mse_workspace_bytes());
    DeviceGuard g(device);
    WG_CUDA(g.err);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const int grid = 2 * wg::kNumSMs;
    wg::mse_grad_kernel<<<grid, wg::kMseThreads, 0, st>>>(out, y, d_out, static_cast<double*>(workspace), n,
                                                         (float)(2.0 / (double)n));
    WG_CUDA(cudaGetLastError());
    wg::mse_finish_kernel<<<1, 32, 0, st>>>(static_cast<double*>(workspace), grid, n, loss);
    WG_CUDA(cudaGetLastError());
    return WG_OK;
}

int wg_adam_step_f32(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, int64_t n, double lr,
                     double beta1, double beta2, double eps, int64_t step, double grad_scale, int device,
                     void* stream) {
    if (n < 0 || step < 1) return fail(WG_ERR_BAD_ARG, "adam: n >= 0 and step >= 1 required");
    if (n == 0) return WG_OK;
    if (any_null({param, grad, exp_avg, exp_avg_sq})) return fail(WG_ERR_BAD_ARG, "null pointer argument");
    DeviceGuard g(device);
    WG_CUDA(g.err);
    const double bc1 = 1.0 - std::pow(beta1, (double)step), bc2 = 1.0 - std::pow(beta2, (double)step);
    const long long blocks = (n + 255) / 256;
    const unsigned grid = (unsigned)(blocks < 8LL * wg::kNumSMs ? blocks : 8LL * wg::kNumSMs);
    wg::adam_kernel<<<grid, 256, 0, static_cast<cudaStream_t>(stream)>>>(
        param, grad, exp_avg, exp_avg_sq, n, (float)grad_scale, (float)beta1, (float)beta2, (float)(1.0 - beta1),
        (float)(1.0 - beta2), (float)(lr / bc1),
        (float)sqrt(bc2), (float)eps);
    WG_CUDA(cudaGetLastError());
    return WG_OK;
}

#ifdef WG_RC_TRACE
// debug build only (not declared in the public header)
int wg_debug_read_unit_trace(long long* host, int n) {
    if (n > 8 * 256 * 5) n = 8 * 256 * 5;
    return (int)cudaMemcpyFromSymbol(host, wg::g_ru_trace, sizeof(long long) * n);
}
#endif

double wg_measure_ffma_tflops(int device, int iters) {
    DeviceGuard g(device);
    if (g.err != cudaSuccess) {
        fail(WG_ERR_CUDA, "cudaSetDevice failed: %s", cudaGetErrorString(g.err));
        return -1.0;
    }
    if (iters < 1) iters = 1;
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) return -1.0;
    const int blocks = prop.multiProcessorCount * 8;  // 8 x 256 threads = 64 warps per SM
    const int loop = 4096;
    float* sink = nullptr;
    if (cudaMalloc(&sink, 4) != cudaSuccess) return -1.0;
    cudaEvent_t e0, e1;
    cudaEventCreate(&e0);
    cudaEventCreate(&e1);
    ffma_peak_kernel<<<blocks, 256>>>(sink, loop, 0.999f, 0.001f);  // warm-up
    cudaEventRecord(e0);
    for (int i = 0; i < iters; ++i) ffma_peak_kernel<<<blocks, 256>>>(sink, loop, 0.999f, 0.001f);
    cudaEventRecord(e1);
    cudaError_t e = cudaEventSynchronize(e1);
    float ms = 0.f;
    cudaEventElapsedTime(&ms, e0, e1);
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    cudaFree(sink);
    if (e != cudaSuccess || ms <= 0.f) {
        fail(WG_ERR_CUDA, "ffma microbenchmark failed: %s", cudaGetErrorString(e));
        return -1.0;
    }
    const double flops = 2.0 * 8 * 16 * (double)loop * 256.0 * blocks * iters;
    return flops / (ms * 1e-3) / 1e12;
}

}  // extern "C"
