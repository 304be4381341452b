// Value head: the last Linear(K,1) of ValueEstimator (value_estimator.py:27), its MSE loss (ppo_learner.py:176)
// and the backward into the last hidden activation, as one fused SIMT pass.  A 1-wide output would waste a
// 128xN tensor-core tile, and this pass is HBM-bound anyway: it reads H[M,K] once (2K bytes/row) and, when
// training, writes dH[M,K] once.
//   v = H w + b;  dv = 2*inv_batch*(v - target);  dH = dv * w (.) (H > 0);  dw += sum_m dv*H;  db += sum dv.
// UPSTREAM (rlppo_value_head_backward): the same pass with dv = d_values[row] loaded -- the backward of
// ValueEstimator.forward for an arbitrary upstream gradient (value_estimator.py:30-36).
// K is the true width of the layer below; H and dH rows are read / written as Kp = pad8(K) columns of 16-byte
// chunks.  H's padding columns must hold zeros (the layer-wise forward writes padding units so); dH's are then written
// as +0.  No load or atomic touches w[K..] / dw[K..].  K <= 2048: one warp per row, each lane keeping its slice of w, H and dw in registers.  Wider K
// runs value_head_wide_kernel (below).
#include "common.cuh"

namespace {

constexpr int kThreads = 256;
constexpr int kWarps = kThreads / 32;
constexpr int kMaxK = 28672;           // wide form: w and the dw partials (8 Kp bytes) in <= 227 KB of shared memory

// NI = number of 16-byte (8 x bf16) chunks each lane owns: K <= NI * 256
template <int NI, bool TRAIN, bool UPSTREAM = false>
__global__ void __launch_bounds__(kThreads)
value_head_kernel(const uint16_t* __restrict__ h, int64_t ldh, const float* __restrict__ w, const float* __restrict__ bias,
                  int64_t M, int K, float* __restrict__ values_out, const float* __restrict__ targets, float inv_batch,
                  uint16_t* __restrict__ dh, int64_t lddh, float* __restrict__ dw, float* __restrict__ db,
                  float* __restrict__ metrics, int h_parts, int64_t h_pstride, int dh_parts, int64_t dh_pstride) {
    // UPSTREAM: `targets` holds d_values
    extern __shared__ float s_mem[];   // [pad8(K)] dw partials (TRAIN)
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int nvec = (K + 7) >> 3;
    float wreg[NI][8];
#pragma unroll
    for (int i = 0; i < NI; ++i) {
        const int c = lane + 32 * i;
#pragma unroll
        for (int j = 0; j < 8; ++j) wreg[i][j] = (c * 8 + j < K) ? __ldg(w + c * 8 + j) : 0.f;
    }
    const float b = bias ? __ldg(bias) : 0.f;
    float gw[NI][8];
#pragma unroll
    for (int i = 0; i < NI; ++i)
#pragma unroll
        for (int j = 0; j < 8; ++j) gw[i][j] = 0.f;
    float sum_dv = 0.f, sum_sq = 0.f, rows = 0.f;
    if (TRAIN) {
        for (int i = threadIdx.x; i < nvec * 8; i += kThreads) s_mem[i] = 0.f;
        __syncthreads();
    }
    for (int64_t row = (int64_t)blockIdx.x * kWarps + warp; row < M; row += (int64_t)gridDim.x * kWarps) {
        float hv[NI][8];
        float dot = 0.f;
#pragma unroll
        for (int i = 0; i < NI; ++i) {
            const int c = lane + 32 * i;
            uint4 q = make_uint4(0, 0, 0, 0);
            if (c < nvec) q = __ldg(reinterpret_cast<const uint4*>(h + row * ldh) + c);
            const uint32_t u[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                hv[i][2 * j] = __uint_as_float(u[j] << 16);
                hv[i][2 * j + 1] = __uint_as_float(u[j] & 0xFFFF0000u);
            }
            // split activations (rlppo_split): H = part0 + part1 + ..., parts h_pstride columns apart
            for (int pt = 1; pt < h_parts; ++pt) {
                uint4 q2 = make_uint4(0, 0, 0, 0);
                if (c < nvec) q2 = __ldg(reinterpret_cast<const uint4*>(h + row * ldh + pt * h_pstride) + c);
                const uint32_t u2[4] = {q2.x, q2.y, q2.z, q2.w};
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    hv[i][2 * j] += __uint_as_float(u2[j] << 16);
                    hv[i][2 * j + 1] += __uint_as_float(u2[j] & 0xFFFF0000u);
                }
            }
#pragma unroll
            for (int j = 0; j < 8; ++j) dot = fmaf(hv[i][j], wreg[i][j], dot);
        }
        const float v = rlppo::warp_sum(dot) + b;
        if (values_out != nullptr && lane == 0) values_out[row] = v;
        if (TRAIN) {
            const float err = UPSTREAM ? 0.f : v - __ldg(targets + row);
            const float dv = UPSTREAM ? __ldg(targets + row) : 2.0f * inv_batch * err;
            if (lane == 0) {
                sum_dv += dv;
                sum_sq += err * err;
                rows += 1.f;
            }
#pragma unroll
            for (int i = 0; i < NI; ++i) {
                const int c = lane + 32 * i;
                if (c < nvec) {
                    float o[8];
#pragma unroll
                    for (int j = 0; j < 8; ++j) {
                        gw[i][j] = fmaf(dv, hv[i][j], gw[i][j]);
                        o[j] = hv[i][j] > 0.f ? dv * wreg[i][j] : 0.f;   // ReLU mask of the layer that made H
                    }
                    uint4 q;
                    q.x = rlppo::pack_bf16x2(o[0], o[1]);
                    q.y = rlppo::pack_bf16x2(o[2], o[3]);
                    q.z = rlppo::pack_bf16x2(o[4], o[5]);
                    q.w = rlppo::pack_bf16x2(o[6], o[7]);
                    reinterpret_cast<uint4*>(dh + row * lddh)[c] = q;
                    for (int pt = 1; pt < dh_parts; ++pt) {
                        const uint32_t qq[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
                        for (int j = 0; j < 4; ++j) {
                            o[2 * j] -= __uint_as_float(qq[j] << 16);
                            o[2 * j + 1] -= __uint_as_float(qq[j] & 0xFFFF0000u);
                        }
                        q.x = rlppo::pack_bf16x2(o[0], o[1]);
                        q.y = rlppo::pack_bf16x2(o[2], o[3]);
                        q.z = rlppo::pack_bf16x2(o[4], o[5]);
                        q.w = rlppo::pack_bf16x2(o[6], o[7]);
                        reinterpret_cast<uint4*>(dh + row * lddh + pt * dh_pstride)[c] = q;
                    }
                }
            }
        }
    }
    if (TRAIN) {
#pragma unroll
        for (int i = 0; i < NI; ++i) {
            const int c = lane + 32 * i;
            if (c < nvec) {
#pragma unroll
                for (int j = 0; j < 8; ++j) atomicAdd(&s_mem[c * 8 + j], gw[i][j]);
            }
        }
        __syncthreads();
        for (int i = threadIdx.x; i < K; i += kThreads) atomicAdd(dw + i, s_mem[i]);
        if (lane == 0) {
            if (db) atomicAdd(db, sum_dv);
            if (!UPSTREAM && metrics) {
                atomicAdd(metrics + 5, sum_sq);
                atomicAdd(metrics + 6, rows);
            }
        }
    }
}

// Wide form (K > 2048): a lane's share of w, H and dw no longer fits in registers.  The block takes kRows rows at a
// time, and each of its threads owns the 16-byte column chunks c = tid, tid + 256, ...  Pass 1 reads the tile's H and
// forms per-thread partial dot products, which a block reduction turns into v and dv.  Pass 2 reads the tile's H again
// (from L2: the grid is sized so that the tiles in flight stay well inside it) and writes dH.  It adds dv*H into the
// block's dw partials in shared memory; each column chunk belongs to one thread, so no atomics are needed there.
// w is staged in shared memory, H comes from HBM once, dH goes to HBM once.
constexpr int kRows = 8;

__device__ __forceinline__ void load_h8(const uint16_t* __restrict__ h, int64_t row, int64_t ldh, int h_parts,
                                        int64_t h_pstride, int c, float (&hv)[8]) {
    const uint16_t* base = h + row * ldh + (int64_t)c * 8;
    const uint4 q = __ldg(reinterpret_cast<const uint4*>(base));
    const uint32_t u[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        hv[2 * j] = __uint_as_float(u[j] << 16);
        hv[2 * j + 1] = __uint_as_float(u[j] & 0xFFFF0000u);
    }
    for (int pt = 1; pt < h_parts; ++pt) {
        const uint4 q2 = __ldg(reinterpret_cast<const uint4*>(base + pt * h_pstride));
        const uint32_t u2[4] = {q2.x, q2.y, q2.z, q2.w};
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            hv[2 * j] += __uint_as_float(u2[j] << 16);
            hv[2 * j + 1] += __uint_as_float(u2[j] & 0xFFFF0000u);
        }
    }
}

// Pass 2 of one row tile: dH = dv w (.) (H > 0) written as dh_parts parts, dv*H added into this thread's dw partials.
__device__ __forceinline__ void wide_backward_tile(const uint16_t* __restrict__ h, int64_t ldh, int h_parts,
                                                   int64_t h_pstride, uint16_t* __restrict__ dh, int64_t lddh,
                                                   int dh_parts, int64_t dh_pstride, const float* s_w, float* s_dw,
                                                   const float* s_dv, int64_t r0, int nr, int nvec) {
    float dvr[kRows];
#pragma unroll
    for (int r = 0; r < kRows; ++r) dvr[r] = s_dv[r];
    for (int c = threadIdx.x; c < nvec; c += kThreads) {
        const float4 w0 = *reinterpret_cast<const float4*>(s_w + c * 8);
        const float4 w1 = *reinterpret_cast<const float4*>(s_w + c * 8 + 4);
        const float wv[8] = {w0.x, w0.y, w0.z, w0.w, w1.x, w1.y, w1.z, w1.w};
        float4 g0 = *reinterpret_cast<const float4*>(s_dw + c * 8);
        float4 g1 = *reinterpret_cast<const float4*>(s_dw + c * 8 + 4);
        float g[8] = {g0.x, g0.y, g0.z, g0.w, g1.x, g1.y, g1.z, g1.w};
#pragma unroll
        for (int r = 0; r < kRows; ++r) {
            if (r < nr) {
                float hv[8], o[8];
                load_h8(h, r0 + r, ldh, h_parts, h_pstride, c, hv);
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    g[j] = fmaf(dvr[r], hv[j], g[j]);
                    o[j] = hv[j] > 0.f ? dvr[r] * wv[j] : 0.f;   // ReLU mask of the layer that made H
                }
                uint16_t* out = dh + (r0 + r) * lddh + (int64_t)c * 8;
                for (int pt = 0; pt < dh_parts; ++pt) {
                    uint4 q;
                    q.x = rlppo::pack_bf16x2(o[0], o[1]);
                    q.y = rlppo::pack_bf16x2(o[2], o[3]);
                    q.z = rlppo::pack_bf16x2(o[4], o[5]);
                    q.w = rlppo::pack_bf16x2(o[6], o[7]);
                    *reinterpret_cast<uint4*>(out + pt * dh_pstride) = q;
                    const uint32_t qq[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        o[2 * j] -= __uint_as_float(qq[j] << 16);
                        o[2 * j + 1] -= __uint_as_float(qq[j] & 0xFFFF0000u);
                    }
                }
            }
        }
        *reinterpret_cast<float4*>(s_dw + c * 8) = make_float4(g[0], g[1], g[2], g[3]);
        *reinterpret_cast<float4*>(s_dw + c * 8 + 4) = make_float4(g[4], g[5], g[6], g[7]);
    }
}

template <bool TRAIN, bool UPSTREAM = false>
__global__ void __launch_bounds__(kThreads, 2)
value_head_wide_kernel(const uint16_t* __restrict__ h, int64_t ldh, const float* __restrict__ w,
                       const float* __restrict__ bias, int64_t M, int K, float* __restrict__ values_out,
                       const float* __restrict__ targets, float inv_batch, uint16_t* __restrict__ dh, int64_t lddh,
                       float* __restrict__ dw, float* __restrict__ db, float* __restrict__ metrics, int h_parts,
                       int64_t h_pstride, int dh_parts, int64_t dh_pstride) {
    // UPSTREAM: `targets` holds d_values
    extern __shared__ __align__(16) float s_mem[];   // [Kp] w, then (TRAIN) [Kp] dw partials
    __shared__ float s_red[kWarps][kRows];
    __shared__ float s_dv[kRows];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int nvec = (K + 7) >> 3, Kp = nvec * 8;
    float* s_w = s_mem;
    float* s_dw = s_mem + Kp;
    for (int i = threadIdx.x; i < Kp; i += kThreads) {
        s_w[i] = i < K ? __ldg(w + i) : 0.f;
        if (TRAIN) s_dw[i] = 0.f;
    }
    __syncthreads();
    const float b = bias ? __ldg(bias) : 0.f;
    float sum_dv = 0.f, sum_sq = 0.f, rows = 0.f;
    for (int64_t r0 = (int64_t)blockIdx.x * kRows; r0 < M; r0 += (int64_t)gridDim.x * kRows) {
        const int nr = M - r0 < kRows ? (int)(M - r0) : kRows;
        float dot[kRows];
#pragma unroll
        for (int r = 0; r < kRows; ++r) dot[r] = 0.f;
        for (int c = threadIdx.x; c < nvec; c += kThreads) {
            const float4 w0 = *reinterpret_cast<const float4*>(s_w + c * 8);
            const float4 w1 = *reinterpret_cast<const float4*>(s_w + c * 8 + 4);
            const float wv[8] = {w0.x, w0.y, w0.z, w0.w, w1.x, w1.y, w1.z, w1.w};
#pragma unroll
            for (int r = 0; r < kRows; ++r) {
                if (r < nr) {
                    float hv[8];
                    load_h8(h, r0 + r, ldh, h_parts, h_pstride, c, hv);
#pragma unroll
                    for (int j = 0; j < 8; ++j) dot[r] = fmaf(hv[j], wv[j], dot[r]);
                }
            }
        }
#pragma unroll
        for (int r = 0; r < kRows; ++r) {
            const float sr = rlppo::warp_sum(dot[r]);
            if (lane == 0) s_red[warp][r] = sr;
        }
        __syncthreads();
        if (threadIdx.x < kRows) {
            const int r = threadIdx.x;
            float dv = 0.f;
            if (r < nr) {
                const int64_t row = r0 + r;
                float v = 0.f;
#pragma unroll
                for (int wp = 0; wp < kWarps; ++wp) v += s_red[wp][r];
                v += b;
                if (values_out != nullptr) values_out[row] = v;
                if (TRAIN) {
                    const float err = UPSTREAM ? 0.f : v - __ldg(targets + row);
                    dv = UPSTREAM ? __ldg(targets + row) : 2.0f * inv_batch * err;
                    sum_dv += dv;
                    sum_sq += err * err;
                    rows += 1.f;
                }
            }
            s_dv[r] = dv;
        }
        __syncthreads();     // s_dv ready; s_red free for the next tile
        if (TRAIN) wide_backward_tile(h, ldh, h_parts, h_pstride, dh, lddh, dh_parts, dh_pstride, s_w, s_dw, s_dv, r0, nr, nvec);
    }
    if (TRAIN) {
        __syncthreads();
        for (int i = threadIdx.x; i < K; i += kThreads) atomicAdd(dw + i, s_dw[i]);
        if (threadIdx.x < kRows) {
            if (db) atomicAdd(db, sum_dv);
            if (!UPSTREAM && metrics) {
                atomicAdd(metrics + 5, sum_sq);
                atomicAdd(metrics + 6, rows);
            }
        }
    }
}

template <bool TRAIN, bool UPSTREAM>
int launch_wide(const uint16_t* h, int64_t ldh, const float* w, const float* bias, int64_t M, int K, float* values_out,
                const float* targets, float inv_batch, uint16_t* dh, int64_t lddh, float* dw, float* db, float* metrics,
                int h_parts, int64_t h_pstride, int dh_parts, int64_t dh_pstride, cudaStream_t s) {
    auto kfn = value_head_wide_kernel<TRAIN, UPSTREAM>;
    const int Kp = (K + 7) / 8 * 8;
    const size_t smem = (size_t)Kp * sizeof(float) * (TRAIN ? 2 : 1);
    static bool configured = false;
    if (!configured) {
        RLPPO_CUDA(cudaFuncSetAttribute(kfn, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                        (int)((size_t)kMaxK * sizeof(float) * (TRAIN ? 2 : 1))));
        configured = true;
    }
    // two blocks per SM: 16 independent 16-byte loads per thread in flight cover HBM latency, and the tiles pass 2
    // reads back (kRows rows x all parts) stay a small share of L2
    const int64_t want = (M + kRows - 1) / kRows;
    const int64_t cap = (int64_t)rlppo::num_sms() * 2;
    const unsigned grid = (unsigned)(want < cap ? want : cap);
    kfn<<<grid, kThreads, smem, s>>>(h, ldh, w, bias, M, K, values_out, targets, inv_batch, dh, lddh, dw, db, metrics,
                                     h_parts, h_pstride, dh_parts, dh_pstride);
    RLPPO_LAUNCH_CHECK();
    return RLPPO_OK;
}

template <int NI>
int launch(const uint16_t* h, int64_t ldh, const float* w, const float* bias, int64_t M, int K, float* values_out,
           const float* targets, float inv_batch, uint16_t* dh, int64_t lddh, float* dw, float* db, float* metrics,
           int h_parts, int64_t h_pstride, int dh_parts, int64_t dh_pstride, cudaStream_t s, bool upstream = false) {
    const int64_t want = (M + kWarps - 1) / kWarps;
    const int64_t cap = (int64_t)rlppo::num_sms() * 8;
    const unsigned grid = (unsigned)(want < cap ? want : cap);
    const size_t smem = (size_t)(K + 7) / 8 * 8 * sizeof(float);
    if (upstream)
        value_head_kernel<NI, true, true><<<grid, kThreads, smem, s>>>(h, ldh, w, nullptr, M, K, nullptr, targets, 0.f,
                                                                       dh, lddh, dw, db, nullptr, h_parts, h_pstride,
                                                                       dh_parts, dh_pstride);
    else if (targets != nullptr)
        value_head_kernel<NI, true><<<grid, kThreads, smem, s>>>(h, ldh, w, bias, M, K, values_out, targets, inv_batch,
                                                                 dh, lddh, dw, db, metrics, h_parts, h_pstride, dh_parts,
                                                                 dh_pstride);
    else
        value_head_kernel<NI, false><<<grid, kThreads, 0, s>>>(h, ldh, w, bias, M, K, values_out, nullptr, 0.f, nullptr, 0,
                                                               nullptr, nullptr, nullptr, h_parts, h_pstride, 1, 0);
    RLPPO_LAUNCH_CHECK();
    return RLPPO_OK;
}

// Argument checks shared by both entry points; Kp = pad8(K) columns of H (and dH) are read (written).
int check_shape(const uint16_t* h, int64_t ldh, int K, int h_parts, int64_t h_pstride, int dh_parts,
                int64_t dh_pstride) {
    const int64_t Kp = ((int64_t)K + 7) / 8 * 8;
    RLPPO_CHECK_ARG(K >= 1 && K <= kMaxK && ldh % 8 == 0 && ldh >= Kp,
                    "K must be in [1,%d] and ldh a multiple of 8 covering pad8(K)", kMaxK);
    RLPPO_CHECK_ARG((reinterpret_cast<uintptr_t>(h) & 15) == 0, "H must be 16-byte aligned");
    RLPPO_CHECK_ARG(h_parts >= 1 && h_parts <= 3 && dh_parts >= 1 && dh_parts <= 3 && h_pstride % 8 == 0 &&
                        dh_pstride % 8 == 0 && (h_parts == 1 || h_pstride >= Kp) && (dh_parts == 1 || dh_pstride >= Kp),
                    "split: 1..3 parts, strides multiples of 8 covering pad8(K)");
    return RLPPO_OK;
}

}  // namespace

extern "C" int rlppo_value_head(const uint16_t* h, int64_t ldh, const float* w, const float* bias, int64_t M, int K,
                                float* values_out, const float* targets, float inv_batch, uint16_t* dh, int64_t lddh,
                                float* dw, float* db, float* metrics, int h_parts, int64_t h_pstride, int dh_parts,
                                int64_t dh_pstride, void* stream) {
    RLPPO_REQUIRE_DEVICE();
    RLPPO_CHECK_ARG(h && w && M >= 1, "bad argument");
    int rc = check_shape(h, ldh, K, h_parts, h_pstride, dh_parts, dh_pstride);
    if (rc) return rc;
    if (targets != nullptr) {
        RLPPO_CHECK_ARG(dh && dw && lddh % 8 == 0 && lddh >= (K + 7) / 8 * 8,
                        "training mode needs dh (ld a multiple of 8 covering pad8(K)) and dw");
        RLPPO_CHECK_ARG((reinterpret_cast<uintptr_t>(dh) & 15) == 0, "dH must be 16-byte aligned");
    }
    cudaStream_t s = static_cast<cudaStream_t>(stream);
#define RLPPO_VH(NI_) launch<NI_>(h, ldh, w, bias, M, K, values_out, targets, inv_batch, dh, lddh, dw, db, metrics, h_parts, \
                                  h_pstride, dh_parts, dh_pstride, s)
    if (K <= 256) return RLPPO_VH(1);
    if (K <= 512) return RLPPO_VH(2);
    if (K <= 1024) return RLPPO_VH(4);
    if (K <= 2048) return RLPPO_VH(8);
#undef RLPPO_VH
    if (targets != nullptr)
        return launch_wide<true, false>(h, ldh, w, bias, M, K, values_out, targets, inv_batch, dh, lddh, dw, db, metrics,
                                        h_parts, h_pstride, dh_parts, dh_pstride, s);
    return launch_wide<false, false>(h, ldh, w, bias, M, K, values_out, nullptr, 0.f, nullptr, 0, nullptr, nullptr,
                                     nullptr, h_parts, h_pstride, 1, 0, s);
}

// Backward of ValueEstimator.forward (value_estimator.py:27, the last Linear(K,1) over ReLU activations H) for an
// arbitrary upstream gradient d_values f32[M] (device): dH = dv * w (.) (H > 0), dw[K] += sum_m dv*H, db[1] += sum dv.
extern "C" int rlppo_value_head_backward(const uint16_t* h, int64_t ldh, const float* w, int64_t M, int K,
                                         const float* d_values, uint16_t* dh, int64_t lddh, float* dw, float* db,
                                         int h_parts, int64_t h_pstride, int dh_parts, int64_t dh_pstride, void* stream) {
    RLPPO_REQUIRE_DEVICE();
    RLPPO_CHECK_ARG(h && w && d_values && dh && dw && M >= 1, "bad argument");
    int rc = check_shape(h, ldh, K, h_parts, h_pstride, dh_parts, dh_pstride);
    if (rc) return rc;
    RLPPO_CHECK_ARG((reinterpret_cast<uintptr_t>(dh) & 15) == 0, "H and dH must be 16-byte aligned");
    RLPPO_CHECK_ARG(lddh % 8 == 0 && lddh >= (K + 7) / 8 * 8, "lddh must be a multiple of 8 covering pad8(K)");
    cudaStream_t s = static_cast<cudaStream_t>(stream);
#define RLPPO_VHB(NI_) launch<NI_>(h, ldh, w, nullptr, M, K, nullptr, d_values, 0.f, dh, lddh, dw, db, nullptr, h_parts, \
                                   h_pstride, dh_parts, dh_pstride, s, true)
    if (K <= 256) return RLPPO_VHB(1);
    if (K <= 512) return RLPPO_VHB(2);
    if (K <= 1024) return RLPPO_VHB(4);
    if (K <= 2048) return RLPPO_VHB(8);
#undef RLPPO_VHB
    return launch_wide<true, true>(h, ldh, w, nullptr, M, K, nullptr, d_values, 0.f, dh, lddh, dw, db, nullptr, h_parts,
                                   h_pstride, dh_parts, dh_pstride, s);
}
