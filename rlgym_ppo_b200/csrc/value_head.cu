// Value head: the last Linear(K,1) of ValueEstimator (value_estimator.py:27), its MSE loss (ppo_learner.py:176)
// and the backward into the last hidden activation, as one fused SIMT pass.  A 1-wide output would waste a
// 128xN tensor-core tile, and this pass is HBM-bound anyway: it reads H[M,K] once (2K bytes/row) and, when
// training, writes dH[M,K] once.
//   v = H w + b;  dv = 2*inv_batch*(v - target);  dH = dv * w (.) (H > 0);  dw += sum_m dv*H;  db += sum dv.
// UPSTREAM (rlppo_value_head_backward): the same pass with dv = d_values[row] loaded -- the backward of
// ValueEstimator.forward for an arbitrary upstream gradient (value_estimator.py:30-36).
#include "common.cuh"

namespace {

constexpr int kThreads = 256;
constexpr int kWarps = kThreads / 32;

// NI = number of 16-byte (8 x bf16) chunks each lane owns: K <= NI * 256
template <int NI, bool TRAIN, bool UPSTREAM = false>
__global__ void __launch_bounds__(kThreads)
value_head_kernel(const uint16_t* __restrict__ h, int64_t ldh, const float* __restrict__ w, const float* __restrict__ bias,
                  int64_t M, int K, float* __restrict__ values_out, const float* __restrict__ targets, float inv_batch,
                  uint16_t* __restrict__ dh, int64_t lddh, float* __restrict__ dw, float* __restrict__ db,
                  float* __restrict__ metrics, int h_parts, int64_t h_pstride, int dh_parts, int64_t dh_pstride) {
    // UPSTREAM: `targets` holds d_values
    extern __shared__ float s_mem[];   // [K] dw partials (TRAIN)
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int nvec = K >> 3;
    float wreg[NI][8];
#pragma unroll
    for (int i = 0; i < NI; ++i) {
        const int c = lane + 32 * i;
#pragma unroll
        for (int j = 0; j < 8; ++j) wreg[i][j] = (c < nvec) ? __ldg(w + c * 8 + j) : 0.f;
    }
    const float b = bias ? __ldg(bias) : 0.f;
    float gw[NI][8];
#pragma unroll
    for (int i = 0; i < NI; ++i)
#pragma unroll
        for (int j = 0; j < 8; ++j) gw[i][j] = 0.f;
    float sum_dv = 0.f, sum_sq = 0.f, rows = 0.f;
    if (TRAIN) {
        for (int i = threadIdx.x; i < K; i += kThreads) s_mem[i] = 0.f;
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

template <int NI>
int launch(const uint16_t* h, int64_t ldh, const float* w, const float* bias, int64_t M, int K, float* values_out,
           const float* targets, float inv_batch, uint16_t* dh, int64_t lddh, float* dw, float* db, float* metrics,
           int h_parts, int64_t h_pstride, int dh_parts, int64_t dh_pstride, cudaStream_t s, bool upstream = false) {
    const int64_t want = (M + kWarps - 1) / kWarps;
    const int64_t cap = (int64_t)rlppo::num_sms() * 8;
    const unsigned grid = (unsigned)(want < cap ? want : cap);
    if (upstream)
        value_head_kernel<NI, true, true><<<grid, kThreads, K * sizeof(float), s>>>(h, ldh, w, nullptr, M, K, nullptr,
                                                                                   targets, 0.f, dh, lddh, dw, db, nullptr,
                                                                                   h_parts, h_pstride, dh_parts, dh_pstride);
    else if (targets != nullptr)
        value_head_kernel<NI, true><<<grid, kThreads, K * sizeof(float), s>>>(h, ldh, w, bias, M, K, values_out, targets,
                                                                             inv_batch, dh, lddh, dw, db, metrics,
                                                                             h_parts, h_pstride, dh_parts, dh_pstride);
    else
        value_head_kernel<NI, false><<<grid, kThreads, 0, s>>>(h, ldh, w, bias, M, K, values_out, nullptr, 0.f, nullptr, 0,
                                                               nullptr, nullptr, nullptr, h_parts, h_pstride, 1, 0);
    RLPPO_LAUNCH_CHECK();
    return RLPPO_OK;
}

}  // namespace

extern "C" int rlppo_value_head(const uint16_t* h, int64_t ldh, const float* w, const float* bias, int64_t M, int K,
                                float* values_out, const float* targets, float inv_batch, uint16_t* dh, int64_t lddh,
                                float* dw, float* db, float* metrics, int h_parts, int64_t h_pstride, int dh_parts,
                                int64_t dh_pstride, void* stream) {
    RLPPO_REQUIRE_DEVICE();
    RLPPO_CHECK_ARG(h && w && M >= 1, "bad argument");
    RLPPO_CHECK_ARG(K % 8 == 0 && K >= 8 && K <= 2048 && ldh % 8 == 0, "K must be a multiple of 8 in [8,2048]");
    RLPPO_CHECK_ARG((reinterpret_cast<uintptr_t>(h) & 15) == 0, "H must be 16-byte aligned");
    RLPPO_CHECK_ARG(h_parts >= 1 && h_parts <= 3 && dh_parts >= 1 && dh_parts <= 3 && h_pstride % 8 == 0 &&
                        dh_pstride % 8 == 0 && (h_parts == 1 || h_pstride >= K) && (dh_parts == 1 || dh_pstride >= K),
                    "split: 1..3 parts, strides multiples of 8 covering K");
    if (targets != nullptr) {
        RLPPO_CHECK_ARG(dh && dw && lddh % 8 == 0 && lddh >= K, "training mode needs dh (ld %% 8) and dw");
        RLPPO_CHECK_ARG((reinterpret_cast<uintptr_t>(dh) & 15) == 0, "dH must be 16-byte aligned");
    }
    cudaStream_t s = static_cast<cudaStream_t>(stream);
#define RLPPO_VH(NI_) launch<NI_>(h, ldh, w, bias, M, K, values_out, targets, inv_batch, dh, lddh, dw, db, metrics, h_parts, \
                                  h_pstride, dh_parts, dh_pstride, s)
    if (K <= 256) return RLPPO_VH(1);
    if (K <= 512) return RLPPO_VH(2);
    if (K <= 1024) return RLPPO_VH(4);
    return RLPPO_VH(8);
#undef RLPPO_VH
}

// Backward of ValueEstimator.forward (value_estimator.py:27, the last Linear(K,1) over ReLU activations H) for an
// arbitrary upstream gradient d_values f32[M] (device): dH = dv * w (.) (H > 0), dw[K] += sum_m dv*H, db[1] += sum dv.
extern "C" int rlppo_value_head_backward(const uint16_t* h, int64_t ldh, const float* w, int64_t M, int K,
                                         const float* d_values, uint16_t* dh, int64_t lddh, float* dw, float* db,
                                         int h_parts, int64_t h_pstride, int dh_parts, int64_t dh_pstride, void* stream) {
    RLPPO_REQUIRE_DEVICE();
    RLPPO_CHECK_ARG(h && w && d_values && dh && dw && M >= 1, "bad argument");
    RLPPO_CHECK_ARG(K % 8 == 0 && K >= 8 && K <= 2048 && ldh % 8 == 0, "K must be a multiple of 8 in [8,2048]");
    RLPPO_CHECK_ARG((reinterpret_cast<uintptr_t>(h) & 15) == 0 && (reinterpret_cast<uintptr_t>(dh) & 15) == 0,
                    "H and dH must be 16-byte aligned");
    RLPPO_CHECK_ARG(lddh % 8 == 0 && lddh >= K, "lddh must be a multiple of 8 covering K");
    RLPPO_CHECK_ARG(h_parts >= 1 && h_parts <= 3 && dh_parts >= 1 && dh_parts <= 3 && h_pstride % 8 == 0 &&
                        dh_pstride % 8 == 0 && (h_parts == 1 || h_pstride >= K) && (dh_parts == 1 || dh_pstride >= K),
                    "split: 1..3 parts, strides multiples of 8 covering K");
    cudaStream_t s = static_cast<cudaStream_t>(stream);
#define RLPPO_VHB(NI_) launch<NI_>(h, ldh, w, nullptr, M, K, nullptr, d_values, 0.f, dh, lddh, dw, db, nullptr, h_parts, \
                                   h_pstride, dh_parts, dh_pstride, s, true)
    if (K <= 256) return RLPPO_VHB(1);
    if (K <= 512) return RLPPO_VHB(2);
    if (K <= 1024) return RLPPO_VHB(4);
    return RLPPO_VHB(8);
#undef RLPPO_VHB
}
