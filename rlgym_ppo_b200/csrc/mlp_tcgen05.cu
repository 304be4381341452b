// Policy / value MLP GEMMs on the 5th-generation tensor cores (tcgen05 + TMEM + TMA), replacing the
// nn.Sequential Linear/ReLU/Softmax stacks of discrete_policy.py:22-42 and value_estimator.py:19-36 and their
// autograd backward (ppo_learner.py:179-180).
//
// Two kernels:
//  (I)  rowgemm_kernel  C[M,N] = A[M,K] * B[N,K]^T, both operands K-major.  Persistent over 128-row tiles:
//         warp 0  : TMA producer (4-stage smem ring, 128B-swizzled tiles, mbarrier full/empty)
//         warp 1  : allocates TMEM, then one thread issues tcgen05.mma (128 x BLOCK_N x 16, bf16 -> fp32)
//         warps 2-5: epilogue; each thread owns one row of the 128-lane TMEM accumulator (double buffered, so
//                   the epilogue of tile i overlaps the MMAs of tile i+1) and applies one of
//           EPI_BIAS_ACT    y = relu?(acc + bias) -> bf16                         (forward hidden layers)
//           EPI_RELU_MASK   dx = acc * (h_prev > 0) -> bf16                       (dgrad through ReLU)
//           EPI_HEAD_SAMPLE softmax -> clamp -> inverse-CDF sample -> log-prob    (DiscreteFF.get_action)
//           EPI_HEAD_TRAIN  softmax/clamp/log-prob/entropy/ratio/clip/KL/clip-fraction and d(loss)/d(logits)
//           EPI_HEAD_BWD    d(logits) from arbitrary upstream gradients of log-prob / mean entropy / probabilities
//                           (get_backprop_data + ppo_learner.py:153-177 + SURVEY A.3), dz -> bf16
//  (II) wgrad_kernel    dW[N,K] += dY[M,N]^T * X[M,K]: both operands MN-major (the contraction runs over rows),
//         split over M across all SMs, fp32 accumulation in TMEM, coalesced fp32 atomics into the grad arena.
#include <mutex>
#include <unordered_map>
#include <math.h>

#include <stdlib.h>

#include "tc_common.cuh"

namespace rlppo {
namespace tc {

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn get_encode_fn() {
    static EncodeTiledFn fn = nullptr;
    if (fn == nullptr) {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
            q == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<EncodeTiledFn>(p);
    }
    return fn;
}

int make_tmap_bf16_2d(CUtensorMap* out, const void* base, uint64_t rows, uint64_t cols, uint64_t ld,
                      uint32_t box_rows) {
    EncodeTiledFn fn = get_encode_fn();
    if (fn == nullptr) {
        set_error("cuTensorMapEncodeTiled not available from the driver");
        return RLPPO_ERR_CUDA;
    }
    RLPPO_CHECK_ARG((reinterpret_cast<uintptr_t>(base) & 15) == 0, "TMA operand must be 16-byte aligned");
    RLPPO_CHECK_ARG((ld * 2) % 16 == 0 && cols <= ld && cols >= 1 && rows >= 1, "TMA operand: ld must be a multiple of 8");
    RLPPO_CHECK_ARG(box_rows >= 1 && box_rows <= 256, "TMA box rows out of range");
    // A descriptor is a pure function of these five values, and an eager training step asks for the same ~50 of them at
    // every launch (the driver call costs ~1 us each: a quarter of the fused kernel's own duration): keep them.
    struct Key {
        const void* base;
        uint64_t rows, cols, ld;
        uint32_t box_rows;
        bool operator==(const Key& o) const {
            return base == o.base && rows == o.rows && cols == o.cols && ld == o.ld && box_rows == o.box_rows;
        }
    };
    struct KeyHash {
        size_t operator()(const Key& k) const {
            uint64_t h = reinterpret_cast<uintptr_t>(k.base) * 0x9E3779B97F4A7C15ull;
            h ^= (k.rows + 0x9E3779B97F4A7C15ull + (h << 6) + (h >> 2));
            h ^= (k.cols * 0xC2B2AE3D27D4EB4Full + (h << 6) + (h >> 2));
            h ^= (k.ld * 0x165667B19E3779F9ull + (h << 6) + (h >> 2));
            return (size_t)(h ^ k.box_rows);
        }
    };
    static std::mutex mu;
    static std::unordered_map<Key, CUtensorMap, KeyHash> cache;
    const Key key{base, rows, cols, ld, box_rows};
    {
        std::lock_guard<std::mutex> lock(mu);
        auto it = cache.find(key);
        if (it != cache.end()) {
            *out = it->second;
            return RLPPO_OK;
        }
    }
    cuuint64_t gdim[2] = {cols, rows};
    cuuint64_t gstride[1] = {ld * 2};
    cuuint32_t box[2] = {64, box_rows};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = fn(out, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), gdim, gstride, box, estr,
                    CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                    CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
        set_error("cuTensorMapEncodeTiled failed with CUresult %d (rows=%llu cols=%llu ld=%llu box_rows=%u)", (int)r,
                  (unsigned long long)rows, (unsigned long long)cols, (unsigned long long)ld, box_rows);
        return RLPPO_ERR_CUDA;
    }
    {
        std::lock_guard<std::mutex> lock(mu);
        if (cache.size() >= 4096) cache.clear();      // (workspaces that were reallocated leave stale keys behind)
        cache.emplace(key, *out);
    }
    return RLPPO_OK;
}

}  // namespace tc
}  // namespace rlppo

namespace {

using namespace rlppo;
using namespace rlppo::tc;

constexpr int BLOCK_M = 128;
constexpr int BLOCK_K = 64;  // 64 bf16 = one 128-byte swizzle row
constexpr int UMMA_K = 16;
constexpr int kStages = 4;
constexpr int kThreads = 192;
constexpr uint32_t A_BYTES = BLOCK_M * BLOCK_K * 2;  // 16 KB

enum { EPI_BIAS_ACT = 0, EPI_RELU_MASK = 1, EPI_HEAD_SAMPLE = 2, EPI_HEAD_TRAIN = 3, EPI_HEAD_BWD = 4 };

// Split ("fp32-exact") operands: a logical f32 matrix is stored as `parts` bf16 matrices side by side in one buffer
// (part q in columns [q * pstride, q * pstride + cols), value = part0 + part1 + ...; see rlppo_split in rlppo.h).  A GEMM
// over split operands is the SAME kernel running a longer k loop: schedule entry s pairs part a_off[s] of A with part
// b_off[s] of B (column offsets in elements); all products land in one fp32 TMEM accumulator, smallest terms first.
constexpr int MAX_SCHED = 6;
struct KSched {
    int n;                  // entries (0 = plain single-part operands)
    int kpp;                // 64-wide k-blocks per entry
    int a_off[MAX_SCHED];
    int b_off[MAX_SCHED];
};

struct RowGemmParams {
    int64_t M;
    int N, K;
    int num_m_tiles, num_n_tiles, num_k_blocks;
    KSched sched;
    int out_parts;          // 1 (plain bf16 output) .. 3: the f32 result is written as hi / mid / lo bf16 parts
    int64_t out_pstride;    // column offset between consecutive output parts (elements)
    int out_cols;           // heads: columns of d(logits) to write per part (padding columns are written as zeros)
    // bias/act and relu-mask epilogues
    uint16_t* out;
    int64_t ldo;
    const float* bias;
    int bias_n;             // entries of `bias` (<= N; columns past it take no bias)
    int relu;
    const uint16_t* mask;
    int64_t ldmask;
    float* colsum;   // EPI_RELU_MASK: optional f32[N], += column sums of the bf16 output (= bias gradient of the layer below)
    // heads
    int n_actions;
    const float* actions;
    const float* old_logp;
    const float* adv;
    float inv_batch, clip, ent_coef;
    float* logp_out;
    float* metrics;
    const float* u_inject;
    uint64_t seed, offset;
    int deterministic;
    float* actions_out;
    int64_t* actions_i64_out;
    float* probs_out;
    // EPI_HEAD_BWD: upstream gradients (each optional)
    const float* d_logp;
    const float* d_ent;
    const float* d_probs;
};

__device__ __forceinline__ uint4 philox4x32_10(uint4 c, uint2 k) {
#pragma unroll
    for (int i = 0; i < 10; ++i) {
        const uint32_t hi0 = __umulhi(0xD2511F53u, c.x), lo0 = 0xD2511F53u * c.x;
        const uint32_t hi1 = __umulhi(0xCD9E8D57u, c.z), lo1 = 0xCD9E8D57u * c.z;
        c = make_uint4(hi1 ^ c.y ^ k.x, lo1, hi0 ^ c.w ^ k.y, lo0);
        k.x += 0x9E3779B9u;
        k.y += 0xBB67AE85u;
    }
    return c;
}

template <int BLOCK_N>
struct SmemLayout {
    static constexpr uint32_t B_BYTES = BLOCK_N * BLOCK_K * 2;
    static constexpr uint32_t STAGE = A_BYTES + B_BYTES;
    static constexpr uint32_t BAR_OFF = kStages * STAGE;
    static constexpr uint32_t BIAS_OFF = BAR_OFF + 256;
    static constexpr uint32_t AUX_FLOATS = 4096;   // bias vector of the whole layer (EPI_BIAS_ACT) / per-tile scratch
    static constexpr uint32_t TOTAL = BIAS_OFF + AUX_FLOATS * 4 + 1024;  // + slack for 1024-byte alignment
};

// ---------------------------------------------------------------------------------------------------------
// epilogues (one thread = one output row; `trow` = TMEM address of that row's first accumulator column)
// ---------------------------------------------------------------------------------------------------------
// lane j returns sum over the 32 lanes of v[j] (v is destroyed): a 31-shuffle reduce-scatter
__device__ __forceinline__ float warp_colsum32_rg(float (&v)[32], int lane) {
#pragma unroll
    for (int w = 16; w >= 1; w >>= 1) {
        const bool up = (lane & w) != 0;
#pragma unroll
        for (int i = 0; i < w; ++i) {
            const float send = up ? v[i] : v[i + w];
            const float keep = up ? v[i + w] : v[i];
            v[i] = keep + __shfl_xor_sync(0xffffffffu, send, w);
        }
    }
    return v[0];
}

// The accumulator chunk and (dgrad) the ReLU-mask vectors of chunk c+1 are requested before chunk c is processed, and
// the forward bias comes from shared memory (the whole layer's vector, loaded once per CTA): ncu on the first version
// showed 52 % of this kernel's stall samples on the FADDs waiting for per-element __ldg(bias) / mask loads, and an
// epilogue of ~12 us per 128x256 tile -- as long as the MMAs of a K = 1024 tile it is supposed to hide behind.
template <int EPI>
__device__ __forceinline__ void epilogue_store_bf16(const RowGemmParams& p, uint32_t trow, int64_t row, int n0,
                                                    int n_valid, float* s_aux, int lane) {
    const int nch = (n_valid + 31) >> 5;
    const bool row_ok = row < p.M;
    const bool want_sum = EPI == EPI_RELU_MASK && p.colsum != nullptr;
    const bool bias_smem = EPI == EPI_BIAS_ACT && p.bias != nullptr && p.N <= 4096;
    const bool use_mask = EPI == EPI_RELU_MASK && p.mask != nullptr;
    uint32_t rb[32];
    uint4 mk_next[4];
    auto fetch_mask = [&](int c) {
#pragma unroll
        for (int g = 0; g < 4; ++g) {
            const int col = n0 + c * 32 + g * 8;
            mk_next[g] = (use_mask && row_ok && col + 8 <= p.N)
                             ? __ldg(reinterpret_cast<const uint4*>(p.mask + row * p.ldmask + col))
                             : make_uint4(0u, 0u, 0u, 0u);
        }
    };
    tmem_ld32_issue(trow, rb);
    fetch_mask(0);
    for (int c = 0; c < nch; ++c) {
        float v[32];
        uint4 mk[4];
        tmem_ld32_wait(rb);
#pragma unroll
        for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(rb[i]);
#pragma unroll
        for (int g = 0; g < 4; ++g) mk[g] = mk_next[g];
        if (c + 1 < nch) {
            tmem_ld32_issue(trow + (c + 1) * 32, rb);
            fetch_mask(c + 1);
        }
        if (!row_ok && !want_sum) continue;
#pragma unroll
        for (int g = 0; g < 4; ++g) {
            const int col = n0 + c * 32 + g * 8;
            float x[8];
#pragma unroll
            for (int j = 0; j < 8; ++j) x[j] = v[g * 8 + j];
            if (!row_ok || col + 8 > p.N) {
#pragma unroll
                for (int j = 0; j < 8; ++j) v[g * 8 + j] = 0.f;
                continue;
            }
            if (EPI == EPI_BIAS_ACT) {
                if (bias_smem) {
                    const float4 b0 = *reinterpret_cast<const float4*>(s_aux + col);
                    const float4 b1 = *reinterpret_cast<const float4*>(s_aux + col + 4);
                    x[0] += b0.x; x[1] += b0.y; x[2] += b0.z; x[3] += b0.w;
                    x[4] += b1.x; x[5] += b1.y; x[6] += b1.z; x[7] += b1.w;
                } else if (p.bias != nullptr) {
#pragma unroll
                    for (int j = 0; j < 8; ++j) x[j] += col + j < p.bias_n ? __ldg(p.bias + col + j) : 0.f;
                }
                if (p.relu) {
#pragma unroll
                    for (int j = 0; j < 8; ++j) x[j] = fmaxf(x[j], 0.f);
                }
            } else {  // EPI_RELU_MASK
                if (use_mask) {
                    const uint32_t w[4] = {mk[g].x, mk[g].y, mk[g].z, mk[g].w};
#pragma unroll
                    for (int j = 0; j < 8; ++j) {
                        const uint32_t bits = (w[j >> 1] >> ((j & 1) * 16)) & 0xFFFFu;
                        const bool pos = (bits & 0x7FFFu) != 0 && (bits & 0x8000u) == 0;
                        x[j] = pos ? x[j] : 0.f;
                    }
                }
            }
            uint4 o;
            o.x = pack_bf16x2(x[0], x[1]);
            o.y = pack_bf16x2(x[2], x[3]);
            o.z = pack_bf16x2(x[4], x[5]);
            o.w = pack_bf16x2(x[6], x[7]);
            *reinterpret_cast<uint4*>(p.out + row * p.ldo + col) = o;
            if (p.out_parts > 1) {
                // split output: part q = bf16(x - part_0 - ... - part_{q-1}); the column sums take the f32 values
                if (want_sum) {
#pragma unroll
                    for (int j = 0; j < 8; ++j) v[g * 8 + j] = x[j];
                }
                for (int q = 1; q < p.out_parts; ++q) {
                    const uint32_t ow[4] = {o.x, o.y, o.z, o.w};
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        x[2 * j] -= __uint_as_float(ow[j] << 16);
                        x[2 * j + 1] -= __uint_as_float(ow[j] & 0xFFFF0000u);
                    }
                    o.x = pack_bf16x2(x[0], x[1]);
                    o.y = pack_bf16x2(x[2], x[3]);
                    o.z = pack_bf16x2(x[4], x[5]);
                    o.w = pack_bf16x2(x[6], x[7]);
                    *reinterpret_cast<uint4*>(p.out + row * p.ldo + q * p.out_pstride + col) = o;
                }
            } else if (want_sum) {
                // sum what was STORED (bf16-rounded): the same values the separate column-sum pass used to read back
                const uint32_t ow[4] = {o.x, o.y, o.z, o.w};
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    v[g * 8 + 2 * j] = __uint_as_float(ow[j] << 16);
                    v[g * 8 + 2 * j + 1] = __uint_as_float(ow[j] & 0xFFFF0000u);
                }
            }
        }
        if (want_sum) {
            const float cs = warp_colsum32_rg(v, lane);          // lane j: column c*32+j over this warp's 32 rows
            atomicAdd(&s_aux[c * 32 + lane], cs);                // four row-quarter warps add into the same word
        }
    }
}

__device__ __forceinline__ void head_max_sum(uint32_t trow, const float* s_bias, int nact, int nch, float& mx,
                                             float& S, int& argmax) {
    mx = -INFINITY;
    argmax = 0;
    for (int c = 0; c < nch; ++c) {
        float v[32];
        tmem_ld32(trow + c * 32, v);
#pragma unroll
        for (int j = 0; j < 32; ++j) {
            const int col = c * 32 + j;
            if (col < nact) {
                const float z = v[j] + s_bias[col];
                if (z > mx) {
                    mx = z;
                    argmax = col;
                }
            }
        }
    }
    S = 0.f;
    for (int c = 0; c < nch; ++c) {
        float v[32];
        tmem_ld32(trow + c * 32, v);
#pragma unroll
        for (int j = 0; j < 32; ++j) {
            const int col = c * 32 + j;
            if (col < nact) S += __expf(v[j] + s_bias[col] - mx);
        }
    }
}

// DiscreteFF.get_action (discrete_policy.py:44-62)
__device__ __forceinline__ void epilogue_head_sample(const RowGemmParams& p, uint32_t trow, int64_t row,
                                                     const float* s_bias) {
    const int nact = p.n_actions;
    const int nch = (nact + 31) >> 5;
    const bool row_ok = row < p.M;
    float mx, S;
    int argmax;
    head_max_sum(trow, s_bias, nact, nch, mx, S, argmax);
    const float invS = 1.0f / S;
    // total clamped mass (torch.multinomial normalises whatever it is given)
    float P = 0.f;
    for (int c = 0; c < nch; ++c) {
        float v[32];
        tmem_ld32(trow + c * 32, v);
#pragma unroll
        for (int j = 0; j < 32; ++j) {
            const int col = c * 32 + j;
            if (col < nact) {
                const float s = __expf(v[j] + s_bias[col] - mx) * invS;
                P += fminf(fmaxf(s, 1e-11f), 1.0f);                                   // :54
                if (p.probs_out != nullptr && row_ok) p.probs_out[row * nact + col] = s;  // get_output (:35-42)
            }
        }
    }
    float u = 0.f;
    if (row_ok) {
        if (p.u_inject != nullptr) {
            u = __ldg(p.u_inject + row);
        } else {
            const uint64_t ctr = p.offset + (uint64_t)row;
            const uint4 r = philox4x32_10(make_uint4((uint32_t)ctr, (uint32_t)(ctr >> 32), 0u, 0u),
                                          make_uint2((uint32_t)p.seed, (uint32_t)(p.seed >> 32)));
            u = (float)(r.x >> 8) * (1.0f / 16777216.0f);
        }
    }
    int act = nact - 1;
    float pa = 0.f;
    if (p.deterministic) {
        act = argmax;
        pa = fminf(fmaxf(invS, 1e-11f), 1.0f);   // exp(0)/S
    } else {
        const float thr = u * P;
        float run = 0.f, plast = 0.f;
        bool found = false;
        for (int c = 0; c < nch; ++c) {
            float v[32];
            tmem_ld32(trow + c * 32, v);
#pragma unroll
            for (int j = 0; j < 32; ++j) {
                const int col = c * 32 + j;
                if (col < nact) {
                    const float s = __expf(v[j] + s_bias[col] - mx) * invS;
                    const float pj = fminf(fmaxf(s, 1e-11f), 1.0f);
                    run += pj;
                    plast = pj;
                    if (!found && run > thr) {
                        found = true;
                        act = col;
                        pa = pj;
                    }
                }
            }
        }
        if (!found) pa = plast;
    }
    if (row_ok) {
        if (p.actions_out) p.actions_out[row] = (float)act;          // batched_agent_manager.py:204
        if (p.actions_i64_out) p.actions_i64_out[row] = (int64_t)act;
        if (p.logp_out) p.logp_out[row] = logf(pa);                  // :60
    }
}

// get_backprop_data (discrete_policy.py:64-80) + PPO loss (ppo_learner.py:153-177) + backward (SURVEY A.3).
// UPSTREAM (EPI_HEAD_BWD, rlppo_policy_head_backward): no loss block; the upstream gradients of the forward's outputs are
// loaded instead -- d_logp[row] of the gathered log-prob, d_ent[0] of the MEAN entropy (each row's share d_ent / M) and
// d_probs[row, j] of get_output's unclamped softmax (added outside the clamp mask: torch.clamp sits after it).
template <bool UPSTREAM>
__device__ __forceinline__ void epilogue_head_train(const RowGemmParams& p, uint32_t trow, int64_t row,
                                                    const float* s_bias, int lane) {
    const int nact = p.n_actions;
    const int nch = (nact + 31) >> 5;
    const bool row_ok = row < p.M;
    int a = 0;
    float old_lp = 0.f, advv = 0.f, up_lp = 0.f;
    if (row_ok) {
        if (UPSTREAM) {
            if (p.d_logp != nullptr) {
                a = (int)__ldg(p.actions + row);
                a = min(max(a, 0), nact - 1);
                up_lp = __ldg(p.d_logp + row);
            }
        } else {
            a = (int)__ldg(p.actions + row);                 // acts.long(), :71
            a = min(max(a, 0), nact - 1);
            old_lp = __ldg(p.old_logp + row);
            advv = __ldg(p.adv + row);
        }
    }
    float mx, S;
    int argmax;
    head_max_sum(trow, s_bias, nact, nch, mx, S, argmax);
    const float invS = 1.0f / S;

    // pass: entropy and the action's probability
    float H = 0.f, s_a = 0.f;
    for (int c = 0; c < nch; ++c) {
        float v[32];
        tmem_ld32(trow + c * 32, v);
#pragma unroll
        for (int j = 0; j < 32; ++j) {
            const int col = c * 32 + j;
            if (col < nact) {
                const float s = __expf(v[j] + s_bias[col] - mx) * invS;
                const float pj = fminf(fmaxf(s, 1e-11f), 1.0f);     // :74
                if (!UPSTREAM) H -= pj * __logf(pj);                // :78
                if (col == a) s_a = s;
            }
        }
    }
    const float p_a = fminf(fmaxf(s_a, 1e-11f), 1.0f);
    const float logp = logf(p_a);                                   // :76-77
    float ga, cw, kl = 0.f, clipc = 0.f, surr = 0.f;
    if (UPSTREAM) {
        ga = up_lp / p_a;                                           // dL/dp_a = d_logp / p_a
        cw = p.d_ent != nullptr ? -__ldg(p.d_ent) / (float)p.M : 0.f;   // dL/dp_j = -(d_ent/M)(log p_j + 1)
    } else {
        const float log_ratio = logp - old_lp;
        const float ratio = expf(log_ratio);                        // ppo_learner.py:153
        const float lo = 1.0f - p.clip, hi = 1.0f + p.clip;
        const float clipped = fminf(fmaxf(ratio, lo), hi);          // :154-156
        const float s1 = ratio * advv, s2 = clipped * advv;
        surr = fminf(s1, s2);                                       // :172-174
        kl = (ratio - 1.0f) - log_ratio;                            // :161
        clipc = fabsf(ratio - 1.0f) > p.clip ? 1.f : 0.f;           // :166
        // backward of -mean(min(s1,s2)): torch.minimum splits ties 0.5/0.5; clamp passes gradient inside [lo,hi]
        const float in_range = (ratio >= lo && ratio <= hi) ? 1.f : 0.f;
        const float d1 = s1 < s2 ? 1.f : (s1 == s2 ? 0.5f : 0.f);
        const float d2 = s1 > s2 ? 1.f : (s1 == s2 ? 0.5f : 0.f);
        const float d_logp = -p.inv_batch * advv * (d1 + d2 * in_range) * ratio;
        ga = d_logp / p_a;                   // dL/dp_a through the log-prob gather
        cw = p.ent_coef * p.inv_batch;       // dL/dp_j through -ent_coef * entropy: cw * (log p_j + 1)
    }
    const float* dpr = (UPSTREAM && row_ok && p.d_probs != nullptr) ? p.d_probs + row * nact : nullptr;

    // pass: G = sum_j g_j s_j
    float G = 0.f;
    for (int c = 0; c < nch; ++c) {
        float v[32];
        tmem_ld32(trow + c * 32, v);
#pragma unroll
        for (int j = 0; j < 32; ++j) {
            const int col = c * 32 + j;
            if (col < nact) {
                const float s = __expf(v[j] + s_bias[col] - mx) * invS;
                const float pj = fminf(fmaxf(s, 1e-11f), 1.0f);
                float g = cw * (__logf(pj) + 1.0f) + (col == a ? ga : 0.f);
                g = (s >= 1e-11f && s <= 1.0f) ? g : 0.f;            // clamp mask
                if (UPSTREAM && dpr != nullptr) g += __ldg(dpr + col);
                G += g * s;
            }
        }
    }
    // pass: dz_j = s_j (g_j - G) -> bf16 (padding columns up to lddz are written as zeros)
    const int ncols_out = p.out_cols;
    const int nch_out = (ncols_out + 31) >> 5;
    for (int c = 0; c < nch_out; ++c) {
        float v[32];
        tmem_ld32(trow + c * 32, v);
        if (!row_ok) continue;
        float dz[32];
#pragma unroll
        for (int j = 0; j < 32; ++j) {
            const int col = c * 32 + j;
            float o = 0.f;
            if (col < nact) {
                const float s = __expf(v[j] + s_bias[col] - mx) * invS;
                const float pj = fminf(fmaxf(s, 1e-11f), 1.0f);
                float g = cw * (__logf(pj) + 1.0f) + (col == a ? ga : 0.f);
                g = (s >= 1e-11f && s <= 1.0f) ? g : 0.f;
                if (UPSTREAM && dpr != nullptr) g += __ldg(dpr + col);
                o = s * (g - G);
            }
            dz[j] = o;
        }
#pragma unroll
        for (int g8 = 0; g8 < 4; ++g8) {
            const int col = c * 32 + g8 * 8;
            if (col + 8 > ncols_out) continue;
            uint4 o;
            o.x = pack_bf16x2(dz[g8 * 8 + 0], dz[g8 * 8 + 1]);
            o.y = pack_bf16x2(dz[g8 * 8 + 2], dz[g8 * 8 + 3]);
            o.z = pack_bf16x2(dz[g8 * 8 + 4], dz[g8 * 8 + 5]);
            o.w = pack_bf16x2(dz[g8 * 8 + 6], dz[g8 * 8 + 7]);
            *reinterpret_cast<uint4*>(p.out + row * p.ldo + col) = o;
            for (int q = 1; q < p.out_parts; ++q) {
                const uint32_t ow[4] = {o.x, o.y, o.z, o.w};
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    dz[g8 * 8 + 2 * j] -= __uint_as_float(ow[j] << 16);
                    dz[g8 * 8 + 2 * j + 1] -= __uint_as_float(ow[j] & 0xFFFF0000u);
                }
                o.x = pack_bf16x2(dz[g8 * 8 + 0], dz[g8 * 8 + 1]);
                o.y = pack_bf16x2(dz[g8 * 8 + 2], dz[g8 * 8 + 3]);
                o.z = pack_bf16x2(dz[g8 * 8 + 4], dz[g8 * 8 + 5]);
                o.w = pack_bf16x2(dz[g8 * 8 + 6], dz[g8 * 8 + 7]);
                *reinterpret_cast<uint4*>(p.out + row * p.ldo + q * p.out_pstride + col) = o;
            }
        }
    }
    if (UPSTREAM) return;
    if (row_ok && p.logp_out) p.logp_out[row] = logp;
    // metrics: one atomic per warp and quantity
    const float okf = row_ok ? 1.f : 0.f;
    const float mH = warp_sum(H * okf), mkl = warp_sum(kl * okf), mcl = warp_sum(clipc * okf),
                msu = warp_sum(surr * okf), mrows = warp_sum(okf);
    if (lane == 0 && p.metrics != nullptr && mrows > 0.f) {
        atomicAdd(p.metrics + 0, mH);
        atomicAdd(p.metrics + 1, mkl);
        atomicAdd(p.metrics + 2, mcl);
        atomicAdd(p.metrics + 3, msu);
        atomicAdd(p.metrics + 4, mrows);
    }
}

// ---------------------------------------------------------------------------------------------------------
// (I) C[M,N] = A[M,K] * B[N,K]^T
// ---------------------------------------------------------------------------------------------------------
template <int BLOCK_N, int EPI>
__global__ void __launch_bounds__(kThreads, 1)
rowgemm_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB, RowGemmParams p) {
    using L = SmemLayout<BLOCK_N>;
    constexpr uint32_t TMEM_COLS = 2 * BLOCK_N;  // two accumulator stages
    static_assert(TMEM_COLS >= 32 && TMEM_COLS <= 512 && (TMEM_COLS & (TMEM_COLS - 1)) == 0, "TMEM columns");
    static_assert(BLOCK_N % 16 == 0 && BLOCK_N >= 16 && BLOCK_N <= 256, "UMMA N");

    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
    uint64_t* full = reinterpret_cast<uint64_t*>(smem + L::BAR_OFF);
    uint64_t* empty = full + kStages;
    uint64_t* tfull = empty + kStages;
    uint64_t* tempty = tfull + 2;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty + 2);
    float* s_bias = reinterpret_cast<float*>(smem + L::BIAS_OFF);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (threadIdx.x == 0) {
        tma_prefetch_desc(&tmA);
        tma_prefetch_desc(&tmB);
        for (int i = 0; i < kStages; ++i) {
            mbar_init(&full[i], 1);
            mbar_init(&empty[i], 1);
        }
        for (int i = 0; i < 2; ++i) {
            mbar_init(&tfull[i], 1);
            mbar_init(&tempty[i], 4);
        }
        fence_barrier_init();
    }
    if (warp == 1) tmem_alloc(tmem_slot, TMEM_COLS);
    if (EPI == EPI_HEAD_SAMPLE || EPI == EPI_HEAD_TRAIN || EPI == EPI_HEAD_BWD) {
        for (int i = threadIdx.x; i < BLOCK_N; i += kThreads)
            s_bias[i] = (i < p.n_actions && p.bias != nullptr) ? __ldg(p.bias + i) : 0.f;
    } else if (EPI == EPI_RELU_MASK) {
        for (int i = threadIdx.x; i < BLOCK_N; i += kThreads) s_bias[i] = 0.f;     // column-sum accumulators
    } else if (EPI == EPI_BIAS_ACT) {
        if (p.bias != nullptr && p.N <= (int)L::AUX_FLOATS)                        // the whole layer's bias vector
            for (int i = threadIdx.x; i < (int)L::AUX_FLOATS; i += kThreads) s_bias[i] = i < p.bias_n ? __ldg(p.bias + i) : 0.f;
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    const int total_tiles = p.num_m_tiles * p.num_n_tiles;

    if (warp == 0) {
        if (lane == 0) {
            uint32_t stage = 0, phase = 0;
            for (int t = blockIdx.x; t < total_tiles; t += gridDim.x) {
                const int m_blk = t / p.num_n_tiles, n_blk = t % p.num_n_tiles;
                int se = 0, sj = 0;       // schedule entry, k-block inside it
                for (int kb = 0; kb < p.num_k_blocks; ++kb) {
                    mbar_wait(&empty[stage], phase ^ 1);
                    mbar_expect_tx(&full[stage], L::STAGE);
                    uint8_t* sa = smem + stage * L::STAGE;
                    int ka = kb * BLOCK_K, kbb = kb * BLOCK_K;
                    if (p.sched.n > 0) {
                        ka = p.sched.a_off[se] + sj * BLOCK_K;
                        kbb = p.sched.b_off[se] + sj * BLOCK_K;
                        if (++sj == p.sched.kpp) {
                            sj = 0;
                            ++se;
                        }
                    }
                    tma_load_2d(&tmA, &full[stage], sa, ka, m_blk * BLOCK_M);
                    tma_load_2d(&tmB, &full[stage], sa + A_BYTES, kbb, n_blk * BLOCK_N);
                    if (++stage == kStages) {
                        stage = 0;
                        phase ^= 1;
                    }
                }
            }
        }
    } else if (warp == 1) {
        if (lane == 0) {
            constexpr uint32_t idesc = umma_idesc_bf16(BLOCK_M, BLOCK_N, 0, 0);
            uint32_t stage = 0, phase = 0, it = 0;
            for (int t = blockIdx.x; t < total_tiles; t += gridDim.x, ++it) {
                const uint32_t acc = it & 1, acc_phase = (it >> 1) & 1;
                mbar_wait(&tempty[acc], acc_phase ^ 1);
                tc_fence_after();
                const uint32_t d_tmem = tmem_base + acc * BLOCK_N;
                for (int kb = 0; kb < p.num_k_blocks; ++kb) {
                    mbar_wait(&full[stage], phase);
                    tc_fence_after();
                    const uint32_t a_addr = smem_u32(smem + stage * L::STAGE);
                    const uint32_t b_addr = a_addr + A_BYTES;
#pragma unroll
                    for (int k = 0; k < BLOCK_K / UMMA_K; ++k) {
                        const uint64_t ad = umma_smem_desc(a_addr + k * (UMMA_K * 2), 16, 1024);
                        const uint64_t bd = umma_smem_desc(b_addr + k * (UMMA_K * 2), 16, 1024);
                        umma_bf16(d_tmem, ad, bd, idesc, (kb | k) != 0 ? 1u : 0u);
                    }
                    umma_commit(&empty[stage]);  // smem slot is free once these MMAs have read it
                    if (++stage == kStages) {
                        stage = 0;
                        phase ^= 1;
                    }
                }
                umma_commit(&tfull[acc]);  // accumulator complete -> epilogue
            }
        }
    } else {
        const int ew = warp & 3;  // TMEM lane quarter this warp may access
        uint32_t it = 0;
        for (int t = blockIdx.x; t < total_tiles; t += gridDim.x, ++it) {
            const int m_blk = t / p.num_n_tiles, n_blk = t % p.num_n_tiles;
            const uint32_t acc = it & 1, acc_phase = (it >> 1) & 1;
            mbar_wait(&tfull[acc], acc_phase);
            tc_fence_after();
            const uint32_t trow = tmem_base + ((uint32_t)(ew * 32) << 16) + acc * BLOCK_N;
            const int64_t row = (int64_t)m_blk * BLOCK_M + ew * 32 + lane;
            if (EPI == EPI_BIAS_ACT || EPI == EPI_RELU_MASK) {
                const int n0 = n_blk * BLOCK_N;
                epilogue_store_bf16<EPI>(p, trow, row, n0, min(BLOCK_N, p.N - n0), s_bias, lane);
                if (EPI == EPI_RELU_MASK && p.colsum != nullptr) {
                    // flush this tile's column sums (bias gradient of the layer below) and clear the accumulators
                    asm volatile("bar.sync 2, 128;" ::: "memory");
                    const int et = threadIdx.x - 64;                    // 0..127 over the four epilogue warps
                    for (int j = et; j < BLOCK_N; j += 128) {
                        const float cs = s_bias[j];
                        s_bias[j] = 0.f;
                        if (n0 + j < p.N && cs != 0.f) atomicAdd(p.colsum + n0 + j, cs);
                    }
                    asm volatile("bar.sync 2, 128;" ::: "memory");
                }
            } else if (EPI == EPI_HEAD_SAMPLE) {
                epilogue_head_sample(p, trow, row, s_bias);
            } else {
                epilogue_head_train<EPI == EPI_HEAD_BWD>(p, trow, row, s_bias, lane);
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&tempty[acc]);
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        tc_fence_after();
        tmem_dealloc(tmem_base, TMEM_COLS);
    }
}

// ---------------------------------------------------------------------------------------------------------
// (II) dW[n,k] += sum_m dY[m,n] X[m,k].  TMEM holds the transposed tile (lane = k, column = n) so that the
// 32 lanes of a warp hit 32 consecutive floats of a dW row: coalesced fp32 atomics.
// ---------------------------------------------------------------------------------------------------------
struct WgradParams {
    int64_t M;
    int N, K;  // out features, in features (true, un-padded extents of dW)
    float* dw;
    int64_t lddw;
    int64_t m_per_split;  // multiple of BLOCK_K
    int splits, n_tiles_n, n_tiles_k;
    // split operands: per 64-row block, n_sched (X part, dY part) pairs accumulate into the same tile (0 = plain)
    int n_sched;
    int x_off[MAX_SCHED], dy_off[MAX_SCHED];
};

template <int BN>
__global__ void __launch_bounds__(kThreads, 1)
wgrad_kernel(const __grid_constant__ CUtensorMap tmX, const __grid_constant__ CUtensorMap tmDY, WgradParams p) {
    constexpr uint32_t CHUNK = 64 * BLOCK_K * 2;       // one TMA box: 64 MN-elements x 64 rows = 8 KB
    constexpr uint32_t XA_BYTES = 2 * CHUNK;           // 128 k
    constexpr uint32_t DY_BYTES = (BN / 64) * CHUNK;   // BN n
    constexpr uint32_t STAGE = XA_BYTES + DY_BYTES;
    constexpr uint32_t TMEM_COLS = BN < 32 ? 32 : BN;
    static_assert(BN % 64 == 0 && BN <= 256, "wgrad n tile");

    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
    uint64_t* full = reinterpret_cast<uint64_t*>(smem + kStages * STAGE);
    uint64_t* empty = full + kStages;
    uint64_t* tfull = empty + kStages;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tfull + 1);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (threadIdx.x == 0) {
        tma_prefetch_desc(&tmX);
        tma_prefetch_desc(&tmDY);
        for (int i = 0; i < kStages; ++i) {
            mbar_init(&full[i], 1);
            mbar_init(&empty[i], 1);
        }
        mbar_init(tfull, 1);
        fence_barrier_init();
    }
    if (warp == 1) tmem_alloc(tmem_slot, TMEM_COLS);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    const int split = blockIdx.x % p.splits;
    const int tile = blockIdx.x / p.splits;
    const int k_tile = tile % p.n_tiles_k, n_tile = tile / p.n_tiles_k;
    const int64_t m0 = (int64_t)split * p.m_per_split;
    const int64_t m1 = min(p.M, m0 + p.m_per_split);
    const int nkb = m1 > m0 ? (int)((m1 - m0 + BLOCK_K - 1) / BLOCK_K) : 0;

    const int nsch = p.n_sched > 0 ? p.n_sched : 1;
    if (warp == 0) {
        if (lane == 0) {
            uint32_t stage = 0, phase = 0;
            for (int kb = 0; kb < nkb; ++kb) {
              const int mrow = (int)(m0 + (int64_t)kb * BLOCK_K);
              for (int se = 0; se < nsch; ++se) {
                mbar_wait(&empty[stage], phase ^ 1);
                mbar_expect_tx(&full[stage], STAGE);
                uint8_t* sx = smem + stage * STAGE;
                const int xo = p.n_sched > 0 ? p.x_off[se] : 0, yo = p.n_sched > 0 ? p.dy_off[se] : 0;
#pragma unroll
                for (int c = 0; c < 2; ++c)
                    tma_load_2d(&tmX, &full[stage], sx + c * CHUNK, xo + k_tile * 128 + c * 64, mrow);
#pragma unroll
                for (int c = 0; c < BN / 64; ++c)
                    tma_load_2d(&tmDY, &full[stage], sx + XA_BYTES + c * CHUNK, yo + n_tile * BN + c * 64, mrow);
                if (++stage == kStages) {
                    stage = 0;
                    phase ^= 1;
                }
              }
            }
        }
    } else if (warp == 1) {
        if (lane == 0 && nkb > 0) {
            constexpr uint32_t idesc = umma_idesc_bf16(128, BN, 1, 1);  // both operands MN-major
            uint32_t stage = 0, phase = 0;
            for (int kb = 0; kb < nkb * nsch; ++kb) {
                mbar_wait(&full[stage], phase);
                tc_fence_after();
                const uint32_t a_addr = smem_u32(smem + stage * STAGE);
                const uint32_t b_addr = a_addr + XA_BYTES;
#pragma unroll
                for (int ks = 0; ks < BLOCK_K / UMMA_K; ++ks) {
                    // 16 contraction rows = 2 swizzle atoms of 8 rows x 128 B; MN chunks are CHUNK bytes apart
                    const uint64_t ad = umma_smem_desc(a_addr + ks * (UMMA_K * 128), CHUNK, 1024);
                    const uint64_t bd = umma_smem_desc(b_addr + ks * (UMMA_K * 128), CHUNK, 1024);
                    umma_bf16(tmem_base, ad, bd, idesc, (kb | ks) != 0 ? 1u : 0u);
                }
                umma_commit(&empty[stage]);
                if (++stage == kStages) {
                    stage = 0;
                    phase ^= 1;
                }
            }
            umma_commit(tfull);
        }
    } else if (nkb > 0) {
        const int ew = warp & 3;
        mbar_wait(tfull, 0);
        tc_fence_after();
        const uint32_t trow = tmem_base + ((uint32_t)(ew * 32) << 16);
        const int k = k_tile * 128 + ew * 32 + lane;
        const int n0 = n_tile * BN;
        const int nch = (min(BN, p.N - n0) + 31) >> 5;
        for (int c = 0; c < nch; ++c) {
            float v[32];
            tmem_ld32(trow + c * 32, v);
            if (k < p.K) {
#pragma unroll
                for (int j = 0; j < 32; ++j) {
                    const int n = n0 + c * 32 + j;
                    if (n < p.N) atomicAdd(p.dw + (int64_t)n * p.lddw + k, v[j]);
                }
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        tc_fence_after();
        tmem_dealloc(tmem_base, TMEM_COLS);
    }
}

// ---------------------------------------------------------------------------------------------------------
// (III) all weight gradients of a learner step in ONE persistent launch.
// Work item = (layer, 256-wide n tile, 256-wide k pair, row split).  Per 64-row block a CTA stages X [64 x <=256 k]
// and dY [64 x <=256 n] ONCE and issues up to two M=128 MMAs (the two 128-row k tiles) against the same dY tile, so
// dY is read once (the per-layer kernel above reads it once per k tile).  Row splits are sized from each layer's
// byte volume so that the ~148 items finish together.  HBM-bound: reads dY and X exactly once.
// Bias gradients ride along: while the MMA thread works on a stage, the four drain warps (idle until the item ends) add
// the staged dY tile's columns into registers (warp w: 64-column chunk w, lane: one bf16x2 column pair, conflict-free
// reads of the swizzled rows), so db_l = colsum(dY_l) costs no extra HBM traffic and no epilogue work in the fused
// kernel that produced dY.
// ---------------------------------------------------------------------------------------------------------
constexpr int MAXW = 8;
struct alignas(64) WMaps {
    CUtensorMap x[MAXW];
    CUtensorMap dy[MAXW];
};
struct WLayer {
    float* dw;
    float* db;      // optional: += column sums of dY (bias gradient), formed by the drain warps from the staged dY tiles
    int64_t lddw, M, m_per_split;
    int N, K, n_tiles_n, n_kpairs, splits, first_item;
};
struct WMultiParams {
    WLayer L[MAXW];
    int n_layers, total_items;
};

__global__ void __launch_bounds__(kThreads, 1)
wgrad_multi_kernel(const __grid_constant__ WMaps maps, const WMultiParams p) {
    constexpr uint32_t CHUNK = 64 * BLOCK_K * 2;       // 8 KB: 64 MN-elements x 64 rows
    constexpr uint32_t STAGE = 8 * CHUNK;              // X: 4 chunks (256 k), dY: 4 chunks (256 n)
    constexpr int NST = 3;

    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
    uint64_t* full = reinterpret_cast<uint64_t*>(smem + NST * STAGE);
    uint64_t* empty = full + NST;
    uint64_t* tfull = empty + NST;
    uint64_t* tempty = tfull + 1;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty + 1);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (threadIdx.x == 0) {
        for (int i = 0; i < NST; ++i) {
            mbar_init(&full[i], 1);
            mbar_init(&empty[i], 1 + 4);      // the MMA commit + the four drain warps (column sums read the dY tile)
        }
        mbar_init(tfull, 1);
        mbar_init(tempty, 4);
        fence_barrier_init();
    }
    if (warp == 1) tmem_alloc(tmem_slot, 512);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    pdl_wait();       // the operands are the previous kernel's outputs
    pdl_trigger();    // one item per CTA, all resident: the optimiser launch may be scheduled as items finish

    // decode a work item (identical in every role)
    struct Item {
        int layer, n0, k0, nkb, n_x, n_y, bn;
        int64_t m0;
    };
    auto decode = [&](int w) {
        Item it;
        int l = 0;
        while (l + 1 < p.n_layers && w >= p.L[l + 1].first_item) ++l;
        const WLayer& L = p.L[l];
        const int local = w - L.first_item;
        const int split = local % L.splits, tile = local / L.splits;
        const int kp = tile % L.n_kpairs, nt = tile / L.n_kpairs;
        it.layer = l;
        it.n0 = nt * 256;
        it.k0 = kp * 256;
        it.m0 = (int64_t)split * L.m_per_split;
        const int64_t m1 = min(L.M, it.m0 + L.m_per_split);
        it.nkb = m1 > it.m0 ? (int)((m1 - it.m0 + BLOCK_K - 1) / BLOCK_K) : 0;
        it.n_x = (min(256, L.K - it.k0) + 63) / 64;            // 64-wide k chunks that hold data
        it.n_y = (min(256, L.N - it.n0) + 63) / 64;
        it.bn = (min(256, L.N - it.n0) + 15) / 16 * 16;        // UMMA N
        return it;
    };

    if (warp == 0) {
        if (lane == 0) {
            uint32_t stage = 0, phase = 0;
            for (int w = blockIdx.x; w < p.total_items; w += gridDim.x) {
                const Item it = decode(w);
                for (int kb = 0; kb < it.nkb; ++kb) {
                    mbar_wait(&empty[stage], phase ^ 1);
                    mbar_expect_tx(&full[stage], (uint32_t)(it.n_x + it.n_y) * CHUNK);
                    uint8_t* sx = smem + stage * STAGE;
                    const int mrow = (int)(it.m0 + (int64_t)kb * BLOCK_K);
                    for (int c = 0; c < it.n_x; ++c)
                        tma_load_2d_hint(&maps.x[it.layer], &full[stage], sx + c * CHUNK, it.k0 + c * 64, mrow, L2_EVICT_FIRST);
                    for (int c = 0; c < it.n_y; ++c)
                        tma_load_2d_hint(&maps.dy[it.layer], &full[stage], sx + (4 + c) * CHUNK, it.n0 + c * 64, mrow, L2_EVICT_FIRST);
                    if (++stage == NST) {
                        stage = 0;
                        phase ^= 1;
                    }
                }
            }
        }
    } else if (warp == 1) {
        if (lane == 0) {
            uint32_t stage = 0, phase = 0, n_done = 0;
            for (int w = blockIdx.x; w < p.total_items; w += gridDim.x) {
                const Item it = decode(w);
                if (it.nkb == 0) continue;
                mbar_wait(tempty, (n_done & 1) ^ 1);       // the previous item's accumulators have been drained
                tc_fence_after();
                const uint32_t idesc = umma_idesc_bf16(128, it.bn, 1, 1);   // both operands MN-major
                const int n_kt = (it.n_x + 1) / 2;                           // 128-wide k tiles with data
                for (int kb = 0; kb < it.nkb; ++kb) {
                    mbar_wait(&full[stage], phase);
                    tc_fence_after();
                    const uint32_t x_addr = smem_u32(smem + stage * STAGE);
                    const uint32_t b_addr = x_addr + 4 * CHUNK;
                    for (int kt = 0; kt < n_kt; ++kt) {
#pragma unroll
                        for (int ks = 0; ks < BLOCK_K / UMMA_K; ++ks) {
                            const uint64_t ad = umma_smem_desc(x_addr + kt * 2 * CHUNK + ks * (UMMA_K * 128), CHUNK, 1024);
                            const uint64_t bd = umma_smem_desc(b_addr + ks * (UMMA_K * 128), CHUNK, 1024);
                            umma_bf16(tmem_base + kt * 256, ad, bd, idesc, (kb | ks) != 0 ? 1u : 0u);
                        }
                    }
                    umma_commit(&empty[stage]);
                    if (++stage == NST) {
                        stage = 0;
                        phase ^= 1;
                    }
                }
                umma_commit(tfull);
                ++n_done;
            }
        }
    } else {
        const int ew = warp & 3;
        uint32_t n_done = 0, stage = 0, phase = 0;
        for (int w = blockIdx.x; w < p.total_items; w += gridDim.x) {
            const Item it = decode(w);
            if (it.nkb == 0) continue;
            const WLayer& L = p.L[it.layer];
            // ---- column sums of the staged dY tiles (bias gradient), one stage behind the TMA like the MMA thread ----
            const bool want_db = L.db != nullptr && it.k0 == 0 && ew < it.n_y;
            float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
            for (int kb = 0; kb < it.nkb; ++kb) {
                mbar_wait(&full[stage], phase);
                if (want_db) {
                    const uint8_t* tile = smem + stage * STAGE + (4 + ew) * CHUNK;
                    const uint32_t sub = (uint32_t)(lane & 3) * 4u, c16 = (uint32_t)lane >> 2;
#pragma unroll 8
                    for (int r = 0; r < BLOCK_K; r += 2) {
                        const uint32_t w0 = *reinterpret_cast<const uint32_t*>(tile + r * 128 + ((c16 ^ (uint32_t)(r & 7)) << 4) + sub);
                        const uint32_t w1 = *reinterpret_cast<const uint32_t*>(tile + (r + 1) * 128 + ((c16 ^ (uint32_t)((r + 1) & 7)) << 4) + sub);
                        s0 += __uint_as_float(w0 << 16);
                        s1 += __uint_as_float(w0 & 0xFFFF0000u);
                        s2 += __uint_as_float(w1 << 16);
                        s3 += __uint_as_float(w1 & 0xFFFF0000u);
                    }
                }
                __syncwarp();
                if (lane == 0) mbar_arrive(&empty[stage]);
                if (++stage == NST) {
                    stage = 0;
                    phase ^= 1;
                }
            }
            if (want_db) {
                const int n = it.n0 + ew * 64 + 2 * lane;
                if (n < L.N) atomicAdd(L.db + n, s0 + s2);
                if (n + 1 < L.N) atomicAdd(L.db + n + 1, s1 + s3);
            }
            mbar_wait(tfull, n_done & 1);
            tc_fence_after();
            const int n_kt = (it.n_x + 1) / 2;
            const int nch = (min(256, L.N - it.n0) + 31) >> 5;
            for (int kt = 0; kt < n_kt; ++kt) {
                const uint32_t trow = tmem_base + ((uint32_t)(ew * 32) << 16) + kt * 256;
                const int k = it.k0 + kt * 128 + ew * 32 + lane;
                for (int c = 0; c < nch; ++c) {
                    float v[32];
                    tmem_ld32(trow + c * 32, v);
                    if (k < L.K) {
#pragma unroll
                        for (int j = 0; j < 32; ++j) {
                            const int n = it.n0 + c * 32 + j;
                            if (n < L.N) atomicAdd(L.dw + (int64_t)n * L.lddw + k, v[j]);
                        }
                    }
                }
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(tempty);
            ++n_done;
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        tc_fence_after();
        tmem_dealloc(tmem_base, 512);
    }
}

// column sums of a bf16 matrix: db[n] += sum_m dY[m,n]   (bias gradients)
__global__ void colsum_kernel(const uint16_t* __restrict__ dy, int64_t ld, int64_t M, int N, int n8,
                              float* __restrict__ db, int64_t rows_per_block) {
    extern __shared__ float s_acc[];  // n8 floats (N rounded up to 8; the padding columns of dY are zero)
    for (int i = threadIdx.x; i < n8; i += blockDim.x) s_acc[i] = 0.f;
    __syncthreads();
    const int groups = n8 >> 3;                      // 8 columns (16 B) per thread
    const int g = threadIdx.x % groups;
    const int rlane = threadIdx.x / groups;
    const int rstride = blockDim.x / groups;
    const int64_t r0 = (int64_t)blockIdx.x * rows_per_block;
    const int64_t r1 = min(M, r0 + rows_per_block);
    float acc[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    if (rlane < rstride) {
#pragma unroll 4
        for (int64_t r = r0 + rlane; r < r1; r += rstride) {
            const uint4 q = __ldg(reinterpret_cast<const uint4*>(dy + r * ld + g * 8));
            const uint32_t w[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                acc[2 * j] += __uint_as_float(w[j] << 16);
                acc[2 * j + 1] += __uint_as_float(w[j] & 0xFFFF0000u);
            }
        }
#pragma unroll
        for (int j = 0; j < 8; ++j) atomicAdd(&s_acc[g * 8 + j], acc[j]);
    }
    __syncthreads();
    for (int i = threadIdx.x; i < N; i += blockDim.x) atomicAdd(db + i, s_acc[i]);
}

// ---------------------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------------------
template <int BLOCK_N, int EPI>
int launch_rowgemm_t(const CUtensorMap& tmA, const CUtensorMap& tmB, RowGemmParams& p, cudaStream_t s) {
    using L = SmemLayout<BLOCK_N>;
    static bool configured = false;
    auto kfn = rowgemm_kernel<BLOCK_N, EPI>;
    if (!configured) {
        RLPPO_CUDA(cudaFuncSetAttribute(kfn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)L::TOTAL));
        configured = true;
    }
    p.num_m_tiles = (int)((p.M + BLOCK_M - 1) / BLOCK_M);
    p.num_n_tiles = (p.N + BLOCK_N - 1) / BLOCK_N;
    p.num_k_blocks = (p.K + BLOCK_K - 1) / BLOCK_K * (p.sched.n > 0 ? p.sched.n : 1);
    const int tiles = p.num_m_tiles * p.num_n_tiles;
    const int grid = tiles < num_sms() ? tiles : num_sms();
    kfn<<<grid, kThreads, L::TOTAL, s>>>(tmA, tmB, p);
    RLPPO_LAUNCH_CHECK();
    return RLPPO_OK;
}

// Fills the k schedule of a GEMM over split operands: every (i, j) with i < a_parts, j < b_parts, i + j < order,
// ordered by decreasing i + j so that the smallest products are accumulated first.
int fill_sched(const rlppo_split* sp, int K, int* n, int* a_off, int* b_off) {
    *n = 0;
    if (sp == nullptr) return RLPPO_OK;
    RLPPO_CHECK_ARG(sp->a_parts >= 1 && sp->a_parts <= 3 && sp->b_parts >= 1 && sp->b_parts <= 3 && sp->order >= 1 &&
                        sp->order <= 3 && sp->out_parts >= 1 && sp->out_parts <= 3,
                    "split: parts and order must be in [1,3]");
    const int Kp = (K + 63) / 64 * 64;
    RLPPO_CHECK_ARG((sp->a_parts == 1 || (sp->a_pstride % 64 == 0 && sp->a_pstride >= Kp)) &&
                        (sp->b_parts == 1 || (sp->b_pstride % 64 == 0 && sp->b_pstride >= Kp)),
                    "split: part strides must be multiples of 64 columns and cover the contraction width");
    for (int sum = sp->order - 1; sum >= 0; --sum)
        for (int i = 0; i < sp->a_parts; ++i) {
            const int j = sum - i;
            if (j < 0 || j >= sp->b_parts) continue;
            RLPPO_CHECK_ARG(*n < MAX_SCHED, "split: too many products");
            a_off[*n] = (int)(i * sp->a_pstride);
            b_off[*n] = (int)(j * sp->b_pstride);
            ++*n;
        }
    return RLPPO_OK;
}

template <int EPI>
int launch_rowgemm(const uint16_t* a, int64_t lda, const uint16_t* b, int64_t ldb, int64_t b_rows,
                   RowGemmParams& p, int min_block_n, const rlppo_split* sp, cudaStream_t s) {
    RLPPO_CHECK_ARG(p.M >= 1 && p.N >= 1 && p.K >= 1, "empty GEMM");
    RLPPO_CHECK_ARG(p.M < (1ll << 31), "M too large for TMA coordinates");
    int bn = p.N <= 64 ? 64 : (p.N <= 128 ? 128 : 256);
    if (bn < min_block_n) bn = min_block_n;
    int rc = fill_sched(sp, p.K, &p.sched.n, p.sched.a_off, p.sched.b_off);
    if (rc) return rc;
    p.sched.kpp = (p.K + BLOCK_K - 1) / BLOCK_K;
    p.out_parts = sp ? sp->out_parts : 1;
    p.out_pstride = sp ? sp->out_pstride : 0;
    RLPPO_CHECK_ARG(p.out_parts == 1 || p.out_pstride % 8 == 0, "split: output part stride must be a multiple of 8");
    // split operands: the tensor maps span all parts (the k schedule addresses them by column offset)
    const uint64_t a_cols = sp && sp->a_parts > 1 ? (uint64_t)lda : (uint64_t)p.K;
    const uint64_t b_cols = sp && sp->b_parts > 1 ? (uint64_t)ldb : (uint64_t)p.K;
    CUtensorMap tmA, tmB;
    rc = make_tmap_bf16_2d(&tmA, a, (uint64_t)p.M, a_cols, (uint64_t)lda, BLOCK_M);
    if (rc) return rc;
    rc = make_tmap_bf16_2d(&tmB, b, (uint64_t)b_rows, b_cols, (uint64_t)ldb, (uint32_t)bn);
    if (rc) return rc;
    if (EPI == EPI_HEAD_SAMPLE || EPI == EPI_HEAD_TRAIN || EPI == EPI_HEAD_BWD) {
        if (bn <= 128) return launch_rowgemm_t<128, EPI>(tmA, tmB, p, s);
        return launch_rowgemm_t<256, EPI>(tmA, tmB, p, s);
    }
    if (bn == 64) return launch_rowgemm_t<64, EPI>(tmA, tmB, p, s);
    if (bn == 128) return launch_rowgemm_t<128, EPI>(tmA, tmB, p, s);
    return launch_rowgemm_t<256, EPI>(tmA, tmB, p, s);
}

template <int BN>
int launch_wgrad_t(const CUtensorMap& tmX, const CUtensorMap& tmDY, const WgradParams& p, cudaStream_t s) {
    constexpr uint32_t SMEM = kStages * (2 * 8192 + (BN / 64) * 8192) + 256 + 1024;
    static bool configured = false;
    auto kfn = wgrad_kernel<BN>;
    if (!configured) {
        RLPPO_CUDA(cudaFuncSetAttribute(kfn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SMEM));
        configured = true;
    }
    const int grid = p.n_tiles_n * p.n_tiles_k * p.splits;
    kfn<<<grid, kThreads, SMEM, s>>>(tmX, tmDY, p);
    RLPPO_LAUNCH_CHECK();
    return RLPPO_OK;
}

}  // namespace

extern "C" {

int rlppo_linear_fwd_split(const uint16_t* x, int64_t ldx, const uint16_t* w, int64_t ldw, const float* bias,
                           int bias_n, uint16_t* y, int64_t ldy, int64_t M, int N, int K, int relu,
                           const rlppo_split* sp, void* stream) {
    RLPPO_REQUIRE_DEVICE();
    RLPPO_CHECK_ARG(x && w && y, "null pointer");
    RLPPO_CHECK_ARG(N % 8 == 0 && ldy >= N && ldy % 8 == 0, "N and ldy must be multiples of 8");
    RLPPO_CHECK_ARG(bias_n >= 0 && bias_n <= N, "bias_n must be in [0, N]");
    RowGemmParams p{};
    p.M = M; p.N = N; p.K = K;
    p.out = y; p.ldo = ldy; p.bias = bias; p.bias_n = bias_n > 0 ? bias_n : N; p.relu = relu;
    return launch_rowgemm<EPI_BIAS_ACT>(x, ldx, w, ldw, N, p, 0, sp, static_cast<cudaStream_t>(stream));
}

int rlppo_linear_fwd(const uint16_t* x, int64_t ldx, const uint16_t* w, int64_t ldw, const float* bias, uint16_t* y,
                     int64_t ldy, int64_t M, int N, int K, int relu, void* stream) {
    return rlppo_linear_fwd_split(x, ldx, w, ldw, bias, 0, y, ldy, M, N, K, relu, nullptr, stream);
}

int rlppo_linear_dgrad_split(const uint16_t* dy, int64_t lddy, const uint16_t* wt, int64_t ldwt, const uint16_t* hprev,
                             int64_t ldh, uint16_t* dx, int64_t lddx, float* db_below, int64_t M, int N, int K,
                             const rlppo_split* sp, void* stream) {
    RLPPO_REQUIRE_DEVICE();
    RLPPO_CHECK_ARG(dy && wt && dx, "null pointer");
    RLPPO_CHECK_ARG(K % 8 == 0 && lddx >= K && lddx % 8 == 0, "K and lddx must be multiples of 8");
    RLPPO_CHECK_ARG(!hprev || ldh % 8 == 0, "ldh must be a multiple of 8");
    // dX[M,K] = dY[M,N] * (W^T)[K,N]^T : the GEMM's "N" is K (in features), its contraction runs over N
    RowGemmParams p{};
    p.M = M; p.N = K; p.K = N;
    p.out = dx; p.ldo = lddx; p.mask = hprev; p.ldmask = ldh; p.colsum = db_below;
    return launch_rowgemm<EPI_RELU_MASK>(dy, lddy, wt, ldwt, K, p, 0, sp, static_cast<cudaStream_t>(stream));
}

int rlppo_linear_dgrad(const uint16_t* dy, int64_t lddy, const uint16_t* wt, int64_t ldwt, const uint16_t* hprev,
                       int64_t ldh, uint16_t* dx, int64_t lddx, int64_t M, int N, int K, void* stream) {
    return rlppo_linear_dgrad_split(dy, lddy, wt, ldwt, hprev, ldh, dx, lddx, nullptr, M, N, K, nullptr, stream);
}

int rlppo_linear_dgrad_db(const uint16_t* dy, int64_t lddy, const uint16_t* wt, int64_t ldwt, const uint16_t* hprev,
                          int64_t ldh, uint16_t* dx, int64_t lddx, float* db_below, int64_t M, int N, int K,
                          void* stream) {
    return rlppo_linear_dgrad_split(dy, lddy, wt, ldwt, hprev, ldh, dx, lddx, db_below, M, N, K, nullptr, stream);
}

int rlppo_policy_head_sample_split(const uint16_t* h, int64_t ldh, const uint16_t* w, int64_t ldw, const float* bias,
                                   int64_t M, int n_actions, int K, const float* u_inject, uint64_t seed,
                                   uint64_t offset, int deterministic, float* actions_out, int64_t* actions_i64_out,
                                   float* logp_out, float* probs_out, const rlppo_split* sp, void* stream) {
    RLPPO_REQUIRE_DEVICE();
    RLPPO_CHECK_ARG(h && w, "null pointer");
    RLPPO_CHECK_ARG(n_actions >= 1 && n_actions <= 256, "n_actions must be in [1,256]");
    RowGemmParams p{};
    p.M = M; p.N = (n_actions + 7) / 8 * 8; p.K = K;
    p.bias = bias; p.n_actions = n_actions;
    p.u_inject = u_inject; p.seed = seed; p.offset = offset; p.deterministic = deterministic;
    p.actions_out = actions_out; p.actions_i64_out = actions_i64_out; p.logp_out = logp_out; p.probs_out = probs_out;
    return launch_rowgemm<EPI_HEAD_SAMPLE>(h, ldh, w, ldw, n_actions, p, 128, sp, static_cast<cudaStream_t>(stream));
}

int rlppo_policy_head_sample(const uint16_t* h, int64_t ldh, const uint16_t* w, int64_t ldw, const float* bias,
                             int64_t M, int n_actions, int K, const float* u_inject, uint64_t seed, uint64_t offset,
                             int deterministic, float* actions_out, int64_t* actions_i64_out, float* logp_out,
                             float* probs_out, void* stream) {
    return rlppo_policy_head_sample_split(h, ldh, w, ldw, bias, M, n_actions, K, u_inject, seed, offset, deterministic,
                                          actions_out, actions_i64_out, logp_out, probs_out, nullptr, stream);
}

int rlppo_policy_head_train_split(const uint16_t* h, int64_t ldh, const uint16_t* w, int64_t ldw, const float* bias,
                                  int64_t M, int n_actions, int K, const float* actions, const float* old_logp,
                                  const float* adv, float inv_batch, float clip, float ent_coef, uint16_t* dz,
                                  int64_t lddz, float* logp_out, float* metrics, const rlppo_split* sp, void* stream) {
    RLPPO_REQUIRE_DEVICE();
    RLPPO_CHECK_ARG(h && w && actions && old_logp && adv && dz, "null pointer");
    RLPPO_CHECK_ARG(n_actions >= 1 && n_actions <= 256, "n_actions must be in [1,256]");
    // columns written per output part: the whole (padded) row of d(logits)
    const int64_t cols = sp && sp->out_parts > 1 ? sp->out_pstride : lddz;
    RLPPO_CHECK_ARG(cols >= n_actions && cols % 8 == 0 && cols <= 256 && lddz >= cols && lddz % 8 == 0,
                    "d(logits) row width must be a multiple of 8 in [n_actions,256]");
    RowGemmParams p{};
    p.M = M; p.N = (n_actions + 7) / 8 * 8; p.K = K;
    p.bias = bias; p.n_actions = n_actions;
    p.actions = actions; p.old_logp = old_logp; p.adv = adv;
    p.inv_batch = inv_batch; p.clip = clip; p.ent_coef = ent_coef;
    p.out = dz; p.ldo = lddz; p.out_cols = (int)cols; p.logp_out = logp_out; p.metrics = metrics;
    const int min_bn = cols > 128 ? 256 : 128;
    return launch_rowgemm<EPI_HEAD_TRAIN>(h, ldh, w, ldw, n_actions, p, min_bn, sp, static_cast<cudaStream_t>(stream));
}

int rlppo_policy_head_train(const uint16_t* h, int64_t ldh, const uint16_t* w, int64_t ldw, const float* bias,
                            int64_t M, int n_actions, int K, const float* actions, const float* old_logp,
                            const float* adv, float inv_batch, float clip, float ent_coef, uint16_t* dz, int64_t lddz,
                            float* logp_out, float* metrics, void* stream) {
    return rlppo_policy_head_train_split(h, ldh, w, ldw, bias, M, n_actions, K, actions, old_logp, adv, inv_batch, clip,
                                         ent_coef, dz, lddz, logp_out, metrics, nullptr, stream);
}

// Backward of get_backprop_data (discrete_policy.py:64-80: clamp(softmax(z), 1e-11, 1) -> log -> gather / entropy mean)
// and of get_output (:35-42, the unclamped softmax) for arbitrary upstream gradients; the clamp passes gradient where
// 1e-11 <= s_j <= 1 (torch.clamp's backward):
//   g_j = mask_j * (d_logp/p_a [j == a] - (d_ent/M)(log p_j + 1)) + d_probs_j,  dz = s (.) (g - sum g.s).
int rlppo_policy_head_backward_split(const uint16_t* h, int64_t ldh, const uint16_t* w, int64_t ldw, const float* bias,
                                     int64_t M, int n_actions, int K, const float* actions, const float* d_logp,
                                     const float* d_ent, const float* d_probs, uint16_t* dz, int64_t lddz,
                                     const rlppo_split* sp, void* stream) {
    RLPPO_REQUIRE_DEVICE();
    RLPPO_CHECK_ARG(h && w && dz && (d_logp == nullptr || actions != nullptr), "null pointer");
    RLPPO_CHECK_ARG(n_actions >= 1 && n_actions <= 256, "n_actions must be in [1,256]");
    const int64_t cols = sp && sp->out_parts > 1 ? sp->out_pstride : lddz;
    RLPPO_CHECK_ARG(cols >= n_actions && cols % 8 == 0 && cols <= 256 && lddz >= cols && lddz % 8 == 0,
                    "d(logits) row width must be a multiple of 8 in [n_actions,256]");
    RowGemmParams p{};
    p.M = M; p.N = (n_actions + 7) / 8 * 8; p.K = K;
    p.bias = bias; p.n_actions = n_actions; p.actions = actions;
    p.d_logp = d_logp; p.d_ent = d_ent; p.d_probs = d_probs;
    p.out = dz; p.ldo = lddz; p.out_cols = (int)cols;
    const int min_bn = cols > 128 ? 256 : 128;
    return launch_rowgemm<EPI_HEAD_BWD>(h, ldh, w, ldw, n_actions, p, min_bn, sp, static_cast<cudaStream_t>(stream));
}

int rlppo_policy_head_backward(const uint16_t* h, int64_t ldh, const uint16_t* w, int64_t ldw, const float* bias,
                               int64_t M, int n_actions, int K, const float* actions, const float* d_logp,
                               const float* d_ent, const float* d_probs, uint16_t* dz, int64_t lddz, void* stream) {
    return rlppo_policy_head_backward_split(h, ldh, w, ldw, bias, M, n_actions, K, actions, d_logp, d_ent, d_probs, dz,
                                            lddz, nullptr, stream);
}

int rlppo_linear_wgrad_split(const uint16_t* dy, int64_t lddy, const uint16_t* x, int64_t ldx, float* dw, int64_t lddw,
                             float* db, int64_t M, int N, int K, const rlppo_split* sp, void* stream) {
    RLPPO_REQUIRE_DEVICE();
    RLPPO_CHECK_ARG(dy && x && dw && M >= 1 && N >= 1 && K >= 1, "bad argument");
    RLPPO_CHECK_ARG(M < (1ll << 31), "M too large for TMA coordinates");
    RLPPO_CHECK_ARG(lddy % 8 == 0 && ldx % 8 == 0, "lddy and ldx must be multiples of 8");
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    const int bn = N <= 64 ? 64 : (N <= 128 ? 128 : 256);
    WgradParams p{};
    p.M = M; p.N = N; p.K = K; p.dw = dw; p.lddw = lddw;
    p.n_tiles_n = (N + bn - 1) / bn;
    p.n_tiles_k = (K + 127) / 128;
    // split operands: a = dY (contraction over rows, so the "width" the parts must cover is N), b = X (width K)
    if (sp != nullptr) {
        rlppo_split t = *sp;
        const int Np = (N + 63) / 64 * 64, Kp = (K + 63) / 64 * 64;
        RLPPO_CHECK_ARG((t.a_parts == 1 || t.a_pstride >= Np) && (t.b_parts == 1 || t.b_pstride >= Kp),
                        "split: part strides must cover the operand widths");
        // fill_sched validates strides against ONE contraction width; here the two operands have different widths
        int rc0 = fill_sched(&t, 1, &p.n_sched, p.dy_off, p.x_off);
        if (rc0) return rc0;
    }
    const int tiles = p.n_tiles_n * p.n_tiles_k;
    const int64_t kblocks = (M + BLOCK_K - 1) / BLOCK_K;
    int64_t splits = num_sms() / tiles;
    if (splits < 1) splits = 1;
    if (splits > kblocks) splits = kblocks;
    p.m_per_split = ((kblocks + splits - 1) / splits) * BLOCK_K;
    p.splits = (int)((M + p.m_per_split - 1) / p.m_per_split);
    // the tensor maps expose the padded widths (ld) so 64-wide boxes past N / K read zeros or padding
    const bool xs = sp && sp->b_parts > 1, ys = sp && sp->a_parts > 1;
    const uint64_t x_cols = xs ? (uint64_t)ldx : (uint64_t)min((int64_t)((K + 7) / 8 * 8), ldx);
    const uint64_t dy_cols = ys ? (uint64_t)lddy : (uint64_t)min((int64_t)((N + 7) / 8 * 8), lddy);
    CUtensorMap tmX, tmDY;
    int rc = make_tmap_bf16_2d(&tmX, x, (uint64_t)M, x_cols, (uint64_t)ldx, 64);
    if (rc) return rc;
    rc = make_tmap_bf16_2d(&tmDY, dy, (uint64_t)M, dy_cols, (uint64_t)lddy, 64);
    if (rc) return rc;
    if (bn == 64) rc = launch_wgrad_t<64>(tmX, tmDY, p, s);
    else if (bn == 128) rc = launch_wgrad_t<128>(tmX, tmDY, p, s);
    else rc = launch_wgrad_t<256>(tmX, tmDY, p, s);
    if (rc) return rc;
    if (db != nullptr) {
        const int n8 = (N + 7) / 8 * 8;
        RLPPO_CHECK_ARG(n8 <= lddy && n8 / 8 <= 256, "bias-gradient pass needs N padded to 8 within lddy");
        // padded columns of dY are zero by construction, so summing n8 columns is safe; only N are written
        // ~8 blocks per SM: with 512 rows per block a 50 000-row dY gave 98 blocks of 512 dependent 16-byte loads per
        // thread -- 2 TB/s, and at the wide nets (N = 2048) the pass cost 72 % of the weight-gradient GEMM it follows
        int64_t rows_per_block = (M + (int64_t)num_sms() * 8 - 1) / ((int64_t)num_sms() * 8);
        rows_per_block = (rows_per_block + 7) / 8 * 8;
        if (rows_per_block < 32) rows_per_block = 32;
        const unsigned blocks = (unsigned)((M + rows_per_block - 1) / rows_per_block);
        int threads = 256;
        if (threads < n8 / 8) threads = n8 / 8;
        const int dy_parts = sp ? sp->a_parts : 1;
        for (int q = 0; q < dy_parts; ++q) {     // every part of a split dY contributes to the column sums
            colsum_kernel<<<blocks, threads, n8 * sizeof(float), s>>>(dy + (sp ? q * sp->a_pstride : 0), lddy, M, N, n8, db,
                                                                      rows_per_block);
            RLPPO_LAUNCH_CHECK();
        }
    }
    return RLPPO_OK;
}

int rlppo_linear_wgrad(const uint16_t* dy, int64_t lddy, const uint16_t* x, int64_t ldx, float* dw, int64_t lddw,
                       float* db, int64_t M, int N, int K, void* stream) {
    return rlppo_linear_wgrad_split(dy, lddy, x, ldx, dw, lddw, db, M, N, K, nullptr, stream);
}

int rlppo_wgrad_multi(const rlppo_wgrad_item* h_items, int n_items, void* stream) {
    RLPPO_REQUIRE_DEVICE();
    RLPPO_CHECK_ARG(h_items && n_items >= 1 && n_items <= MAXW, "1..%d weight-gradient items per launch", MAXW);
    WMaps maps;
    WMultiParams p{};
    p.n_layers = n_items;
    double bytes[MAXW], total_bytes = 0.0;
    for (int i = 0; i < n_items; ++i) {
        const rlppo_wgrad_item& it = h_items[i];
        RLPPO_CHECK_ARG(it.dy && it.x && it.dw && it.M >= 1 && it.N >= 1 && it.K >= 1, "bad item %d", i);
        RLPPO_CHECK_ARG(it.M < (1ll << 31) && it.lddy % 8 == 0 && it.ldx % 8 == 0, "item %d: ld must be a multiple of 8", i);
        WLayer& L = p.L[i];
        L.dw = it.dw; L.db = it.db; L.lddw = it.lddw; L.M = it.M; L.N = it.N; L.K = it.K;
        L.n_tiles_n = (it.N + 255) / 256;
        L.n_kpairs = (it.K + 255) / 256;
        const uint64_t x_cols = (uint64_t)min((int64_t)((it.K + 7) / 8 * 8), it.ldx);
        const uint64_t dy_cols = (uint64_t)min((int64_t)((it.N + 7) / 8 * 8), it.lddy);
        int rc = make_tmap_bf16_2d(&maps.x[i], it.x, (uint64_t)it.M, x_cols, (uint64_t)it.ldx, 64);
        if (rc) return rc;
        rc = make_tmap_bf16_2d(&maps.dy[i], it.dy, (uint64_t)it.M, dy_cols, (uint64_t)it.lddy, 64);
        if (rc) return rc;
        // bytes one pass over this layer's tiles reads
        bytes[i] = (double)it.M * 2.0 * ((double)L.n_tiles_n * min(it.K, 256 * L.n_kpairs) + (double)L.n_kpairs * min(it.N, 256 * L.n_tiles_n));
        total_bytes += bytes[i];
    }
    const int ctas = num_sms();
    // Row splits per layer, proportional to the bytes the layer reads, such that the launch is ONE wave: never more items
    // than CTAs (an extra item would double the launch time).  Floor of the ideal share first, then the spare CTAs go to
    // the layers that were rounded down the most.
    int64_t splits[MAXW], kblocks[MAXW];
    double ideal[MAXW];
    int used = 0;
    for (int i = 0; i < n_items; ++i) {
        const WLayer& L = p.L[i];
        const int tiles = L.n_tiles_n * L.n_kpairs;
        kblocks[i] = (L.M + BLOCK_K - 1) / BLOCK_K;
        ideal[i] = ctas * (bytes[i] / total_bytes) / tiles;
        splits[i] = (int64_t)ideal[i];
        if (splits[i] < 1) splits[i] = 1;
        if (splits[i] > kblocks[i]) splits[i] = kblocks[i];
        used += tiles * (int)splits[i];
    }
    for (;;) {
        int best = -1;
        double best_gap = 0.0;
        for (int i = 0; i < n_items; ++i) {
            const int tiles = p.L[i].n_tiles_n * p.L[i].n_kpairs;
            const double gap = ideal[i] - (double)splits[i];
            if (splits[i] < kblocks[i] && used + tiles <= ctas && gap > best_gap) {
                best = i;
                best_gap = gap;
            }
        }
        if (best < 0) break;
        ++splits[best];
        used += p.L[best].n_tiles_n * p.L[best].n_kpairs;
    }
    int first = 0;
    for (int i = 0; i < n_items; ++i) {
        WLayer& L = p.L[i];
        const int tiles = L.n_tiles_n * L.n_kpairs;
        L.m_per_split = ((kblocks[i] + splits[i] - 1) / splits[i]) * BLOCK_K;
        L.splits = (int)((L.M + L.m_per_split - 1) / L.m_per_split);
        L.first_item = first;
        first += tiles * L.splits;
    }
    p.total_items = first;
    constexpr uint32_t SMEM = 3 * 8 * 8192 + 256 + 1024;
    static bool configured = false;
    if (!configured) {
        RLPPO_CUDA(cudaFuncSetAttribute(wgrad_multi_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SMEM));
        configured = true;
    }
    const int grid = p.total_items < ctas ? p.total_items : ctas;
    RLPPO_CUDA(launch_pdl(wgrad_multi_kernel, dim3(grid), dim3(kThreads), SMEM, static_cast<cudaStream_t>(stream), maps, p));
    return RLPPO_OK;
}
}
