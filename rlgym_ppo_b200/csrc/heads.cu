// The other two action heads of the reference (SURVEY.md 8(f)-4; selected by policy_type at ppo_learner.py:34-50):
//   MultiDiscreteFF   multi_discrete_policy.py:16-89 + torch_functions.MultiDiscreteRolv (:81-122): 21 logits = eight
//                     categoricals (bins 3,3,3,3,3,2,2,2); log-prob and entropy summed over the eight.
//   ContinuousPolicy  continuous_policy.py:23-120 + MapContinuousToAction (torch_functions.py:15-33): Tanh over 2n outputs,
//                     mean = first half, std = second half mapped onto [var_min, var_max], diagonal Gaussian.
// Their last Linear runs on the tensor-core GEMM (rlppo_linear_fwd, output written as three bf16 parts so the
// logits keep fp32 precision); these kernels are the per-row tails -- sampling (get_action), and for training
// get_backprop_data + the PPO loss block (ppo_learner.py:146-185) + its analytic backward into the logits.  At most 21 /
// 2n <= 64 columns per row: one thread per row, HBM-bound, ~100-200 B per row.
// UPSTREAM instantiations (rlppo_head_*_backward): the same backward into the logits with the PPO block replaced by
// loaded upstream gradients of get_backprop_data's outputs (d_logp f32[M], d_ent f32[1] of the mean entropy) and, for
// the continuous head, of get_output's (mean, std) -- any of them NULL.
// The wide discrete head (DiscreteFF with 257..4096 actions, head_discrete_kernel below) is the same kind of tail for
// the softmax policy whose rows are too wide for the fused epilogue of the head GEMM: one warp per row.
#include <math.h>

#include "common.cuh"

namespace {

using namespace rlppo;

struct ZView {               // split bf16 matrix (rlppo_split layout): value = sum of parts
    const uint16_t* p;
    int64_t ld;
    int parts;
    int64_t pstride;
};
__device__ __forceinline__ float zload(const ZView& z, int64_t row, int col) {
    float s = 0.f;
    for (int q = z.parts - 1; q >= 0; --q) s += bf16_bits_to_f32(z.p[row * z.ld + q * z.pstride + col]);
    return s;
}
struct DzView {
    uint16_t* p;
    int64_t ld;
    int parts;
    int64_t pstride;
};
__device__ __forceinline__ void dzstore(const DzView& d, int64_t row, int col, float x) {
    for (int q = 0; q < d.parts; ++q) {
        const uint16_t b = f32_to_bf16_bits(x);
        d.p[row * d.ld + q * d.pstride + col] = b;
        x -= bf16_bits_to_f32(b);
    }
}

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
__device__ __forceinline__ float u01(uint32_t r) { return (float)(r >> 8) * (1.0f / 16777216.0f); }

// The PPO loss block shared by every head (ppo_learner.py:153-177) and its derivative with respect to the log-prob.
struct PpoRow {
    float d_logp, kl, clipc, surr;
};
__device__ __forceinline__ PpoRow ppo_row(float logp, float old_lp, float advv, float clip, float inv_batch) {
    const float log_ratio = logp - old_lp;
    const float ratio = expf(log_ratio);
    const float lo = 1.0f - clip, hi = 1.0f + clip;
    const float clipped = fminf(fmaxf(ratio, lo), hi);
    const float s1 = ratio * advv, s2 = clipped * advv;
    const float in_range = (ratio >= lo && ratio <= hi) ? 1.f : 0.f;
    const float d1 = s1 < s2 ? 1.f : (s1 == s2 ? 0.5f : 0.f);      // torch.min backward, ties 0.5 / 0.5
    const float d2 = s1 > s2 ? 1.f : (s1 == s2 ? 0.5f : 0.f);
    PpoRow r;
    r.d_logp = -inv_batch * advv * (d1 + d2 * in_range) * ratio;
    r.kl = (ratio - 1.0f) - log_ratio;
    r.clipc = fabsf(ratio - 1.0f) > clip ? 1.f : 0.f;
    r.surr = fminf(s1, s2);
    return r;
}
__device__ __forceinline__ void metrics_add(float* metrics, float ent, const PpoRow& r, bool ok) {
    const float f = ok ? 1.f : 0.f;
    const float a = warp_sum(ent * f), b = warp_sum(r.kl * f), c = warp_sum(r.clipc * f), d = warp_sum(r.surr * f),
                e = warp_sum(f);
    if ((threadIdx.x & 31) == 0 && metrics != nullptr && e > 0.f) {
        atomicAdd(metrics + 0, a);
        atomicAdd(metrics + 1, b);
        atomicAdd(metrics + 2, c);
        atomicAdd(metrics + 3, d);
        atomicAdd(metrics + 4, e);
    }
}

constexpr int MD_GROUPS = 8;
__constant__ int kBins[MD_GROUPS] = {3, 3, 3, 3, 3, 2, 2, 2};     // multi_discrete_policy.py:21
__constant__ int kStart[MD_GROUPS] = {0, 3, 6, 9, 12, 15, 17, 19};

// ---- MultiDiscrete -----------------------------------------------------------------------------------------------
template <bool TRAIN, bool UPSTREAM = false>
__global__ void head_md_kernel(ZView z, int64_t M, const float* __restrict__ actions, int64_t ld_act,
                               const float* __restrict__ old_logp, const float* __restrict__ adv, float inv_batch,
                               float clip, float ent_coef, DzView dz, int dz_cols, float* __restrict__ logp_out,
                               float* __restrict__ metrics, uint64_t seed, uint64_t offset, int deterministic,
                               const float* __restrict__ u_inject, float* __restrict__ actions_out, int64_t ld_aout,
                               const float* __restrict__ up_logp, const float* __restrict__ up_ent) {
    const int64_t row = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const bool ok = row < M;
    float logp = 0.f, ent = 0.f;
    float lsm[21], pr[21], hg[MD_GROUPS];
    int act[MD_GROUPS];
    if (ok) {
        uint4 rnd[2] = {make_uint4(0, 0, 0, 0), make_uint4(0, 0, 0, 0)};
        if (!TRAIN && !deterministic && u_inject == nullptr) {
            const uint64_t ctr = offset + (uint64_t)row;
            const uint2 key = make_uint2((uint32_t)seed, (uint32_t)(seed >> 32));
            rnd[0] = philox4x32_10(make_uint4((uint32_t)ctr, (uint32_t)(ctr >> 32), 0u, 0u), key);
            rnd[1] = philox4x32_10(make_uint4((uint32_t)ctr, (uint32_t)(ctr >> 32), 1u, 0u), key);
        }
        for (int g = 0; g < MD_GROUPS; ++g) {
            const int s = kStart[g], nb = kBins[g];
            float zz[3], mx = -INFINITY;
            for (int j = 0; j < nb; ++j) {
                zz[j] = zload(z, row, s + j);
                mx = fmaxf(mx, zz[j]);
            }
            float se = 0.f;
            for (int j = 0; j < nb; ++j) se += expf(zz[j] - mx);
            const float lse = mx + logf(se);                   // Categorical(logits=...) normalisation
            float h = 0.f;
            for (int j = 0; j < nb; ++j) {
                lsm[s + j] = zz[j] - lse;
                pr[s + j] = expf(lsm[s + j]);                  // logits_to_probs
                h -= lsm[s + j] * pr[s + j];
            }
            hg[g] = h;
            ent += h;                                          // MultiDiscreteRolv.entropy: sum over the 8 (:121)
            int a;
            if (TRAIN) {
                a = (UPSTREAM && actions == nullptr) ? 0 : (int)actions[row * ld_act + g];
                a = min(max(a, 0), nb - 1);
            } else if (deterministic) {
                a = 0;
                for (int j = 1; j < nb; ++j) a = zz[j] > zz[a] ? j : a;      // argmax, first of ties (:60-66)
            } else {
                const uint32_t rr[8] = {rnd[0].x, rnd[0].y, rnd[0].z, rnd[0].w, rnd[1].x, rnd[1].y, rnd[1].z, rnd[1].w};
                const float u = u_inject != nullptr ? u_inject[row * MD_GROUPS + g] : u01(rr[g]);
                float run = 0.f;
                a = nb - 1;
                bool found = false;
                for (int j = 0; j < nb; ++j) {
                    run += pr[s + j];
                    if (!found && run > u) {
                        found = true;
                        a = j;
                    }
                }
            }
            act[g] = a;
            logp += lsm[s + a];                                // MultiDiscreteRolv.log_prob: sum over the 8 (:115)
        }
    }
    if (!TRAIN) {
        if (ok) {
            for (int g = 0; g < MD_GROUPS; ++g) actions_out[row * ld_aout + g] = (float)act[g];
            if (logp_out) logp_out[row] = logp;
        }
        return;
    }
    if (UPSTREAM) {
        // MultiDiscreteRolv.log_prob / entropy (torch_functions.py:115, :121) differentiated:
        //   dz_i = d_logp (onehot_i - p_i) - (d_ent / M) p_i (lsm_i + H_g)
        if (!ok) return;
        const float dl = up_logp != nullptr ? up_logp[row] : 0.f;
        const float ce = up_ent != nullptr ? -__ldg(up_ent) / (float)M : 0.f;
        for (int g = 0; g < MD_GROUPS; ++g) {
            const int s = kStart[g], nb = kBins[g];
            for (int j = 0; j < nb; ++j) {
                const float onehot = j == act[g] ? 1.f : 0.f;
                dzstore(dz, row, s + j, dl * (onehot - pr[s + j]) + ce * pr[s + j] * (lsm[s + j] + hg[g]));
            }
        }
        for (int c = 21; c < dz_cols; ++c) dzstore(dz, row, c, 0.f);
        return;
    }
    PpoRow r = {0.f, 0.f, 0.f, 0.f};
    if (ok) {
        r = ppo_row(logp, old_logp[row], adv[row], clip, inv_batch);
        // d(ppo_loss)/dz_i = d_logp (onehot_i - p_i) + ent_coef w p_i (lsm_i + H_g)   [entropy.mean() over the minibatch]
        const float ce = ent_coef * inv_batch;
        for (int g = 0; g < MD_GROUPS; ++g) {
            const int s = kStart[g], nb = kBins[g];
            for (int j = 0; j < nb; ++j) {
                const float onehot = j == act[g] ? 1.f : 0.f;
                dzstore(dz, row, s + j, r.d_logp * (onehot - pr[s + j]) + ce * pr[s + j] * (lsm[s + j] + hg[g]));
            }
        }
        for (int c = 21; c < dz_cols; ++c) dzstore(dz, row, c, 0.f);
        if (logp_out) logp_out[row] = logp;
    }
    metrics_add(metrics, ent, r, ok);
}

// ---- Continuous ----------------------------------------------------------------------------------------------------
constexpr int MAX_CONT = 32;     // actions (2n <= 64 outputs)
template <bool TRAIN, bool UPSTREAM = false>
__global__ void head_ct_kernel(ZView z, int64_t M, int n_act, float var_m, float var_b,
                               const float* __restrict__ actions, int64_t ld_act, const float* __restrict__ old_logp,
                               const float* __restrict__ adv, float inv_batch, float clip, float ent_coef, DzView dz,
                               int dz_cols, float* __restrict__ logp_out, float* __restrict__ metrics, uint64_t seed,
                               uint64_t offset, int deterministic, const float* __restrict__ n_inject,
                               float* __restrict__ actions_out, int64_t ld_aout, const float* __restrict__ up_logp,
                               const float* __restrict__ up_ent, const float* __restrict__ up_mean,
                               const float* __restrict__ up_std) {
    const int64_t row = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const bool ok = row < M;
    const float kTwoPi = 6.283185307179586f;
    if (UPSTREAM) {
        // continuous_policy.py:52-59 / :117-118 differentiated for (d_logp, d_ent), plus get_output's (d_mean, d_std);
        // back through the affine map of the std half (torch_functions.py:30-33) and the Tanh (continuous_policy.py:37)
        if (!ok) return;
        const float dl = up_logp != nullptr ? up_logp[row] : 0.f;
        const float ce = up_ent != nullptr ? __ldg(up_ent) / ((float)M * (float)n_act) : 0.f;
        for (int j = 0; j < n_act; ++j) {
            const float tm = tanhf(zload(z, row, j)), ts = tanhf(zload(z, row, n_act + j));
            const float mean = tm, sd = ts * var_m + var_b, ssq = sd * sd;
            float d_mean = 0.f, d_std = ce / sd;
            if (up_logp != nullptr) {
                const float diff = actions[row * ld_act + j] - mean;
                d_mean = dl * diff / ssq;
                d_std += dl * (diff * diff / (ssq * sd) - 1.0f / sd);
            }
            if (up_mean != nullptr) d_mean += up_mean[row * n_act + j];
            if (up_std != nullptr) d_std += up_std[row * n_act + j];
            dzstore(dz, row, j, d_mean * (1.0f - tm * tm));
            dzstore(dz, row, n_act + j, d_std * var_m * (1.0f - ts * ts));
        }
        for (int c = 2 * n_act; c < dz_cols; ++c) dzstore(dz, row, c, 0.f);
        return;
    }
    float logp = 0.f, ent = 0.f;
    PpoRow r = {0.f, 0.f, 0.f, 0.f};
    if (ok) {
        // pass 1: log-prob (the reference's four terms as written, continuous_policy.py:52-59) and entropy
        for (int j = 0; j < n_act; ++j) {
            const float tm = tanhf(zload(z, row, j)), ts = tanhf(zload(z, row, n_act + j));     // nn.Tanh (:37)
            const float mean = tm, sd = ts * var_m + var_b;                                      // torch_functions.py:30-33
            float x;
            if (TRAIN) {
                x = actions[row * ld_act + j];
            } else if (deterministic) {
                x = mean;
            } else {
                float nrm;
                if (n_inject != nullptr) {
                    nrm = n_inject[row * n_act + j];
                } else {
                    const uint64_t ctr = offset + (uint64_t)row;
                    const uint4 q = philox4x32_10(make_uint4((uint32_t)ctr, (uint32_t)(ctr >> 32), (uint32_t)(j >> 1), 0u),
                                                  make_uint2((uint32_t)seed, (uint32_t)(seed >> 32)));
                    // Box-Muller: two normals per counter, one per action of the pair
                    const float u1 = fmaxf(u01(q.x), 1.0f / 16777216.0f), u2 = u01(q.y);
                    const float rad = sqrtf(-2.0f * logf(u1));
                    nrm = (j & 1) ? rad * sinf(kTwoPi * u2) : rad * cosf(kTwoPi * u2);
                }
                x = fminf(fmaxf(mean + sd * nrm, -1.0f), 1.0f);                                  // Normal.sample().clamp (:92)
            }
            if (!TRAIN) actions_out[row * ld_aout + j] = x;
            const float msq = mean * mean, ssq = sd * sd, xsq = x * x;
            const float t1 = -(msq / (2.0f * ssq)), t2 = (mean * x) / ssq, t3 = -(xsq / (2.0f * ssq));
            const float t4 = logf(1.0f / sqrtf(kTwoPi * ssq));
            logp += ((t1 + t2) + t3) + t4;
            ent += 0.5f + 0.5f * logf(kTwoPi) + logf(sd);                                        // Normal.entropy()
        }
        ent /= (float)n_act;           // entropy.mean() over all mb * n elements: the row's share (:117-118)
        if (!TRAIN) {
            if (logp_out) logp_out[row] = (deterministic ? 0.f : logp);
            return;
        }
        r = ppo_row(logp, old_logp[row], adv[row], clip, inv_batch);
        // pass 2: backward.  d_entropy = -ent_coef * mb * w spread over mb * n elements -> -ent_coef * w / n each
        const float ce = -ent_coef * inv_batch / (float)n_act;
        for (int j = 0; j < n_act; ++j) {
            const float tm = tanhf(zload(z, row, j)), ts = tanhf(zload(z, row, n_act + j));
            const float mean = tm, sd = ts * var_m + var_b, ssq = sd * sd;
            const float x = actions[row * ld_act + j];
            const float diff = x - mean;
            const float d_mean = r.d_logp * diff / ssq;
            const float d_std = r.d_logp * (diff * diff / (ssq * sd) - 1.0f / sd) + ce / sd;
            dzstore(dz, row, j, d_mean * (1.0f - tm * tm));
            dzstore(dz, row, n_act + j, d_std * var_m * (1.0f - ts * ts));
        }
        for (int c = 2 * n_act; c < dz_cols; ++c) dzstore(dz, row, c, 0.f);
        if (logp_out) logp_out[row] = logp;
    } else if (!TRAIN) {
        return;
    }
    metrics_add(metrics, ent, r, ok);
}

// ---- Discrete, wide (257..4096 actions) ---------------------------------------------------------------------------
// DiscreteFF (discrete_policy.py:22-80) for action spaces too wide for the head GEMM's fused epilogue, where a row's
// logits must fit one TMEM tile (<= 256 columns).  The last Linear writes its logits as split parts (rlppo_linear_fwd)
// and this kernel is the per-row tail, one warp per row (grid-stride over the rows):
//   1. the row's logits, summed from their parts, into shared memory (the only HBM read of z: each lane loads 8
//      consecutive columns of a part as one 16-byte word, so a warp reads 512 contiguous bytes per part and load), with
//      the row max and the first argmax;
//   2. e_j = exp(z_j - max) in place, S = sum e;
//   3. sample: total clamped mass P (and probs_out = e/S); train: entropy, the clamp-masked sum of s (log p + 1) and,
//      upstream, sum d_probs . s -- together they give G = sum g s of the epilogue without a pass per term;
//   4. sample: inverse-CDF scan over 32-column chunks (warp inclusive scan, running total carried across chunks);
//      train: d(logits) = s (g - G), written 8 columns (16 bytes) per lane and part.
// The arithmetic is that of epilogue_head_sample / epilogue_head_train (mlp_tcgen05.cu) but for the order of the sums:
// the sampler's running clamped mass is a chunked warp scan rather than one sequential sum, so a u within a few ulps of a
// bucket edge may select the neighbouring action.  The narrow and the wide path never serve the same action count.
// HBM bytes per row: train 2 * z_parts * A in, 2 * dz_parts * dz_cols out, 12 B of scalars; sample 2 * z_parts * A in
// (+ 4 A of probs_out), 12-16 B out.
constexpr int WD_WARPS = 4;          // rows in flight per block (shared memory: 4 * pad8(A) floats)
constexpr int WD_MIN = 257, WD_MAX = 4096;

__device__ __forceinline__ float clamp_p(float s) { return fminf(fmaxf(s, 1e-11f), 1.0f); }     // :54, :74

template <bool TRAIN, bool UPSTREAM = false>
__global__ void __launch_bounds__(WD_WARPS * 32)
head_discrete_kernel(ZView z, int64_t M, int A, const float* __restrict__ actions, const float* __restrict__ old_logp,
                     const float* __restrict__ adv, float inv_batch, float clip, float ent_coef, DzView dz, int dz_cols,
                     float* __restrict__ logp_out, float* __restrict__ metrics, uint64_t seed, uint64_t offset,
                     int deterministic, const float* __restrict__ u_inject, float* __restrict__ actions_out,
                     int64_t* __restrict__ actions_i64_out, float* __restrict__ probs_out,
                     const float* __restrict__ up_logp, const float* __restrict__ up_ent,
                     const float* __restrict__ up_probs) {
    extern __shared__ float4 s_dyn[];
    __shared__ float s_red[WD_WARPS][5];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int A8 = (A + 7) & ~7;
    float* e = reinterpret_cast<float*>(s_dyn) + (size_t)warp * A8;
    float m_ent = 0.f, m_kl = 0.f, m_clip = 0.f, m_surr = 0.f, m_rows = 0.f;
    for (int64_t row = (int64_t)blockIdx.x * WD_WARPS + warp; row < M; row += (int64_t)gridDim.x * WD_WARPS) {
        // pass 1: logits -> shared memory, max and first argmax
        float mx = -INFINITY;
        int amax = 0;
        const uint16_t* zr = z.p + row * z.ld;
#pragma unroll 2
        for (int c0 = lane * 8; c0 < A; c0 += 256) {
            float v[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
            uint4 wq[3];                                   // every part's load in flight before the first add
#pragma unroll
            for (int q = 0; q < 3; ++q)
                if (q < z.parts) wq[q] = __ldg(reinterpret_cast<const uint4*>(zr + q * z.pstride + c0));
#pragma unroll
            for (int q = 2; q >= 0; --q) {                 // the summation order of zload
                if (q >= z.parts) continue;
                const uint32_t ww[4] = {wq[q].x, wq[q].y, wq[q].z, wq[q].w};
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    v[2 * j] += __uint_as_float(ww[j] << 16);
                    v[2 * j + 1] += __uint_as_float(ww[j] & 0xFFFF0000u);
                }
            }
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                if (c0 + j < A && v[j] > mx) {
                    mx = v[j];
                    amax = c0 + j;
                }
            }
            reinterpret_cast<float4*>(e + c0)[0] = make_float4(v[0], v[1], v[2], v[3]);
            reinterpret_cast<float4*>(e + c0)[1] = make_float4(v[4], v[5], v[6], v[7]);
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const float omx = __shfl_xor_sync(0xffffffffu, mx, o);
            const int oa = __shfl_xor_sync(0xffffffffu, amax, o);
            if (omx > mx || (omx == mx && oa < amax)) {
                mx = omx;
                amax = oa;
            }
        }
        __syncwarp();
        // pass 2: e = exp(z - max), S
        float S = 0.f;
        for (int c = lane; c < A; c += 32) {
            const float x = __expf(e[c] - mx);
            e[c] = x;
            S += x;
        }
        S = warp_sum(S);
        __syncwarp();
        const float invS = __frcp_rn(S);   // == 1.0f / S (both round the reciprocal to nearest), no division slow path

        if (!TRAIN) {
            // DiscreteFF.get_action / get_output (discrete_policy.py:35-62)
            float P = 0.f;
            if (probs_out != nullptr || !deterministic) {
                for (int c = lane; c < A; c += 32) {
                    const float s = e[c] * invS;
                    if (probs_out != nullptr) probs_out[row * A + c] = s;                // unclamped softmax (:35-42)
                    P += clamp_p(s);               // total clamped mass: torch.multinomial normalises what it is given
                }
                P = warp_sum(P);
            }
            int act;
            float pa;
            if (deterministic) {
                act = amax;
                pa = clamp_p(invS);                // exp(0) / S
            } else {
                float u;
                if (u_inject != nullptr) {
                    u = __ldg(u_inject + row);
                } else {
                    const uint64_t ctr = offset + (uint64_t)row;
                    const uint4 r = philox4x32_10(make_uint4((uint32_t)ctr, (uint32_t)(ctr >> 32), 0u, 0u),
                                                  make_uint2((uint32_t)seed, (uint32_t)(seed >> 32)));
                    u = u01(r.x);
                }
                const float thr = u * P;
                act = A - 1;                       // no running mass above thr (rounding): the last action
                pa = 0.f;
                float carry = 0.f;
                for (int c0 = 0; c0 < A; c0 += 32) {
                    const int col = c0 + lane;
                    const float pj = col < A ? clamp_p(e[col] * invS) : 0.f;
                    float run = pj;
#pragma unroll
                    for (int o = 1; o < 32; o <<= 1) {
                        const float t = __shfl_up_sync(0xffffffffu, run, o);
                        if (lane >= o) run += t;
                    }
                    run += carry;
                    const unsigned hit = __ballot_sync(0xffffffffu, col < A && run > thr);
                    if (hit != 0u) {
                        const int l = __ffs(hit) - 1;
                        act = c0 + l;
                        pa = __shfl_sync(0xffffffffu, pj, l);
                        break;
                    }
                    carry = __shfl_sync(0xffffffffu, run, 31);
                    pa = __shfl_sync(0xffffffffu, pj, (A - 1) & 31);     // used only after the last chunk
                }
            }
            if (lane == 0) {
                if (actions_out != nullptr) actions_out[row] = (float)act;       // batched_agent_manager.py:204
                if (actions_i64_out != nullptr) actions_i64_out[row] = (int64_t)act;
                if (logp_out != nullptr) logp_out[row] = logf(pa);               // :60
            }
            __syncwarp();
            continue;
        }

        // get_backprop_data (:64-80) + the PPO block (ppo_learner.py:153-177) or upstream gradients, backward into z
        int a = 0;
        float old_lp = 0.f, advv = 0.f, up_lp = 0.f;
        if (UPSTREAM) {
            if (up_logp != nullptr) {
                a = min(max((int)__ldg(actions + row), 0), A - 1);
                up_lp = __ldg(up_logp + row);
            }
        } else {
            a = min(max((int)__ldg(actions + row), 0), A - 1);                   // acts.long(), :71
            old_lp = __ldg(old_logp + row);
            advv = __ldg(adv + row);
        }
        const float* dpr = (UPSTREAM && up_probs != nullptr) ? up_probs + row * A : nullptr;
        // pass 3: entropy, T1 = sum_{mask} s (log p + 1), T2 = sum d_probs . s
        float H = 0.f, T1 = 0.f, T2 = 0.f;
        for (int c = lane; c < A; c += 32) {
            const float s = e[c] * invS;
            const float pj = clamp_p(s);
            const float lg = __logf(pj);
            if (!UPSTREAM) H -= pj * lg;                                          // :78
            if (s >= 1e-11f && s <= 1.0f) T1 += s * (lg + 1.0f);                  // clamp mask
            if (UPSTREAM && dpr != nullptr) T2 += __ldg(dpr + c) * s;
        }
        if (!UPSTREAM) H = warp_sum(H);
        T1 = warp_sum(T1);
        if (UPSTREAM) T2 = warp_sum(T2);
        const float s_a = e[a] * invS;
        const float p_a = clamp_p(s_a);
        const float logp = logf(p_a);                                             // :76-77
        float ga, cw;
        PpoRow r = {0.f, 0.f, 0.f, 0.f};
        if (UPSTREAM) {
            ga = up_lp / p_a;                                                     // dL/dp_a = d_logp / p_a
            cw = up_ent != nullptr ? -__ldg(up_ent) / (float)M : 0.f;            // dL/dp_j = -(d_ent/M)(log p_j + 1)
        } else {
            r = ppo_row(logp, old_lp, advv, clip, inv_batch);
            ga = r.d_logp / p_a;
            cw = ent_coef * inv_batch;
        }
        // G = sum_j g_j s_j with g_j = mask_j (cw (log p_j + 1) + [j == a] ga) + d_probs_j
        const float G = cw * T1 + ((s_a >= 1e-11f && s_a <= 1.0f) ? ga * s_a : 0.f) + T2;
        // pass 4: dz_j = s_j (g_j - G) -> dz parts (columns A..dz_cols zero)
        uint16_t* dr = dz.p + row * dz.ld;
        for (int c0 = lane * 8; c0 < dz_cols; c0 += 256) {
            float o[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
            if (c0 < A) {
                const float4 e0 = reinterpret_cast<const float4*>(e + c0)[0];
                const float4 e1 = reinterpret_cast<const float4*>(e + c0)[1];
                const float ev[8] = {e0.x, e0.y, e0.z, e0.w, e1.x, e1.y, e1.z, e1.w};
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    const int col = c0 + j;
                    if (col < A) {
                        const float s = ev[j] * invS;
                        const float pj = clamp_p(s);
                        float g = cw * (__logf(pj) + 1.0f) + (col == a ? ga : 0.f);
                        g = (s >= 1e-11f && s <= 1.0f) ? g : 0.f;
                        if (UPSTREAM && dpr != nullptr) g += __ldg(dpr + col);
                        o[j] = s * (g - G);
                    }
                }
            }
            for (int q = 0; q < dz.parts; ++q) {
                uint4 w;
                w.x = pack_bf16x2(o[0], o[1]);
                w.y = pack_bf16x2(o[2], o[3]);
                w.z = pack_bf16x2(o[4], o[5]);
                w.w = pack_bf16x2(o[6], o[7]);
                *reinterpret_cast<uint4*>(dr + q * dz.pstride + c0) = w;
                const uint32_t ww[4] = {w.x, w.y, w.z, w.w};
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    o[2 * j] -= __uint_as_float(ww[j] << 16);
                    o[2 * j + 1] -= __uint_as_float(ww[j] & 0xFFFF0000u);
                }
            }
        }
        if (!UPSTREAM) {
            if (lane == 0 && logp_out != nullptr) logp_out[row] = logp;
            m_ent += H;
            m_kl += r.kl;
            m_clip += r.clipc;
            m_surr += r.surr;
            m_rows += 1.f;
        }
        __syncwarp();                      // every lane is done with e before the next row overwrites it
    }
    if (TRAIN && !UPSTREAM) {
        // metrics as the other heads accumulate them, one atomic per block and quantity
        if (lane == 0) {
            s_red[warp][0] = m_ent;
            s_red[warp][1] = m_kl;
            s_red[warp][2] = m_clip;
            s_red[warp][3] = m_surr;
            s_red[warp][4] = m_rows;
        }
        __syncthreads();
        if (threadIdx.x < 5 && metrics != nullptr) {
            float t = 0.f, rows = 0.f;
            for (int w = 0; w < WD_WARPS; ++w) {
                t += s_red[w][threadIdx.x];
                rows += s_red[w][4];
            }
            if (rows > 0.f) atomicAdd(metrics + threadIdx.x, t);
        }
    }
}

template <bool TRAIN, bool UPSTREAM>
int launch_discrete(cudaStream_t s, const ZView& zv, int64_t M, int A, const float* actions, const float* old_logp,
                    const float* adv, float inv_batch, float clip, float ent_coef, const DzView& dv, int dz_cols,
                    float* logp_out, float* metrics, uint64_t seed, uint64_t offset, int deterministic,
                    const float* u_inject, float* actions_out, int64_t* actions_i64_out, float* probs_out,
                    const float* up_logp, const float* up_ent, const float* up_probs) {
    auto kfn = head_discrete_kernel<TRAIN, UPSTREAM>;
    static bool configured = false;
    if (!configured) {
        RLPPO_CUDA(cudaFuncSetAttribute(kfn, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                        (int)(WD_WARPS * WD_MAX * sizeof(float))));
        configured = true;
    }
    const size_t smem = (size_t)WD_WARPS * ((A + 7) & ~7) * sizeof(float);
    static size_t cached_smem = 0;      // resident blocks per SM for the last shared-memory size asked about
    static int per_sm = 0;
    if (smem != cached_smem) {
        RLPPO_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kfn, WD_WARPS * 32, smem));
        if (per_sm < 1) per_sm = 1;
        cached_smem = smem;
    }
    const int64_t need = (M + WD_WARPS - 1) / WD_WARPS;
    const int64_t resident = (int64_t)per_sm * num_sms();
    const unsigned grid = (unsigned)(need < resident ? need : resident);
    kfn<<<grid, WD_WARPS * 32, smem, s>>>(zv, M, A, actions, old_logp, adv, inv_batch, clip, ent_coef, dv, dz_cols,
                                           logp_out, metrics, seed, offset, deterministic, u_inject, actions_out,
                                           actions_i64_out, probs_out, up_logp, up_ent, up_probs);
    RLPPO_LAUNCH_CHECK();
    return RLPPO_OK;
}

// z / dz views the 16-byte accesses of head_discrete_kernel can address: aligned base, ld and part stride in whole
// 8-column groups, each part pad8(A) columns wide
int check_discrete_views(const uint16_t* z, int64_t ldz, int z_parts, int64_t z_pstride, int64_t M, int A,
                         const uint16_t* dz, int64_t lddz, int dz_parts, int64_t dz_pstride, int dz_cols) {
    RLPPO_CHECK_ARG(A >= WD_MIN && A <= WD_MAX, "wide discrete head: n_actions must be in [%d,%d] (got %d)", WD_MIN,
                    WD_MAX, A);
    RLPPO_CHECK_ARG(M >= 1, "bad argument");
    const int A8 = (A + 7) & ~7;
    RLPPO_CHECK_ARG(z != nullptr && z_parts >= 1 && z_parts <= 3 && (reinterpret_cast<uintptr_t>(z) & 15) == 0 &&
                        ldz % 8 == 0 && (z_parts == 1 || (z_pstride % 8 == 0 && z_pstride >= A8)) &&
                        ldz >= (int64_t)(z_parts - 1) * z_pstride + A8,
                    "bad logits view (16-byte aligned, ld and part stride multiples of 8 covering pad8(n_actions))");
    if (dz != nullptr) {
        RLPPO_CHECK_ARG(dz_parts >= 1 && dz_parts <= 3 && dz_cols >= A8 && dz_cols % 8 == 0 &&
                            (reinterpret_cast<uintptr_t>(dz) & 15) == 0 && lddz % 8 == 0 &&
                            (dz_parts == 1 || (dz_pstride % 8 == 0 && dz_pstride >= dz_cols)) &&
                            lddz >= (int64_t)(dz_parts - 1) * dz_pstride + dz_cols,
                        "bad d(logits) view (16-byte aligned, ld, part stride and columns multiples of 8)");
    }
    return RLPPO_OK;
}

int check_z(const uint16_t* z, int64_t ldz, int parts, int64_t pstride, int cols) {
    RLPPO_CHECK_ARG(z != nullptr && parts >= 1 && parts <= 3 && (parts == 1 || pstride >= cols) &&
                        ldz >= (int64_t)(parts - 1) * pstride + cols, "bad logits view");
    return RLPPO_OK;
}

}  // namespace

extern "C" {

int rlppo_head_multi_discrete_train(const uint16_t* z, int64_t ldz, int z_parts, int64_t z_pstride, int64_t M,
                                    const float* actions, int64_t ld_act, const float* old_logp, const float* adv,
                                    float inv_batch, float clip, float ent_coef, uint16_t* dz, int64_t lddz, int dz_parts,
                                    int64_t dz_pstride, int dz_cols, float* logp_out, float* metrics, void* stream) {
    RLPPO_REQUIRE_DEVICE();
    int rc = check_z(z, ldz, z_parts, z_pstride, 21);
    if (rc) return rc;
    RLPPO_CHECK_ARG(actions && old_logp && adv && dz && M >= 1 && ld_act >= 8, "bad argument");
    RLPPO_CHECK_ARG(dz_parts >= 1 && dz_parts <= 3 && dz_cols >= 21 && (dz_parts == 1 || dz_pstride >= dz_cols) &&
                        lddz >= (int64_t)(dz_parts - 1) * dz_pstride + dz_cols, "bad d(logits) view");
    const ZView zv{z, ldz, z_parts, z_pstride};
    const DzView dv{dz, lddz, dz_parts, dz_pstride};
    head_md_kernel<true><<<(unsigned)((M + 127) / 128), 128, 0, static_cast<cudaStream_t>(stream)>>>(
        zv, M, actions, ld_act, old_logp, adv, inv_batch, clip, ent_coef, dv, dz_cols, logp_out, metrics, 0, 0, 0, nullptr,
        nullptr, 0, nullptr, nullptr);
    RLPPO_LAUNCH_CHECK();
    return RLPPO_OK;
}

int rlppo_head_multi_discrete_backward(const uint16_t* z, int64_t ldz, int z_parts, int64_t z_pstride, int64_t M,
                                       const float* actions, int64_t ld_act, const float* d_logp, const float* d_ent,
                                       uint16_t* dz, int64_t lddz, int dz_parts, int64_t dz_pstride, int dz_cols,
                                       void* stream) {
    RLPPO_REQUIRE_DEVICE();
    int rc = check_z(z, ldz, z_parts, z_pstride, 21);
    if (rc) return rc;
    RLPPO_CHECK_ARG(dz && M >= 1 && (d_logp == nullptr || (actions != nullptr && ld_act >= 8)), "bad argument");
    RLPPO_CHECK_ARG(dz_parts >= 1 && dz_parts <= 3 && dz_cols >= 21 && (dz_parts == 1 || dz_pstride >= dz_cols) &&
                        lddz >= (int64_t)(dz_parts - 1) * dz_pstride + dz_cols, "bad d(logits) view");
    const ZView zv{z, ldz, z_parts, z_pstride};
    const DzView dv{dz, lddz, dz_parts, dz_pstride};
    head_md_kernel<true, true><<<(unsigned)((M + 127) / 128), 128, 0, static_cast<cudaStream_t>(stream)>>>(
        zv, M, d_logp != nullptr ? actions : nullptr, ld_act, nullptr, nullptr, 0.f, 0.f, 0.f, dv, dz_cols, nullptr,
        nullptr, 0, 0, 0, nullptr, nullptr, 0, d_logp, d_ent);
    RLPPO_LAUNCH_CHECK();
    return RLPPO_OK;
}

int rlppo_head_multi_discrete_sample(const uint16_t* z, int64_t ldz, int z_parts, int64_t z_pstride, int64_t M,
                                     const float* u_inject, uint64_t seed, uint64_t offset, int deterministic,
                                     float* actions_out, int64_t ld_aout, float* logp_out, void* stream) {
    RLPPO_REQUIRE_DEVICE();
    int rc = check_z(z, ldz, z_parts, z_pstride, 21);
    if (rc) return rc;
    RLPPO_CHECK_ARG(actions_out && M >= 1 && ld_aout >= 8, "bad argument");
    const ZView zv{z, ldz, z_parts, z_pstride};
    const DzView dv{nullptr, 0, 0, 0};
    head_md_kernel<false><<<(unsigned)((M + 127) / 128), 128, 0, static_cast<cudaStream_t>(stream)>>>(
        zv, M, nullptr, 0, nullptr, nullptr, 0.f, 0.f, 0.f, dv, 0, logp_out, nullptr, seed, offset, deterministic, u_inject,
        actions_out, ld_aout, nullptr, nullptr);
    RLPPO_LAUNCH_CHECK();
    return RLPPO_OK;
}

int rlppo_head_continuous_train(const uint16_t* z, int64_t ldz, int z_parts, int64_t z_pstride, int64_t M, int n_act,
                                float var_min, float var_max, const float* actions, int64_t ld_act,
                                const float* old_logp, const float* adv, float inv_batch, float clip, float ent_coef,
                                uint16_t* dz, int64_t lddz, int dz_parts, int64_t dz_pstride, int dz_cols, float* logp_out,
                                float* metrics, void* stream) {
    RLPPO_REQUIRE_DEVICE();
    RLPPO_CHECK_ARG(n_act >= 1 && n_act <= MAX_CONT, "continuous head: 1..%d actions", MAX_CONT);
    int rc = check_z(z, ldz, z_parts, z_pstride, 2 * n_act);
    if (rc) return rc;
    RLPPO_CHECK_ARG(actions && old_logp && adv && dz && M >= 1 && ld_act >= n_act, "bad argument");
    RLPPO_CHECK_ARG(dz_parts >= 1 && dz_parts <= 3 && dz_cols >= 2 * n_act && (dz_parts == 1 || dz_pstride >= dz_cols) &&
                        lddz >= (int64_t)(dz_parts - 1) * dz_pstride + dz_cols, "bad d(logits) view");
    const float m = (var_max - var_min) / 2.0f;          // torch_functions.py:27-28
    const ZView zv{z, ldz, z_parts, z_pstride};
    const DzView dv{dz, lddz, dz_parts, dz_pstride};
    head_ct_kernel<true><<<(unsigned)((M + 127) / 128), 128, 0, static_cast<cudaStream_t>(stream)>>>(
        zv, M, n_act, m, var_min + m, actions, ld_act, old_logp, adv, inv_batch, clip, ent_coef, dv, dz_cols, logp_out,
        metrics, 0, 0, 0, nullptr, nullptr, 0, nullptr, nullptr, nullptr, nullptr);
    RLPPO_LAUNCH_CHECK();
    return RLPPO_OK;
}

int rlppo_head_continuous_backward(const uint16_t* z, int64_t ldz, int z_parts, int64_t z_pstride, int64_t M, int n_act,
                                   float var_min, float var_max, const float* actions, int64_t ld_act,
                                   const float* d_logp, const float* d_ent, const float* d_mean, const float* d_std,
                                   uint16_t* dz, int64_t lddz, int dz_parts, int64_t dz_pstride, int dz_cols,
                                   void* stream) {
    RLPPO_REQUIRE_DEVICE();
    RLPPO_CHECK_ARG(n_act >= 1 && n_act <= MAX_CONT, "continuous head: 1..%d actions", MAX_CONT);
    int rc = check_z(z, ldz, z_parts, z_pstride, 2 * n_act);
    if (rc) return rc;
    RLPPO_CHECK_ARG(dz && M >= 1 && (d_logp == nullptr || (actions != nullptr && ld_act >= n_act)), "bad argument");
    RLPPO_CHECK_ARG(dz_parts >= 1 && dz_parts <= 3 && dz_cols >= 2 * n_act && (dz_parts == 1 || dz_pstride >= dz_cols) &&
                        lddz >= (int64_t)(dz_parts - 1) * dz_pstride + dz_cols, "bad d(logits) view");
    const float m = (var_max - var_min) / 2.0f;
    const ZView zv{z, ldz, z_parts, z_pstride};
    const DzView dv{dz, lddz, dz_parts, dz_pstride};
    head_ct_kernel<true, true><<<(unsigned)((M + 127) / 128), 128, 0, static_cast<cudaStream_t>(stream)>>>(
        zv, M, n_act, m, var_min + m, actions, ld_act, nullptr, nullptr, 0.f, 0.f, 0.f, dv, dz_cols, nullptr, nullptr, 0,
        0, 0, nullptr, nullptr, 0, d_logp, d_ent, d_mean, d_std);
    RLPPO_LAUNCH_CHECK();
    return RLPPO_OK;
}

int rlppo_head_continuous_sample(const uint16_t* z, int64_t ldz, int z_parts, int64_t z_pstride, int64_t M, int n_act,
                                 float var_min, float var_max, const float* n_inject, uint64_t seed, uint64_t offset,
                                 int deterministic, float* actions_out, int64_t ld_aout, float* logp_out, void* stream) {
    RLPPO_REQUIRE_DEVICE();
    RLPPO_CHECK_ARG(n_act >= 1 && n_act <= MAX_CONT, "continuous head: 1..%d actions", MAX_CONT);
    int rc = check_z(z, ldz, z_parts, z_pstride, 2 * n_act);
    if (rc) return rc;
    RLPPO_CHECK_ARG(actions_out && M >= 1 && ld_aout >= n_act, "bad argument");
    const float m = (var_max - var_min) / 2.0f;
    const ZView zv{z, ldz, z_parts, z_pstride};
    const DzView dv{nullptr, 0, 0, 0};
    head_ct_kernel<false><<<(unsigned)((M + 127) / 128), 128, 0, static_cast<cudaStream_t>(stream)>>>(
        zv, M, n_act, m, var_min + m, nullptr, 0, nullptr, nullptr, 0.f, 0.f, 0.f, dv, 0, logp_out, nullptr, seed, offset,
        deterministic, n_inject, actions_out, ld_aout, nullptr, nullptr, nullptr, nullptr);
    RLPPO_LAUNCH_CHECK();
    return RLPPO_OK;
}

int rlppo_head_discrete_train(const uint16_t* z, int64_t ldz, int z_parts, int64_t z_pstride, int64_t M, int n_actions,
                              const float* actions, const float* old_logp, const float* adv, float inv_batch, float clip,
                              float ent_coef, uint16_t* dz, int64_t lddz, int dz_parts, int64_t dz_pstride, int dz_cols,
                              float* logp_out, float* metrics, void* stream) {
    RLPPO_REQUIRE_DEVICE();
    RLPPO_CHECK_ARG(actions && old_logp && adv && dz, "null pointer");
    int rc = check_discrete_views(z, ldz, z_parts, z_pstride, M, n_actions, dz, lddz, dz_parts, dz_pstride, dz_cols);
    if (rc) return rc;
    return launch_discrete<true, false>(static_cast<cudaStream_t>(stream), ZView{z, ldz, z_parts, z_pstride}, M,
                                        n_actions, actions, old_logp, adv, inv_batch, clip, ent_coef,
                                        DzView{dz, lddz, dz_parts, dz_pstride}, dz_cols, logp_out, metrics, 0, 0, 0,
                                        nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr);
}

int rlppo_head_discrete_backward(const uint16_t* z, int64_t ldz, int z_parts, int64_t z_pstride, int64_t M,
                                 int n_actions, const float* actions, const float* d_logp, const float* d_ent,
                                 const float* d_probs, uint16_t* dz, int64_t lddz, int dz_parts, int64_t dz_pstride,
                                 int dz_cols, void* stream) {
    RLPPO_REQUIRE_DEVICE();
    RLPPO_CHECK_ARG(dz && (d_logp == nullptr || actions != nullptr), "null pointer");
    int rc = check_discrete_views(z, ldz, z_parts, z_pstride, M, n_actions, dz, lddz, dz_parts, dz_pstride, dz_cols);
    if (rc) return rc;
    return launch_discrete<true, true>(static_cast<cudaStream_t>(stream), ZView{z, ldz, z_parts, z_pstride}, M,
                                       n_actions, actions, nullptr, nullptr, 0.f, 0.f, 0.f,
                                       DzView{dz, lddz, dz_parts, dz_pstride}, dz_cols, nullptr, nullptr, 0, 0, 0,
                                       nullptr, nullptr, nullptr, nullptr, d_logp, d_ent, d_probs);
}

int rlppo_head_discrete_sample(const uint16_t* z, int64_t ldz, int z_parts, int64_t z_pstride, int64_t M, int n_actions,
                               const float* u_inject, uint64_t seed, uint64_t offset, int deterministic,
                               float* actions_out, int64_t* actions_i64_out, float* logp_out, float* probs_out,
                               void* stream) {
    RLPPO_REQUIRE_DEVICE();
    RLPPO_CHECK_ARG(actions_out || actions_i64_out || logp_out || probs_out, "no output");
    int rc = check_discrete_views(z, ldz, z_parts, z_pstride, M, n_actions, nullptr, 0, 0, 0, 0);
    if (rc) return rc;
    return launch_discrete<false, false>(static_cast<cudaStream_t>(stream), ZView{z, ldz, z_parts, z_pstride}, M,
                                         n_actions, nullptr, nullptr, nullptr, 0.f, 0.f, 0.f, DzView{nullptr, 0, 0, 0},
                                         0, logp_out, nullptr, seed, offset, deterministic, u_inject, actions_out,
                                         actions_i64_out, probs_out, nullptr, nullptr, nullptr);
}
}
