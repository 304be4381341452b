// clip_grad_norm_ + Adam over flat fp32 arenas (ppo_learner.py:187-193; torch.optim.Adam defaults at :56-59).
// Both nets live in one arena [policy params | value params]; "segments" keep their separate norms, clips,
// learning rates and step counters -- launches are fused, the mathematics is not (SURVEY.md section 7).
// HBM-bound: 16 B read + 12 B written per parameter for the Adam pass, 4 B read for the norm pass.
#include "common.cuh"

namespace {

constexpr int kMaxSeg = 8;
struct Segs {
    int64_t off[kMaxSeg + 1];
    int n;
};

__device__ __forceinline__ int seg_of(const Segs& s, int64_t i) {
    int k = 0;
#pragma unroll
    for (int j = 1; j < kMaxSeg; ++j)
        if (j < s.n && i >= s.off[j]) k = j;
    return k;
}

// out[seg] += sum over the segment of f(a[i], b[i]);  DIFF: (a-b)^2, else a^2
template <bool DIFF>
__global__ void seg_sumsq_kernel(const float* __restrict__ a, const float* __restrict__ b, Segs segs,
                                 float* __restrict__ out) {
    __shared__ float s_part[kMaxSeg];
    if (threadIdx.x < kMaxSeg) s_part[threadIdx.x] = 0.f;
    __syncthreads();
    const int64_t total = segs.off[segs.n];
    float acc[kMaxSeg];
#pragma unroll
    for (int k = 0; k < kMaxSeg; ++k) acc[k] = 0.f;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total;
         i += (int64_t)gridDim.x * blockDim.x) {
        float x = __ldg(a + i);
        if (DIFF) x -= __ldg(b + i);
        const int k = seg_of(segs, i);
#pragma unroll
        for (int j = 0; j < kMaxSeg; ++j)
            if (j == k) acc[j] = fmaf(x, x, acc[j]);
    }
#pragma unroll
    for (int k = 0; k < kMaxSeg; ++k) {
        if (k < segs.n) {
            const float w = rlppo::warp_sum(acc[k]);
            if ((threadIdx.x & 31) == 0) atomicAdd(&s_part[k], w);
        }
    }
    __syncthreads();
    if (threadIdx.x < segs.n) atomicAdd(out + threadIdx.x, s_part[threadIdx.x]);
}

// torch.nn.utils.clip_grad_norm_'s coefficient, clamp(max_norm / (total_norm + 1e-6), max=1).  torch.clamp keeps a NaN
// (a NaN anywhere in the segment's gradient turns the whole segment's update into NaN); fminf would return 1 instead.
__device__ __forceinline__ float clip_coef(float max_norm, float total_norm) {
    const float c = max_norm / (total_norm + 1e-6f);
    return c > 1.0f ? 1.0f : c;
}

// step counters are bumped by a one-thread prologue kernel so every Adam thread sees the same value
__global__ void bump_steps_kernel(int64_t* step_count, int n_seg) {
    if (threadIdx.x < n_seg) step_count[threadIdx.x] += 1;
}

constexpr int kMaxViews = 16;
struct Views {
    rlppo_bf16_view v[kMaxViews];
    int n;
};

__global__ void clip_adam_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m,
                                 float* __restrict__ v, Segs segs, const float* __restrict__ sqnorm,
                                 const float* __restrict__ lr, const int64_t* __restrict__ step_count, float max_norm,
                                 double beta1d, double beta2d, float eps, Views views) {
    // the weights torch derives in Python doubles and then casts: (float)(1 - beta)
    const float beta2 = (float)beta2d, omb1 = (float)(1.0 - beta1d), omb2 = (float)(1.0 - beta2d);
    __shared__ float s_coef[kMaxSeg], s_step_size[kMaxSeg], s_bc2_sqrt[kMaxSeg];
    if (threadIdx.x < segs.n) {
        const int k = threadIdx.x;
        // torch.nn.utils.clip_grad_norm_: coef = max_norm / (total_norm + 1e-6), clamped to 1
        const float total_norm = sqrtf(sqnorm[k]);
        s_coef[k] = clip_coef(max_norm, total_norm);
        const double t = (double)step_count[k];
        const double bc1 = 1.0 - pow(beta1d, t);
        const double bc2 = 1.0 - pow(beta2d, t);
        s_step_size[k] = (float)((double)lr[k] / bc1);
        s_bc2_sqrt[k] = (float)sqrt(bc2);
    }
    __syncthreads();
    const int64_t total = segs.off[segs.n];
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total;
         i += (int64_t)gridDim.x * blockDim.x) {
        const int k = seg_of(segs, i);
        const float gi = g[i] * s_coef[k];
        float mi = m[i], vi = v[i];
        mi = mi + (gi - mi) * omb1;                           // exp_avg.lerp_(grad, 1-beta1)
        vi = vi * beta2 + omb2 * gi * gi;                      // exp_avg_sq.mul_(b2).addcmul_(g,g,1-b2)
        const float denom = sqrtf(vi) / s_bc2_sqrt[k] + eps;   // (sqrt(v)/sqrt(bc2)).add_(eps)
        const float pn = p[i] - s_step_size[k] * (mi / denom);   // param.addcdiv_(m, denom, -step_size)
        p[i] = pn;
        m[i] = mi;
        v[i] = vi;
        // refresh the bf16 GEMM operands of the weight this element belongs to (W and W^T), same launch
        for (int q = 0; q < views.n; ++q) {
            const rlppo_bf16_view& w = views.v[q];
            const int64_t rel = i - w.offset;
            if (rel >= 0 && rel < (int64_t)w.out_f * w.in_f) {
                const int r = (int)(rel / w.in_f), c = (int)(rel - (int64_t)r * w.in_f);
                const uint16_t b = rlppo::f32_to_bf16_bits(pn);
                w.wq[(int64_t)r * w.wq_ld + c] = b;
                if (w.wt != nullptr) w.wt[(int64_t)c * w.wt_ld + r] = b;
                break;
            }
        }
    }
}


// ---------------------------------------------------------------------------------------------------------
// One launch for the whole optimiser step: per-segment gradient norms -> clip -> Adam (+ bf16 operand refresh),
// with a grid barrier between the norm and the update.  The norm is summed in a FIXED order (thread-serial by
// index, xor-shuffle tree, warps in order, blocks in order), so it is bit-identical from run to run and from rank
// to rank: data-parallel replicas that all-reduced the same gradients stay bit-identical (the separate
// seg_sumsq_kernel adds its block partials with fp32 atomics in whatever order the blocks finish -- measured on
// 2 x B200: replicas drifted apart by an ulp of the clip coefficient per step).  It also replaces three launches
// (memset + norm, step bump, Adam) by one.
// Workspace: [arrive, depart] counters (zero before the first launch; the last block to leave zeroes them again)
// followed by gridDim.x * kMaxSeg block partials.  Every block of the grid must be resident (grid <= SMs x occupancy).
// ---------------------------------------------------------------------------------------------------------
constexpr int kFusedThreads = 256;
constexpr int kMaxPeers = 8;
// Data-parallel form (rlppo_norm_clip_adam_peers): the gradient all-reduce is done by this kernel itself over NVLink peer
// mappings instead of a separate NCCL launch.  Every rank's gradient arena and a small flag block live in symmetric
// memory that all ranks of the box have mapped; grads[r] / flags[r] are rank r's copies as seen from THIS process.
//   flag block (uint32): [0, 8) "gradients complete" epoch written by peer r, [32, 40) "done reading yours" epoch
//   written by peer r, [64] this rank's own epoch counter (= number of completed launches).
// Flags are monotonic epochs: a stale read only delays, nothing is ever reset.
struct Peers {
    const float* grads[kMaxPeers];
    unsigned int* flags[kMaxPeers];
    float* gsum;                      // local f32[total]: the summed gradient (read back in the update phase)
    int rank, world;
    // two-shot form only: every rank's `gsum` buffer as mapped here (symmetric memory; red[rank] == gsum)
    const float* red[kMaxPeers];
};
constexpr int kFlagDone = 32, kFlagEpoch = 64, kFlagReduced = 96;
// kernel modes: 0 = one rank (gradients in g), 1 = one-shot peer exchange, 2 = two-shot peer exchange (EXPERIMENTAL)
constexpr int kModeLocal = 0, kModeOneShot = 1, kModeTwoShot = 2;

__device__ __forceinline__ void st_release_sys(unsigned int* p, unsigned int v) {
    asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ unsigned int ld_acquire_sys(const unsigned int* p) {
    unsigned int v;
    asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
// spin until the epoch at p has reached `epoch` (wrap-safe); traps instead of hanging if a peer never shows up
__device__ __forceinline__ void wait_epoch(const unsigned int* p, unsigned int epoch) {
    const long long t0 = clock64();
    while ((int)(ld_acquire_sys(p) - epoch) < 0) {
        if (clock64() - t0 > 240000000000LL) __trap();   // ~2 min: ranks may reach their first step seconds apart
        __nanosleep(200);
    }
}

struct FusedWs {
    unsigned int arrive, depart, arrive2, pad;   // arrive2: the two-shot form's extra grid barrier
    float partial[1];    // [gridDim.x][kMaxSeg]
};

template <int MODE>
__global__ void __launch_bounds__(kFusedThreads)
norm_clip_adam_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m, float* __restrict__ v,
                      Segs segs, float* __restrict__ sqnorm_out, const float* __restrict__ lr,
                      int64_t* __restrict__ step_count, float max_norm, double beta1d, double beta2d, float eps,
                      Views views, FusedWs* __restrict__ ws, const Peers pr) {
    constexpr bool PEERS = MODE != kModeLocal;
    const float beta2 = (float)beta2d, omb1 = (float)(1.0 - beta1d), omb2 = (float)(1.0 - beta2d);
    __shared__ float s_w[kFusedThreads / 32][kMaxSeg];
    __shared__ float s_coef[kMaxSeg], s_step_size[kMaxSeg], s_bc2_sqrt[kMaxSeg];
    __shared__ double s_t[kMaxSeg];
    const int64_t total = segs.off[segs.n];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    // Everything up to pdl_wait() below reads only what EARLIER launches wrote (step counts, p, m, v), never the previous
    // kernel's output (the gradients): these loads and the double-precision bias corrections run under the tail of the
    // weight-gradient kernel.  Two things make that safe: this kernel never triggers its own dependents early (no
    // pdl_trigger), so whatever follows an optimiser step in the stream -- another optimiser step included -- starts after
    // it has completed; and the gradients are read with ld.global.cg, never __ldg: the compiler treats ld.global.nc as an
    // invariant load and hoisted it ABOVE griddepcontrol.wait (the graph-replayed and the launch-by-launch iteration then
    // diverged: test_graph_replayed_iteration_equals_eager).
    if (threadIdx.x < segs.n) {
        // step count read BEFORE the barrier (block 0 writes it after); the double-precision bias corrections are formed
        // here too, off the critical path between the barrier and the update
        const double st = (double)(step_count[threadIdx.x] + 1);
        s_t[threadIdx.x] = st;
        s_step_size[threadIdx.x] = (float)((double)lr[threadIdx.x] / (1.0 - pow(beta1d, st)));
        s_bc2_sqrt[threadIdx.x] = (float)sqrt(1.0 - pow(beta2d, st));
    }

    const int64_t gtid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x, gthreads = (int64_t)gridDim.x * blockDim.x;
    // The first kPre elements of every thread (all of them at the example nets: 332k parameters over 83k threads) stay in
    // registers across the grid barrier: the summed gradient is not re-read, and p, m, v are fetched BEFORE the barrier,
    // so the update phase starts without a DRAM round trip.
    constexpr int kPre = 4;
    float g_pre[kPre], p_pre[kPre], m_pre[kPre], v_pre[kPre];
#pragma unroll
    for (int e = 0; e < kPre; ++e) {
        const int64_t i = gtid + e * gthreads;
        g_pre[e] = 0.f;
        if (i < total) {
            p_pre[e] = __ldcs(p + i);
            m_pre[e] = __ldcs(m + i);
            v_pre[e] = __ldcs(v + i);
        }
    }
    rlppo::pdl_wait();      // gradients come from the previous kernel of the stream

    // ---- phase 0 (PEERS): every rank's gradients are complete ----
    // This launch is stream-ordered behind the local backward kernels; block 0 tells every peer so, and every block
    // waits (polling LOCAL memory) until all peers have said the same.
    unsigned int epoch = 0;
    if (PEERS) {
        epoch = *reinterpret_cast<volatile unsigned int*>(pr.flags[pr.rank] + kFlagEpoch) + 1u;
        if (blockIdx.x == 0 && threadIdx.x < pr.world) {
            __threadfence_system();
            st_release_sys(pr.flags[threadIdx.x] + pr.rank, epoch);
        }
        if (threadIdx.x < pr.world) wait_epoch(pr.flags[pr.rank] + threadIdx.x, epoch);
        __syncthreads();
    }

    // ---- phase 1: this block's partial sums of squares, fixed order ----
    float acc[kMaxSeg];
#pragma unroll
    for (int k = 0; k < kMaxSeg; ++k) acc[k] = 0.f;
    // (PEERS) the all-reduce: peer loads over NVLink (L1 bypassed), summed in rank order on every rank -- the same bits
    // everywhere, so the replicas stay identical without a broadcast.  Same thread <-> element mapping and accumulation
    // order as the one-rank kernel; the loads of four elements x all peers are issued before anything is summed: a loop of
    // dependent loads paid one NVLink round trip per peer and element (measured on 8 GPUs: no faster than NCCL).
    if (MODE == kModeTwoShot) {
        // EXPERIMENTAL (not selected by default; see PPOLearner dp_collective="p2p2"): reduce-scatter + all-gather inside
        // the launch.  (a) this rank sums ITS slice of every peer's arena into its own `gsum` (which the peers have
        // mapped), (b) grid barrier, "slice reduced" flags, (c) every rank reads all reduced slices from their owners.
        // 2 * 4n bytes over NVLink per rank instead of (R-1) * 4n: the form for big arenas on many ranks.
        const int64_t slice = ((total + pr.world - 1) / pr.world + 3) & ~(int64_t)3;
        const int64_t lo = slice * pr.rank < total ? slice * pr.rank : total;
        const int64_t hi = lo + slice < total ? lo + slice : total;
        for (int64_t i0 = lo + gtid; i0 < hi; i0 += 4 * gthreads) {
            float xs[4][kMaxPeers];
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                const int64_t i = i0 + e * gthreads;
#pragma unroll
                for (int r = 0; r < kMaxPeers; ++r)
                    if (i < hi && r < pr.world) xs[e][r] = __ldcg(pr.grads[r] + i);
            }
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                const int64_t i = i0 + e * gthreads;
                if (i < hi) {
                    float x = xs[e][0];
#pragma unroll
                    for (int r = 1; r < kMaxPeers; ++r)
                        if (r < pr.world) x += xs[e][r];
                    __stcg(pr.gsum + i, x);
                }
            }
        }
        // grid barrier on its own counter, then tell the peers that this rank's slice is reduced and wait for theirs
        __syncthreads();
        if (threadIdx.x == 0) {
            __threadfence();
            atomicAdd(&ws->arrive2, 1u);
            const long long t0 = clock64();
            while ((unsigned)rlppo::ld_acquire_s32(reinterpret_cast<const int*>(&ws->arrive2)) < gridDim.x)
                if (clock64() - t0 > 8000000000LL) __trap();
        }
        __syncthreads();
        if (blockIdx.x == 0 && threadIdx.x < pr.world) {
            __threadfence_system();
            st_release_sys(pr.flags[threadIdx.x] + kFlagReduced + pr.rank, epoch);
        }
        if (threadIdx.x < pr.world) wait_epoch(pr.flags[pr.rank] + kFlagReduced + threadIdx.x, epoch);
        __syncthreads();
        // (c) gather: the one-rank kernel's thread <-> element mapping and accumulation order
        for (int64_t i0 = gtid; i0 < total; i0 += 4 * gthreads) {
            float xs[4];
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                const int64_t i = i0 + e * gthreads;
                if (i < total) {
                    int64_t o = i / slice;
                    xs[e] = __ldcg(pr.red[o] + i);
                }
            }
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                const int64_t i = i0 + e * gthreads;
                if (i < total) {
                    const float x = xs[e];
                    if (i0 == gtid) g_pre[e] = x;
                    if (i < lo || i >= hi) pr.gsum[i] = x;       // own slice is already in place
                    const int k = seg_of(segs, i);
#pragma unroll
                    for (int j = 0; j < kMaxSeg; ++j)
                        if (j == k) acc[j] = fmaf(x, x, acc[j]);
                }
            }
        }
    }
    if (MODE == kModeOneShot) {
        for (int64_t i0 = gtid; i0 < total; i0 += 4 * gthreads) {
            float xs[4][kMaxPeers];
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                const int64_t i = i0 + e * gthreads;
#pragma unroll
                for (int r = 0; r < kMaxPeers; ++r)
                    if (i < total && r < pr.world) xs[e][r] = __ldcg(pr.grads[r] + i);
            }
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                const int64_t i = i0 + e * gthreads;
                if (i < total) {
                    float x = xs[e][0];
#pragma unroll
                    for (int r = 1; r < kMaxPeers; ++r)
                        if (r < pr.world) x += xs[e][r];
                    if (i0 == gtid) g_pre[e] = x;
                    pr.gsum[i] = x;
                    const int k = seg_of(segs, i);
#pragma unroll
                    for (int j = 0; j < kMaxSeg; ++j)
                        if (j == k) acc[j] = fmaf(x, x, acc[j]);
                }
            }
        }
    }
    if (!PEERS) {
#pragma unroll
        for (int e = 0; e < kPre; ++e) {
            const int64_t i = gtid + e * gthreads;
            if (i < total) g_pre[e] = __ldcg(g + i);      // NOT __ldg: an invariant load may be hoisted above pdl_wait
        }
#pragma unroll
        for (int e = 0; e < kPre; ++e) {                  // same thread-serial order as the plain loop below
            const int64_t i = gtid + e * gthreads;
            if (i < total) {
                const int k = seg_of(segs, i);
#pragma unroll
                for (int j = 0; j < kMaxSeg; ++j)
                    if (j == k) acc[j] = fmaf(g_pre[e], g_pre[e], acc[j]);
            }
        }
        for (int64_t i = gtid + kPre * gthreads; i < total; i += gthreads) {
            const float x = __ldcg(g + i);
            const int k = seg_of(segs, i);
#pragma unroll
            for (int j = 0; j < kMaxSeg; ++j)
                if (j == k) acc[j] = fmaf(x, x, acc[j]);
        }
    }
#pragma unroll
    for (int k = 0; k < kMaxSeg; ++k)
        if (k < segs.n) {
            const float w = rlppo::warp_sum(acc[k]);
            if (lane == 0) s_w[warp][k] = w;
        }
    __syncthreads();
    if (threadIdx.x < segs.n) {
        float t = 0.f;
        for (int w = 0; w < kFusedThreads / 32; ++w) t += s_w[w][threadIdx.x];
        __stcg(&ws->partial[(size_t)blockIdx.x * kMaxSeg + threadIdx.x], t);
    }
    // ---- grid barrier ----
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence();
        atomicAdd(&ws->arrive, 1u);
        const long long t0 = clock64();
        while ((unsigned)rlppo::ld_acquire_s32(reinterpret_cast<const int*>(&ws->arrive)) < gridDim.x)
            if (clock64() - t0 > 8000000000LL) __trap();   // watchdog (~4 s): the grid was not co-resident
    }
    __syncthreads();
    // every block of this rank has finished reading the peers' gradients: let them go on (they wait for this before
    // their launch ends, i.e. before anything can overwrite their arena)
    if (PEERS && blockIdx.x == 0 && threadIdx.x < pr.world) st_release_sys(pr.flags[threadIdx.x] + kFlagDone + pr.rank, epoch);
    // ---- phase 2: every block adds the block partials in block order (identical result everywhere) ----
    if (warp == 0) {
        for (int k = 0; k < segs.n; ++k) {
            float t = 0.f;
            for (unsigned b = lane; b < gridDim.x; b += 32) t += __ldcg(&ws->partial[(size_t)b * kMaxSeg + k]);
            t = rlppo::warp_sum(t);
            if (lane == 0) {
                // torch.nn.utils.clip_grad_norm_: coef = max_norm / (total_norm + 1e-6), clamped to 1
                s_coef[k] = clip_coef(max_norm, sqrtf(t));
                if (blockIdx.x == 0) {
                    if (sqnorm_out != nullptr) sqnorm_out[k] = t;
                    step_count[k] = (int64_t)s_t[k];
                }
            }
        }
    }
    __syncthreads();
    int hint = 0;
    auto update = [&](int64_t i, float graw, float mi, float vi, float pi) {
        const int k = seg_of(segs, i);
        const float gi = graw * s_coef[k];
        mi = mi + (gi - mi) * omb1;                           // exp_avg.lerp_(grad, 1-beta1)
        vi = vi * beta2 + omb2 * gi * gi;                      // exp_avg_sq.mul_(b2).addcmul_(g,g,1-b2)
        const float denom = sqrtf(vi) / s_bc2_sqrt[k] + eps;   // (sqrt(v)/sqrt(bc2)).add_(eps)
        const float pn = pi - s_step_size[k] * (mi / denom);   // param.addcdiv_(m, denom, -step_size)
        p[i] = pn;
        m[i] = mi;
        v[i] = vi;
        // bf16 operands of the weight this element belongs to (W and W^T).  A thread's elements are gridDim*blockDim apart,
        // mostly inside one matrix: try the view that matched last time before searching; 32-bit index arithmetic.
        if (views.n > 0) {
            int64_t rel = i - views.v[hint].offset;
            if (rel < 0 || rel >= (int64_t)views.v[hint].out_f * views.v[hint].in_f) {
                int found = -1;
                for (int q = 0; q < views.n; ++q) {
                    const int64_t rq = i - views.v[q].offset;
                    if (rq >= 0 && rq < (int64_t)views.v[q].out_f * views.v[q].in_f) found = q;
                }
                if (found < 0) return;
                hint = found;
                rel = i - views.v[hint].offset;
            }
            const rlppo_bf16_view& w = views.v[hint];
            const unsigned r = (unsigned)rel / (unsigned)w.in_f, c = (unsigned)rel - r * (unsigned)w.in_f;
            const uint16_t b = rlppo::f32_to_bf16_bits(pn);
            w.wq[(int64_t)r * w.wq_ld + c] = b;
            if (w.wt != nullptr) w.wt[(int64_t)c * w.wt_ld + r] = b;
        }
    };
#pragma unroll
    for (int e = 0; e < kPre; ++e) {
        const int64_t i = gtid + e * gthreads;
        if (i < total) update(i, g_pre[e], m_pre[e], v_pre[e], p_pre[e]);
    }
    for (int64_t i = gtid + kPre * gthreads; i < total; i += gthreads)
        update(i, PEERS ? pr.gsum[i] : __ldcg(g + i), m[i], v[i], p[i]);
    // ---- leave: the last block resets the counters for the next launch ----
    __syncthreads();
    if (threadIdx.x == 0) {
        const unsigned old = atomicAdd(&ws->depart, 1u);
        if (old == gridDim.x - 1) {
            ws->arrive = 0;
            ws->depart = 0;
            if (MODE == kModeTwoShot) ws->arrive2 = 0;
            if (PEERS) {
                // the launch may only end once every peer has finished reading this rank's gradients
                for (int r = 0; r < pr.world; ++r) wait_epoch(pr.flags[pr.rank] + kFlagDone + r, epoch);
                *reinterpret_cast<volatile unsigned int*>(pr.flags[pr.rank] + kFlagEpoch) = epoch;
            }
            __threadfence();
        }
    }
}

int fused_grid(int64_t total, int* out) {
    static int per_sm = 0;
    if (per_sm == 0) {
        RLPPO_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, norm_clip_adam_kernel<kModeOneShot>, kFusedThreads, 0));
        if (per_sm < 1) per_sm = 1;
        if (per_sm > 4) per_sm = 4;
    }
    const int64_t want = (total + 1023) / 1024;      // four elements per thread at the small nets: short serial loops
    const int64_t cap = (int64_t)rlppo::num_sms() * per_sm;
    *out = (int)(want < 1 ? 1 : (want > cap ? cap : want));
    return RLPPO_OK;
}

int make_segs(const int64_t* h_seg_off, int n_seg, Segs* out) {
    RLPPO_CHECK_ARG(h_seg_off && n_seg >= 1 && n_seg <= kMaxSeg, "n_seg must be in [1,%d]", kMaxSeg);
    out->n = n_seg;
    for (int i = 0; i <= n_seg; ++i) {
        out->off[i] = h_seg_off[i];
        RLPPO_CHECK_ARG(i == 0 || h_seg_off[i] >= h_seg_off[i - 1], "segment offsets must be non-decreasing");
    }
    for (int i = n_seg + 1; i <= kMaxSeg; ++i) out->off[i] = h_seg_off[n_seg];
    return RLPPO_OK;
}

unsigned grid_for(int64_t total) {
    const int64_t want = (total + 1023) / 1024;
    const int64_t cap = (int64_t)rlppo::num_sms() * 8;
    return (unsigned)(want < 1 ? 1 : (want > cap ? cap : want));
}

}  // namespace

extern "C" {

int rlppo_grad_sqnorm(const float* grads, const int64_t* h_seg_off, int n_seg, float* sqnorm, void* stream) {
    RLPPO_REQUIRE_DEVICE();
    RLPPO_CHECK_ARG(grads && sqnorm, "null pointer");
    Segs segs;
    int rc = make_segs(h_seg_off, n_seg, &segs);
    if (rc) return rc;
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    RLPPO_CUDA(cudaMemsetAsync(sqnorm, 0, sizeof(float) * n_seg, s));
    seg_sumsq_kernel<false><<<grid_for(segs.off[n_seg]), 256, 0, s>>>(grads, nullptr, segs, sqnorm);
    RLPPO_LAUNCH_CHECK();
    return RLPPO_OK;
}

size_t rlppo_norm_clip_adam_workspace_bytes(void) {
    return sizeof(FusedWs) + sizeof(float) * kMaxSeg * (size_t)rlppo::num_sms() * 4;
}

static int launch_norm_clip_adam(float* params, const float* grads, const Peers* peers, float* m, float* v,
                                 const int64_t* h_seg_off, int n_seg, float* sqnorm_out, const float* lr,
                                 int64_t* step_count, double max_norm, double beta1, double beta2, double eps,
                                 const rlppo_bf16_view* h_views, int n_views, void* ws, size_t ws_bytes, void* stream) {
    RLPPO_REQUIRE_DEVICE();
    RLPPO_CHECK_ARG(params && (grads || peers) && m && v && lr && step_count && ws, "null pointer");
    RLPPO_CHECK_ARG(ws_bytes >= rlppo_norm_clip_adam_workspace_bytes(), "workspace too small");
    Segs segs;
    int rc = make_segs(h_seg_off, n_seg, &segs);
    if (rc) return rc;
    RLPPO_CHECK_ARG(n_views >= 0 && n_views <= kMaxViews && (n_views == 0 || h_views), "0..%d bf16 views", kMaxViews);
    Views views;
    views.n = n_views;
    for (int i = 0; i < n_views; ++i) {
        views.v[i] = h_views[i];
        RLPPO_CHECK_ARG(h_views[i].wq && h_views[i].out_f >= 1 && h_views[i].in_f >= 1, "bad bf16 view %d", i);
    }
    int grid = 1;
    rc = fused_grid(segs.off[n_seg], &grid);
    if (rc) return rc;
    if (peers != nullptr && peers->red[0] != nullptr)
        RLPPO_CUDA(rlppo::launch_pdl(norm_clip_adam_kernel<kModeTwoShot>, dim3(grid), dim3(kFusedThreads), 0,
                                     static_cast<cudaStream_t>(stream), params, (const float*)nullptr, m, v, segs, sqnorm_out, lr,
                                     step_count, (float)max_norm, beta1, beta2, (float)eps, views, static_cast<FusedWs*>(ws),
                                     *peers));
    else if (peers != nullptr)
        RLPPO_CUDA(rlppo::launch_pdl(norm_clip_adam_kernel<kModeOneShot>, dim3(grid), dim3(kFusedThreads), 0,
                                     static_cast<cudaStream_t>(stream), params, (const float*)nullptr, m, v, segs, sqnorm_out, lr,
                                     step_count, (float)max_norm, beta1, beta2, (float)eps, views, static_cast<FusedWs*>(ws),
                                     *peers));
    else
        RLPPO_CUDA(rlppo::launch_pdl(norm_clip_adam_kernel<kModeLocal>, dim3(grid), dim3(kFusedThreads), 0,
                                     static_cast<cudaStream_t>(stream), params, (const float*)grads, m, v, segs, sqnorm_out, lr,
                                     step_count, (float)max_norm, beta1, beta2, (float)eps, views, static_cast<FusedWs*>(ws),
                                     Peers{}));
    RLPPO_LAUNCH_CHECK();
    return RLPPO_OK;
}

int rlppo_norm_clip_adam(float* params, const float* grads, float* m, float* v, const int64_t* h_seg_off, int n_seg,
                         float* sqnorm_out, const float* lr, int64_t* step_count, double max_norm, double beta1,
                         double beta2, double eps, const rlppo_bf16_view* h_views, int n_views, void* ws,
                         size_t ws_bytes, void* stream) {
    RLPPO_CHECK_ARG(grads != nullptr, "null pointer");
    return launch_norm_clip_adam(params, grads, nullptr, m, v, h_seg_off, n_seg, sqnorm_out, lr, step_count, max_norm,
                                 beta1, beta2, eps, h_views, n_views, ws, ws_bytes, stream);
}

size_t rlppo_peer_flag_bytes(void) { return 128 * sizeof(unsigned int); }

int rlppo_norm_clip_adam_peers(float* params, const float* const* h_peer_grads, void* const* h_peer_flags, int rank,
                               int world, float* gsum, float* m, float* v, const int64_t* h_seg_off, int n_seg,
                               float* sqnorm_out, const float* lr, int64_t* step_count, double max_norm, double beta1,
                               double beta2, double eps, const rlppo_bf16_view* h_views, int n_views, void* ws,
                               size_t ws_bytes, void* stream) {
    RLPPO_CHECK_ARG(h_peer_grads && h_peer_flags && gsum, "null pointer");
    RLPPO_CHECK_ARG(world >= 1 && world <= kMaxPeers && rank >= 0 && rank < world, "rank %d of %d (at most %d peers)", rank,
                    world, kMaxPeers);
    Peers pr{};
    for (int r = 0; r < world; ++r) {
        RLPPO_CHECK_ARG(h_peer_grads[r] && h_peer_flags[r], "null peer pointer %d", r);
        pr.grads[r] = h_peer_grads[r];
        pr.flags[r] = static_cast<unsigned int*>(h_peer_flags[r]);
    }
    pr.gsum = gsum;
    pr.rank = rank;
    pr.world = world;
    return launch_norm_clip_adam(params, nullptr, &pr, m, v, h_seg_off, n_seg, sqnorm_out, lr, step_count, max_norm,
                                 beta1, beta2, eps, h_views, n_views, ws, ws_bytes, stream);
}

int rlppo_norm_clip_adam_peers2(float* params, const float* const* h_peer_grads, void* const* h_peer_flags,
                                const float* const* h_peer_red, int rank, int world, float* m, float* v,
                                const int64_t* h_seg_off, int n_seg, float* sqnorm_out, const float* lr,
                                int64_t* step_count, double max_norm, double beta1, double beta2, double eps,
                                const rlppo_bf16_view* h_views, int n_views, void* ws, size_t ws_bytes, void* stream) {
    RLPPO_CHECK_ARG(h_peer_grads && h_peer_flags && h_peer_red, "null pointer");
    RLPPO_CHECK_ARG(world >= 1 && world <= kMaxPeers && rank >= 0 && rank < world, "rank %d of %d (at most %d peers)", rank,
                    world, kMaxPeers);
    Peers pr{};
    for (int r = 0; r < world; ++r) {
        RLPPO_CHECK_ARG(h_peer_grads[r] && h_peer_flags[r] && h_peer_red[r], "null peer pointer %d", r);
        pr.grads[r] = h_peer_grads[r];
        pr.flags[r] = static_cast<unsigned int*>(h_peer_flags[r]);
        pr.red[r] = h_peer_red[r];
    }
    pr.gsum = const_cast<float*>(h_peer_red[rank]);
    pr.rank = rank;
    pr.world = world;
    return launch_norm_clip_adam(params, nullptr, &pr, m, v, h_seg_off, n_seg, sqnorm_out, lr, step_count, max_norm,
                                 beta1, beta2, eps, h_views, n_views, ws, ws_bytes, stream);
}

int rlppo_sqdiff(const float* a, const float* b, const int64_t* h_seg_off, int n_seg, float* out, void* stream) {
    RLPPO_REQUIRE_DEVICE();
    RLPPO_CHECK_ARG(a && b && out, "null pointer");
    Segs segs;
    int rc = make_segs(h_seg_off, n_seg, &segs);
    if (rc) return rc;
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    RLPPO_CUDA(cudaMemsetAsync(out, 0, sizeof(float) * n_seg, s));
    seg_sumsq_kernel<true><<<grid_for(segs.off[n_seg]), 256, 0, s>>>(a, b, segs, out);
    RLPPO_LAUNCH_CHECK();
    return RLPPO_OK;
}

int rlppo_clip_adam(float* params, const float* grads, float* m, float* v, const int64_t* h_seg_off, int n_seg,
                    const float* sqnorm, const float* lr, int64_t* step_count, double max_norm, double beta1,
                    double beta2, double eps, const rlppo_bf16_view* h_views, int n_views, void* stream) {
    RLPPO_REQUIRE_DEVICE();
    RLPPO_CHECK_ARG(params && grads && m && v && sqnorm && lr && step_count, "null pointer");
    Segs segs;
    int rc = make_segs(h_seg_off, n_seg, &segs);
    if (rc) return rc;
    RLPPO_CHECK_ARG(n_views >= 0 && n_views <= kMaxViews && (n_views == 0 || h_views), "0..%d bf16 views", kMaxViews);
    Views views;
    views.n = n_views;
    for (int i = 0; i < n_views; ++i) {
        views.v[i] = h_views[i];
        RLPPO_CHECK_ARG(h_views[i].wq && h_views[i].out_f >= 1 && h_views[i].in_f >= 1, "bad bf16 view %d", i);
    }
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    bump_steps_kernel<<<1, 32, 0, s>>>(step_count, n_seg);
    clip_adam_kernel<<<grid_for(segs.off[n_seg]), 256, 0, s>>>(params, grads, m, v, segs, sqnorm, lr, step_count,
                                                              (float)max_norm, beta1, beta2, (float)eps, views);
    RLPPO_LAUNCH_CHECK();
    return RLPPO_OK;
}
}
