// GAE + returns as a one-pass segmented reverse scan (replaces the Python loop of
// rlgym_ppo/util/torch_functions.py:58-73).
//
// Each timestep t is a pair of affine maps  A_t = bA + aA * A_{t+1},  R_t = bR + aR * R_{t+1}  with
//   aA = f32(gamma*lambda)*(1-done)*(1-trunc),  bA = delta_t (f32),  aR = gamma*(1-done)*(1-trunc),  bR = r_t.
// A done/truncated step has a = 0, which is the segment reset.  Composition (a,b)o(c,d) = (a*c, b + a*d)
// is associative, so the recurrence is a suffix scan: thread-serial over 4 steps, warp shuffle scan over
// lanes, a scan over the 8 warp aggregates of a 1024-step tile, and decoupled look-back across tiles (tile 0 is
// the END of the rollout).  Carries are f64 (HBM-bound kernel; the fp64 work is free) which also reproduces the
// reference's f64 accumulation; delta is formed with the reference's f32 rounding points.
//
// HBM traffic: reads r, done, trunc, V (16 B/step with f32 flags), writes adv, vtarget, ret (12 B/step).
#include <type_traits>

#include "common.cuh"

namespace {

struct Aff {
    double aA, bA, aR, bR;
};

__device__ __forceinline__ Aff aff_identity() { return Aff{1.0, 0.0, 1.0, 0.0}; }
// l = earlier timesteps, r = later timesteps: (l o r)(x) = l(r(x))
__device__ __forceinline__ Aff compose(const Aff& l, const Aff& r) {
    return Aff{l.aA * r.aA, fma(l.aA, r.bA, l.bA), l.aR * r.aR, fma(l.aR, r.bR, l.bR)};
}
__device__ __forceinline__ Aff shfl_down(const Aff& x, int off) {
    return Aff{__shfl_down_sync(0xffffffffu, x.aA, off), __shfl_down_sync(0xffffffffu, x.bA, off),
               __shfl_down_sync(0xffffffffu, x.aR, off), __shfl_down_sync(0xffffffffu, x.bR, off)};
}
__device__ __forceinline__ Aff shfl_idx(const Aff& x, int src) {
    return Aff{__shfl_sync(0xffffffffu, x.aA, src), __shfl_sync(0xffffffffu, x.bA, src),
               __shfl_sync(0xffffffffu, x.aR, src), __shfl_sync(0xffffffffu, x.bR, src)};
}
// inclusive suffix scan over the lanes of a warp (lane l gets l o l+1 o ... o 31)
__device__ __forceinline__ Aff warp_suffix_scan(Aff x, int lane) {
#pragma unroll
    for (int off = 1; off < 32; off <<= 1) {
        Aff y = shfl_down(x, off);
        if (lane + off < 32) x = compose(x, y);
    }
    return x;
}

// Both record arrays hold one 4-double map per tile slot.
struct Workspace {
    double* agg;    // per tile: map of this tile alone
    double* gagg;   // per group of 32 CTAs: map of the group's tiles of one iteration, slot = the group's first tile
};

__device__ __forceinline__ uint32_t smem_addr_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void bulk_g2s(void* smem_dst, const void* gsrc, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     smem_addr_u32(smem_dst)),
                 "l"(gsrc), "r"(bytes), "r"(smem_addr_u32(bar))
                 : "memory");
}
// Tile records without flags or fences: a record (4 doubles) is written with two 16-byte relaxed gpu-scope vector
// stores and polled with two relaxed gpu-scope vector loads.  The workspace is pre-set to all-ones bytes -- a NaN
// pattern no computation produces -- and a record counts as arrived when none of its four doubles is that pattern (each
// 8-byte element is single-copy atomic, so nothing torn can pass the test).  The accesses must be STRONG (.relaxed.gpu),
// not plain .cg: a weak load may be served by the reader's own L2 partition and never observe the other die's store.
// (A status word published with __threadfence() + st.release and polled with ld.acquire cost 12 % of all stall samples
// on the CCTL.IVALL the acquire emits, plus a dependent second load per look-back round.)
__device__ __forceinline__ void rec_store(double* rec, const Aff& m) {
    asm volatile("st.relaxed.gpu.global.v2.f64 [%0], {%1, %2};" ::"l"(rec), "d"(m.aA), "d"(m.bA) : "memory");
    asm volatile("st.relaxed.gpu.global.v2.f64 [%0], {%1, %2};" ::"l"(rec + 2), "d"(m.aR), "d"(m.bR) : "memory");
}
__device__ __forceinline__ bool rec_load(const double* rec, Aff& m) {
    asm volatile("ld.relaxed.gpu.global.v2.f64 {%0, %1}, [%2];" : "=d"(m.aA), "=d"(m.bA) : "l"(rec) : "memory");
    asm volatile("ld.relaxed.gpu.global.v2.f64 {%0, %1}, [%2];" : "=d"(m.aR), "=d"(m.bR) : "l"(rec + 2) : "memory");
    constexpr long long kUnset = -1LL;   // 0xFFFF'FFFF'FFFF'FFFF
    return __double_as_longlong(m.aA) != kUnset && __double_as_longlong(m.bA) != kUnset &&
           __double_as_longlong(m.aR) != kUnset && __double_as_longlong(m.bR) != kUnset;
}

template <bool TRUNC64>
struct StepMaps {
    const float* r;
    const float* d;
    const float* v;   // tile + 1 entries (halo = V of the next row)
    const void* t;
    double gamma, gl64;   // gl64 = (double)gl32
    float gl32, stdv;
    bool has_std;
    // multipliers of local step j exactly as the reference writes them (torch_functions.py:59-60, 69, 72): the generic
    // path, for flags that are not exactly +0 / 1 and for tiles that are not staged
    __device__ __forceinline__ void mults(int j, double& aA, double& aR) const {
        const float dj = d[j];
        const double trj = TRUNC64 ? static_cast<const double*>(t)[j] : (double)static_cast<const float*>(t)[j];
        const float nd = __fsub_rn(1.0f, dj);                                // :59
        const double nt = 1.0 - trj;                                         // :60
        aA = (double)__fmul_rn(gl32, nd) * nt;                               // :72
        aR = gamma * (double)nd * nt;                                        // :69
    }
    // delta (f32, the reference's NumPy>=2 rounding points, :62-68) from the step's r, done, V and V of the next row
    __device__ __forceinline__ float delta_of(float rj, float dj, float vj, float vnext) const {
        const float nd = __fsub_rn(1.0f, dj);                                // :59
        float nr = rj;
        if (has_std) {                                                       // :62-65
            nr = __fdiv_rn(rj, stdv);
            nr = fminf(fmaxf(nr, -10.f), 10.f);
        }
        const float gv = (float)(gamma * (double)vnext);
        const float pred = __fadd_rn(nr, __fmul_rn(gv, nd));                 // :67
        return __fsub_rn(pred, vj);                                          // :68
    }
    __device__ __forceinline__ float delta(int j) const { return delta_of(r[j], d[j], v[j], v[j + 1]); }
};

// ---------------------------------------------------------------------------------------------------------
// Persistent, software-pipelined scan.
//
// With one tile per CTA the scan is latency-bound (a tile waits for its loads, then its look-back, then its stores, at
// 40 % of the DRAM bandwidth however the phases are trimmed).  Here a CTA lives for the whole launch and overlaps the
// three latencies with compute:
//   * 3 CTAs per SM; CTA b takes tiles b, b+G, b+2G, ... (tile 0 = the END of the rollout, 1024 steps per tile).
//   * warp 8 (one thread): producer.  Keeps a 3-stage ring of {r, done, V(+halo), truncated} tiles filled with bulk
//     async copies (mbarrier full/empty per stage), so tile k+1 and k+2 are in flight while tile k is scanned.
//   * warps 0-7: compute.  A(k): flags -> delta -> thread/warp/block aggregates, everything phase B needs moved to
//     REGISTERS (r, V, delta, live mask, the thread's exclusive map) and the stage handed back at once.
//     B(k-1) runs AFTER A(k): by then the look-back of tile k-1 has had a whole A phase to finish.
//   * warp 9: look-back.  Publishes the group aggregates, gathers the records right of the tile, composes them with
//     this CTA's own previous tile's inclusive map, which it still holds in registers, and hands the carry to the
//     compute warps through shared memory.
// A tile is staged only when the launch allows it (every input pointer, and every output pointer when storing, is
// 16-byte aligned) and all of its 1024 steps and the 4-float V halo exist.  Other tiles take bounds-checked global loads
// with the reference's expressions as written.
// Co-residency: the grid is min(tiles, 3 x SMs) CTAs; a CTA waits only for aggregates of lower-numbered tiles, which
// lower-numbered CTAs (scheduled first) or earlier iterations produce, so a partially resident grid still progresses.
// ---------------------------------------------------------------------------------------------------------
constexpr int kItems = 4;                 // steps per thread
constexpr int kTile = 1024;               // steps per tile
constexpr int kCompute = kTile / kItems;  // compute threads
constexpr int kThreads = kCompute + 32;   // + look-back warp
constexpr int kWarps = kCompute / 32;
constexpr int kStages = 3;
constexpr int kCtasPerSm = 3;
constexpr uint32_t kVBytes = kTile * 4u + 16u;            // V tile + 4-float halo (only the first is used)
constexpr uint32_t kOffD = kTile * 4u;
constexpr uint32_t kOffV = 2u * kTile * 4u;
constexpr uint32_t kOffT = kOffV + kVBytes;
__host__ __device__ constexpr uint32_t stage_bytes(bool t64) { return kOffT + kTile * (t64 ? 8u : 4u); }

__device__ __forceinline__ void mbar_init(uint64_t* b, uint32_t cnt) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_addr_u32(b)), "r"(cnt) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* b) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_addr_u32(b)) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* b, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_addr_u32(b)), "r"(bytes) : "memory");
}
// Waiters back off with nanosleep: without it the look-back warp took 11 us for a 300-instruction shuffle scan -- the
// scheduler kept issuing the 24 hot-spinning compute warps of the SM instead.
__device__ __forceinline__ void mbar_wait(uint64_t* b, uint32_t parity) {
    for (;;) {
        uint32_t ok;
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(ok)
            : "r"(smem_addr_u32(b)), "r"(parity)
            : "memory");
        if (ok) return;
        __nanosleep(100);
    }
}

// what phase B needs of a tile, per thread, in registers
struct Pending {
    float r[kItems], v[kItems], dl[kItems];
    Aff e;            // map of everything right of this thread's steps inside the tile
    // bit i < kItems: step i continues the recurrence; bit kItems (kFast): the flags are all exactly 0 / 1 and the tile
    // is a staged one.  One word, not a word and a flag: two of these are live at the 72-register cap of 3 CTAs/SM.
    uint32_t live;
};

template <bool TRUNC64, bool STORE>
__global__ void __launch_bounds__(kThreads, kCtasPerSm)
gae_scan3_kernel(const float* __restrict__ rew, const float* __restrict__ done, const void* __restrict__ trunc,
                 const float* __restrict__ val, int64_t n, double gamma, float gl32,
                 const float* __restrict__ ret_std, float* __restrict__ adv, float* __restrict__ vt,
                 float* __restrict__ ret, double* __restrict__ ret_head, int64_t n_head,
                 const double* __restrict__ carry_in, double* __restrict__ summary_out, Workspace ws, int n_tiles,
                 bool can_stage) {
    extern __shared__ __align__(128) uint8_t smem[];
    __shared__ uint64_t s_full[kStages], s_aggr[2], s_carr[2];
    __shared__ double s_wagg[2][kWarps][4];
    __shared__ double s_agg[2][4];
    __shared__ double s_carry[2][2];

    constexpr uint32_t kStage = stage_bytes(TRUNC64);
    constexpr uint32_t kTB = TRUNC64 ? 8u : 4u;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int G = gridDim.x;
    const int K = (n_tiles - (int)blockIdx.x + G - 1) / G;      // tiles of this CTA (grid <= n_tiles)
    if (tid == 0) {
        for (int i = 0; i < kStages; ++i) {
            mbar_init(&s_full[i], 1);
        }
        for (int i = 0; i < 2; ++i) {
            mbar_init(&s_aggr[i], 1);
            mbar_init(&s_carr[i], 1);
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();

    auto base_of = [&](int k) { return (int64_t)(n_tiles - 1 - ((int)blockIdx.x + k * G)) * kTile; };
    auto staged = [&](int64_t base0) { return can_stage && base0 + kTile + 4 <= n + 1; };

    // stage s takes tile k: four bulk copies (one thread); a tile that is not staged completes its barrier at once
    auto produce = [&](int k) {
        const int s = k % kStages;
        const int64_t base0 = base_of(k);
        if (staged(base0)) {
            uint8_t* st = smem + s * kStage;
            mbar_expect_tx(&s_full[s], 2u * kTile * 4u + kVBytes + kTile * kTB);
            bulk_g2s(st, rew + base0, kTile * 4u, &s_full[s]);
            bulk_g2s(st + kOffD, done + base0, kTile * 4u, &s_full[s]);
            bulk_g2s(st + kOffV, val + base0, kVBytes, &s_full[s]);
            bulk_g2s(st + kOffT, static_cast<const uint8_t*>(trunc) + base0 * kTB, kTile * kTB, &s_full[s]);
        } else {
            mbar_arrive(&s_full[s]);
        }
    };
    if (warp == kWarps) {
        // ===================== look-back =====================
        // Two-level, chain-free.  CTAs form groups of 32 consecutive block ids; the last CTA of a group also publishes
        // the group's aggregate (its own tile's map composed with its 31 peers') in the second record array.  The map of
        // everything right of tile t = bid + k*G, nearest first:
        //   S1  aggregates of the lower peers of this iteration          tiles t-1 .. t-l             (l = bid % 32)
        //   S2  group aggregates of the lower groups of this iteration   groups g-1 .. 0              (g = bid / 32)
        //   S3  group aggregates of the higher groups of iteration k-1   groups NG-1 .. g+1
        //   S4  aggregates of the higher peers of iteration k-1          block ids group end .. bid+1
        //   then this CTA's own previous tile t-G, whose INCLUSIVE map is still in registers.
        // At most 31 + NG-1 records (<= 64: two per lane), all of them published right after a phase A -- no record
        // depends on another CTA's look-back, so nothing propagates serially along the rollout.  (Walking predecessors
        // until an inclusive record turns up advances the inclusive frontier by 32 tiles per L2 round trip: 2^26 steps
        // took 2048 round trips = 757 us whatever the memory system did.)
        const double cA = carry_in ? carry_in[0] : 0.0;
        const double cR = carry_in ? carry_in[1] : 0.0;
        const int bid = (int)blockIdx.x;
        const int NG = (G + 31) >> 5;
        const int g = bid >> 5, l = bid & 31;
        const int gend = ((32 * g + 31 < G - 1) ? 32 * g + 31 : G - 1) - 32 * g;   // local index of the group's last CTA
        const bool group_last = l == gend;
        Aff prev_incl = aff_identity();
        for (int k = 0; k < K; ++k) {
            const int t = bid + k * G;
            mbar_wait(&s_aggr[k & 1], (k >> 1) & 1);
            // read where consumed, not held in registers across the polls (the kernel is at its register cap); the
            // compute warps rewrite s_agg[k & 1] only after lane 0 has handed this tile's carry over, and lane 0 is the
            // only lane whose maps are used
            auto tile_agg = [&]() { return Aff{s_agg[k & 1][0], s_agg[k & 1][1], s_agg[k & 1][2], s_agg[k & 1][3]}; };
            // the record at position p of the nearest-first list (nullptr: none)
            auto rec_at = [&](int p) -> const double* {
                if (p < l) return ws.agg + (size_t)(t - 1 - p) * 4;
                p -= l;
                if (p < g) return ws.gagg + (size_t)(k * G + 32 * (g - 1 - p)) * 4;
                p -= g;
                if (k == 0) return nullptr;
                if (p < NG - 1 - g) return ws.gagg + (size_t)((k - 1) * G + 32 * (NG - 1 - p)) * 4;
                p -= NG - 1 - g;
                if (p < gend - l) return ws.agg + (size_t)((k - 1) * G + 32 * g + gend - p) * 4;
                return nullptr;
            };
            // lane i takes positions 2i and 2i+1 (adjacent: one local compose, then ONE 5-round tree over the lanes)
            const double* pa = rec_at(2 * lane);
            const double* pb = rec_at(2 * lane + 1);
            Aff ma = aff_identity(), mb = aff_identity();
            bool need_a = pa != nullptr, need_b = pb != nullptr;
            const long long t0 = clock64();
            if (group_last) {
                // The group aggregate must not wait for anything but the peers' aggregates (positions 0 .. l-1): publishing
                // it only after the group records of S2/S3 had arrived chained the groups serially, 14 hops per iteration.
                // Warp-uniform polling loops (every lane iterates until the last record is in): lanes that leave a
                // divergent spin loop one by one stay diverged through the shuffle scans below, 11 us from "all records
                // arrived" to "carry handed over" for ~400 instructions.
                Aff s1 = aff_identity();
                const double* ps = lane < l ? ws.agg + (size_t)(t - 1 - lane) * 4 : nullptr;
                bool need_s = ps != nullptr;
                for (;;) {
                    if (need_s && rec_load(ps, s1)) need_s = false;
                    if (!__any_sync(0xffffffffu, need_s)) break;
                    if (clock64() - t0 > 8000000000LL) __trap();   // watchdog (~4 s)
                    __nanosleep(100);                              // back off: 444 warps polling L2 flat out slow everyone down
                }
                if (ps == nullptr) s1 = aff_identity();
#pragma unroll
                for (int off = 1; off < 32; off <<= 1) {   // adjacent pairs first: the maps do not commute
                    const Aff y = shfl_down(s1, off);
                    s1 = compose(s1, y);                       // lanes past the end pull in garbage; lane 0 is exact
                }
                if (lane == 0) rec_store(ws.gagg + (size_t)(k * G + 32 * g) * 4, compose(tile_agg(), s1));
            }
            for (;;) {
                Aff xa, xb;
                bool oka = false, okb = false;
                if (need_a) oka = rec_load(pa, xa);
                if (need_b) okb = rec_load(pb, xb);
                if (oka) {
                    ma = xa;
                    need_a = false;
                }
                if (okb) {
                    mb = xb;
                    need_b = false;
                }
                if (!__any_sync(0xffffffffu, need_a || need_b)) break;
                if (clock64() - t0 > 8000000000LL) __trap();   // watchdog (~4 s)
                __nanosleep(100);
            }
            Aff right = compose(ma, mb);
#pragma unroll
            for (int off = 1; off < 32; off <<= 1) {   // adjacent pairs first: the maps do not commute
                const Aff y = shfl_down(right, off);
                right = compose(right, y);                     // exact on lane 0 (shfl_down past the end returns own value)
            }
            if (k > 0) right = compose(right, prev_incl);      // lane 0 is the only consumer from here on
            const Aff incl = compose(tile_agg(), right);
            prev_incl = incl;
            if (lane == 0) {
                s_carry[k & 1][0] = fma(right.aA, cA, right.bA);
                s_carry[k & 1][1] = fma(right.aR, cR, right.bR);
                if (summary_out != nullptr && t == n_tiles - 1) {
                    summary_out[0] = incl.aA; summary_out[1] = incl.bA;
                    summary_out[2] = incl.aR; summary_out[3] = incl.bR;
                }
                mbar_arrive(&s_carr[k & 1]);       // release: the carry stores above are visible to the waiters
            }
            __syncwarp();
        }
        return;
    }

    // ===================== compute warps =====================
    StepMaps<TRUNC64> sm;
    sm.gamma = gamma; sm.gl32 = gl32; sm.gl64 = (double)gl32;
    sm.has_std = ret_std != nullptr;
    sm.stdv = sm.has_std ? __ldg(ret_std) : 1.f;
    const double g4A = (sm.gl64 * sm.gl64) * (sm.gl64 * sm.gl64);      // multiplier of kItems live steps
    const double g4R = (gamma * gamma) * (gamma * gamma);
    constexpr uint32_t kAllLive = (1u << kItems) - 1u, kFast = 1u << kItems;
    const int j0 = tid * kItems;

    // ---- phase A of tile k: everything up to the tile aggregate; the inputs phase B needs end up in `P` ----
    auto phaseA = [&](int k, Pending& P) {
        const int s = k % kStages;
        const int64_t base0 = base_of(k);
        const bool tile_staged = staged(base0);
        const uint8_t* st = smem + s * kStage;
        mbar_wait(&s_full[s], (k / kStages) & 1);
        Aff agg;
        P.live = 0;
        if (tile_staged) {
            // flags stay in their storage type: the 0/1 fast path only compares them, and an f32 -> f64 conversion per step
            // (quarter-rate pipe) made the f32-flag scan SLOWER than the f64-flag one although it reads 4 bytes less
            using TFlag = typename std::conditional<TRUNC64, double, float>::type;
            float dd[kItems], vn[kItems + 1];
            TFlag tt[kItems];
            const float4 r4 = *reinterpret_cast<const float4*>(st + (size_t)j0 * 4);
            const float4 d4 = *reinterpret_cast<const float4*>(st + kOffD + (size_t)j0 * 4);
            const float4 v4 = *reinterpret_cast<const float4*>(st + kOffV + (size_t)j0 * 4);
            P.r[0] = r4.x; P.r[1] = r4.y; P.r[2] = r4.z; P.r[3] = r4.w;
            dd[0] = d4.x; dd[1] = d4.y; dd[2] = d4.z; dd[3] = d4.w;
            vn[0] = v4.x; vn[1] = v4.y; vn[2] = v4.z; vn[3] = v4.w;
            if (TRUNC64) {
                const double2 t0 = *reinterpret_cast<const double2*>(st + kOffT + (size_t)j0 * 8);
                const double2 t1 = *reinterpret_cast<const double2*>(st + kOffT + (size_t)j0 * 8 + 16);
                tt[0] = t0.x; tt[1] = t0.y; tt[2] = t1.x; tt[3] = t1.y;
            } else {
                const float4 t4 = *reinterpret_cast<const float4*>(st + kOffT + (size_t)j0 * 4);
                tt[0] = t4.x; tt[1] = t4.y; tt[2] = t4.z; tt[3] = t4.w;
            }
            vn[kItems] = *reinterpret_cast<const float*>(st + kOffV + (size_t)(j0 + kItems) * 4);
            bool ok = true;
#pragma unroll
            for (int i = 0; i < kItems; ++i) {
                P.v[i] = vn[i];
                const bool dz = dd[i] == 0.f, tz = tt[i] == (TFlag)0;
                ok = ok && (dz || dd[i] == 1.f) && (tz || tt[i] == (TFlag)1);
                P.live |= (dz && tz ? 1u : 0u) << i;
                P.dl[i] = sm.delta_of(P.r[i], dd[i], vn[i], vn[i + 1]);
            }
            if (ok) {
                // multipliers are 0 or a constant: only the additive parts need arithmetic
                double bA = 0.0, bR = 0.0;
#pragma unroll
                for (int i = kItems - 1; i >= 0; --i) {
                    const bool lv = (P.live >> i) & 1u;
                    bA = fma(lv ? sm.gl64 : 0.0, bA, (double)P.dl[i]);
                    bR = fma(lv ? gamma : 0.0, bR, (double)P.r[i]);
                }
                const bool all = P.live == kAllLive;
                agg = Aff{all ? g4A : 0.0, bA, all ? g4R : 0.0, bR};
                P.live |= kFast;
            } else {
                agg = aff_identity();
#pragma unroll
                for (int i = kItems - 1; i >= 0; --i) {
                    const float nd = __fsub_rn(1.0f, dd[i]);                              // :59
                    const double nt = 1.0 - (double)tt[i];                                // :60
                    const Aff f = Aff{(double)__fmul_rn(gl32, nd) * nt, (double)P.dl[i],  // :72
                                      gamma * (double)nd * nt, (double)P.r[i]};           // :69
                    agg = compose(f, agg);
                }
            }
        } else {
            // tile not staged: bounds-checked global loads, the reference's expressions as written; steps past the end
            // are identity maps so that the carry passes through them
            const int cnt = (int)((n - base0) < (int64_t)kTile ? (n - base0) : (int64_t)kTile);
            sm.r = rew + base0; sm.d = done + base0; sm.v = val + base0;
            sm.t = static_cast<const uint8_t*>(trunc) + base0 * kTB;
            agg = aff_identity();
#pragma unroll
            for (int i = 0; i < kItems; ++i) P.r[i] = P.v[i] = P.dl[i] = 0.f;
#pragma unroll
            for (int i = kItems - 1; i >= 0; --i)
                if (j0 + i < cnt) {
                    Aff f;
                    sm.mults(j0 + i, f.aA, f.aR);
                    P.r[i] = sm.r[j0 + i];
                    P.v[i] = sm.v[j0 + i];
                    P.dl[i] = sm.delta(j0 + i);
                    f.bA = (double)P.dl[i];
                    f.bR = (double)P.r[i];
                    agg = compose(f, agg);
                }
        }
        const Aff incl_w = warp_suffix_scan(agg, lane);
        Aff excl = shfl_down(incl_w, 1);
        if (lane == 31) excl = aff_identity();
        double(*wagg)[4] = s_wagg[k & 1];
        if (lane == 0) {
            wagg[warp][0] = incl_w.aA; wagg[warp][1] = incl_w.bA;
            wagg[warp][2] = incl_w.aR; wagg[warp][3] = incl_w.bR;
        }
        asm volatile("bar.sync 1, %0;" ::"n"(kCompute) : "memory");
        // every compute warp has read stage s into registers by now: refill it with the tile three ahead
        if (tid == 0 && k + kStages < K) {
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // generic-proxy reads before the async-proxy refill
            produce(k + kStages);
        }
        // every warp scans the 8 warp aggregates itself (lanes 0-7): no second barrier
        Aff w = aff_identity();
        if (lane < kWarps) w = Aff{wagg[lane][0], wagg[lane][1], wagg[lane][2], wagg[lane][3]};
#pragma unroll
        for (int off = 1; off < kWarps; off <<= 1) {
            const Aff y = shfl_down(w, off);
            if (lane + off < kWarps) w = compose(w, y);
        }
        // lane l < 8 now holds warps l..7; this warp's exclusive = lane warp+1 (identity for the last warp)
        Aff we = shfl_idx(w, (warp + 1) & 31);
        if (warp == kWarps - 1) we = aff_identity();
        if (tid == 0) {
            // published from here, not by the look-back warp: that one may still be busy with the previous tile
            rec_store(ws.agg + (size_t)((int)blockIdx.x + k * G) * 4, w);
            s_agg[k & 1][0] = w.aA; s_agg[k & 1][1] = w.bA; s_agg[k & 1][2] = w.aR; s_agg[k & 1][3] = w.bR;
            mbar_arrive(&s_aggr[k & 1]);
        }
        P.e = compose(excl, we);
    };

    // ---- phase B of tile k: apply the carry, write the outputs ----
    auto phaseB = [&](int k, const Pending& P) {
        const int64_t base0 = base_of(k);
        mbar_wait(&s_carr[k & 1], (k >> 1) & 1);     // also the flow control that keeps s_agg / s_aggr two tiles deep
        if (!STORE) return;
        const double carryA = s_carry[k & 1][0], carryR = s_carry[k & 1][1];
        double xA = fma(P.e.aA, carryA, P.e.bA);
        double xR = fma(P.e.aR, carryR, P.e.bR);
        const int64_t gbase = base0 + j0;
        const bool head = ret_head != nullptr && gbase < n_head;
        if (P.live & kFast) {
            float oa[kItems], ov[kItems], orr[kItems];
#pragma unroll
            for (int i = kItems - 1; i >= 0; --i) {
                const bool lv = (P.live >> i) & 1u;
                xA = fma(lv ? sm.gl64 : 0.0, xA, (double)P.dl[i]);
                xR = fma(lv ? gamma : 0.0, xR, (double)P.r[i]);
                if (head && gbase + i < n_head) ret_head[gbase + i] = xR;
                oa[i] = (float)xA;                              // :76
                ov[i] = (float)((double)P.v[i] + xA);           // :77
                orr[i] = (float)xR;
            }
            *reinterpret_cast<float4*>(adv + gbase) = make_float4(oa[0], oa[1], oa[2], oa[3]);
            *reinterpret_cast<float4*>(vt + gbase) = make_float4(ov[0], ov[1], ov[2], ov[3]);
            *reinterpret_cast<float4*>(ret + gbase) = make_float4(orr[0], orr[1], orr[2], orr[3]);
        } else {
            // generic flags / tile not staged: the multipliers again, from global memory (rare)
            const int cnt = (int)((n - base0) < (int64_t)kTile ? (n - base0) : (int64_t)kTile);
            StepMaps<TRUNC64> g = sm;
            g.r = rew + base0; g.d = done + base0; g.v = val + base0;
            g.t = static_cast<const uint8_t*>(trunc) + base0 * kTB;
#pragma unroll
            for (int i = kItems - 1; i >= 0; --i)
                if (j0 + i < cnt) {
                    double aA, aR;
                    g.mults(j0 + i, aA, aR);
                    xA = fma(aA, xA, (double)P.dl[i]);
                    xR = fma(aR, xR, (double)P.r[i]);
                    if (head && gbase + i < n_head) ret_head[gbase + i] = xR;
                    adv[gbase + i] = (float)xA;
                    vt[gbase + i] = (float)((double)P.v[i] + xA);
                    ret[gbase + i] = (float)xR;
                }
        }
    };

    // A(k) runs one tile ahead of B(k-1); two register sets alternate (unrolled by two: no dynamic indexing)
    if (tid == 0)
        for (int kk = 0; kk < kStages && kk < K; ++kk) produce(kk);
    Pending P0, P1;
    phaseA(0, P0);
    int k = 1;
    for (; k + 1 < K; k += 2) {
        phaseA(k, P1);
        phaseB(k - 1, P0);
        phaseA(k + 1, P0);
        phaseB(k, P1);
    }
    if (k < K) {
        phaseA(k, P1);
        phaseB(k - 1, P0);
        phaseB(k, P1);
    } else {
        phaseB(k - 1, P0);
    }
}

// the two record arrays of n steps' tiles (see Workspace)
size_t ws_bytes_for(int64_t n) { return 2 * (size_t)((n + kTile - 1) / kTile) * 4 * sizeof(double); }

bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

template <bool STORE>
int launch_gae(const float* rew, const float* done, const void* trunc, int trunc_is_f64, const float* values,
               int64_t n, double gamma, double lambda, const float* ret_std, float* adv, float* vtarget,
               float* ret, double* ret_head64, int64_t n_head, const double* carry_in, double* summary_out,
               void* wsp, size_t ws_bytes, cudaStream_t s) {
    const size_t need = ws_bytes_for(n);
    if (ws_bytes < need || wsp == nullptr) {
        rlppo::set_error("gae workspace too small: %zu < %zu", ws_bytes, need);
        return RLPPO_ERR_WORKSPACE;
    }
    RLPPO_CHECK_ARG(aligned16(wsp), "gae workspace must be 16-byte aligned");
    const int n_tiles = (int)((n + kTile - 1) / kTile);
    Workspace ws{static_cast<double*>(wsp), static_cast<double*>(wsp) + (size_t)n_tiles * 4};
    RLPPO_CUDA(cudaMemsetAsync(wsp, 0xFF, need, s));   // every record unset (see rec_load)
    const float gl32 = (float)(gamma * lambda);
    bool can_stage = aligned16(rew) && aligned16(done) && aligned16(trunc) && aligned16(values);
    if (STORE) can_stage = can_stage && aligned16(adv) && aligned16(vtarget) && aligned16(ret);
    const size_t smem = (size_t)kStages * stage_bytes(trunc_is_f64 != 0);
    static bool configured[2] = {false, false};
    static int resident[2] = {0, 0};
    auto launch = [&](auto kfn, int which) -> cudaError_t {
        if (!configured[which]) {
            cudaError_t e = cudaFuncSetAttribute(kfn, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                                 (int)(kStages * stage_bytes(true)));
            if (e != cudaSuccess) return e;
            // every CTA of the grid must be able to be resident at once (see the kernel's header comment)
            e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&resident[which], kfn, kThreads, kStages * stage_bytes(true));
            if (e != cudaSuccess) return e;
            if (resident[which] < 1) return cudaErrorLaunchOutOfResources;
            configured[which] = true;
        }
        const int cap = resident[which] * rlppo::num_sms();
        const int grid = n_tiles < cap ? n_tiles : cap;
        kfn<<<grid, kThreads, smem, s>>>(rew, done, trunc, values, n, gamma, gl32, ret_std, adv, vtarget, ret, ret_head64,
                                         n_head, carry_in, summary_out, ws, n_tiles, can_stage);
        return cudaSuccess;
    };
    if (trunc_is_f64) RLPPO_CUDA(launch(gae_scan3_kernel<true, STORE>, 1));
    else RLPPO_CUDA(launch(gae_scan3_kernel<false, STORE>, 0));
    RLPPO_LAUNCH_CHECK();
    return RLPPO_OK;
}

// carry of chunk `rank` = the chunks to its right composed onto 0, rightmost first: x -> b + a * x per chunk
__global__ void compose_carry_kernel(const double* __restrict__ summ, int rank, int world, double* __restrict__ carry) {
    double A = 0.0, R = 0.0;
    for (int k = world - 1; k > rank; --k) {
        A = summ[4 * k + 1] + summ[4 * k + 0] * A;
        R = summ[4 * k + 3] + summ[4 * k + 2] * R;
    }
    carry[0] = A;
    carry[1] = R;
}

}  // namespace

extern "C" {

int rlppo_gae_compose_carry(const double* summaries, int rank, int world, double* carry2, void* stream) {
    RLPPO_REQUIRE_DEVICE();
    RLPPO_CHECK_ARG(summaries && carry2 && world >= 1 && rank >= 0 && rank < world, "bad argument");
    compose_carry_kernel<<<1, 1, 0, static_cast<cudaStream_t>(stream)>>>(summaries, rank, world, carry2);
    RLPPO_LAUNCH_CHECK();
    return RLPPO_OK;
}

size_t rlppo_gae_workspace_bytes(int64_t n) { return ws_bytes_for(n < 1 ? 1 : n); }

int rlppo_gae_f32(const float* rew, const float* done, const void* trunc, int trunc_is_f64, const float* values,
                  int64_t n, double gamma, double lambda, const float* ret_std, float* adv, float* vtarget,
                  float* ret, double* ret_head64, int64_t n_head, const double* carry_in, void* ws,
                  size_t ws_bytes, void* stream) {
    RLPPO_REQUIRE_DEVICE();
    RLPPO_CHECK_ARG(n >= 0, "n must be >= 0");
    if (n == 0) return RLPPO_OK;
    RLPPO_CHECK_ARG(n <= (int64_t)kTile * 0x7fffffff, "n too large");
    RLPPO_CHECK_ARG(rew && done && trunc && values && adv && vtarget && ret, "null pointer");
    return launch_gae<true>(rew, done, trunc, trunc_is_f64, values, n, gamma, lambda, ret_std, adv, vtarget, ret,
                            ret_head64, n_head, carry_in, nullptr, ws, ws_bytes, static_cast<cudaStream_t>(stream));
}

int rlppo_gae_chunk_summary(const float* rew, const float* done, const void* trunc, int trunc_is_f64,
                            const float* values, int64_t n, double gamma, double lambda, const float* ret_std,
                            double* out4, void* ws, size_t ws_bytes, void* stream) {
    RLPPO_REQUIRE_DEVICE();
    RLPPO_CHECK_ARG(n >= 1 && rew && done && trunc && values && out4, "bad argument");
    return launch_gae<false>(rew, done, trunc, trunc_is_f64, values, n, gamma, lambda, ret_std, nullptr, nullptr,
                             nullptr, nullptr, 0, nullptr, out4, ws, ws_bytes, static_cast<cudaStream_t>(stream));
}
}
