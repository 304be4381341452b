// Whole-network fused MLP kernel for the PPO update and for inference (hidden widths <= 256).
//
// The layer-by-layer path (mlp_tcgen05.cu) writes every hidden activation to HBM and reads it back in the next
// launch; for the 256-wide nets of the example config every one of those GEMMs is HBM/latency bound.  This kernel
// runs a 128-row tile of samples through the WHOLE network without leaving the SM:
//
//   x tile (TMA) -> [GEMM l -> TMEM -> bias+ReLU epilogue -> bf16 tile in shared memory = A operand of GEMM l+1] x L
//     policy: -> head GEMM -> softmax/clamp/log-prob/entropy/ratio/clip/KL epilogue -> d(loss)/d(logits) tile
//     value : -> value head as a register dot product inside the last epilogue -> d(loss)/dH_L tile
//   backward data path in the same kernel: dH_l = (dH_{l+1} W_{l+1}) (.) relu'(H_l), the ReLU masks kept as bit masks
//   in the registers of the thread that owns the row, bias gradients reduced with warp shuffles and accumulated in
//   registers across tiles.
//
// Per tile the only HBM traffic is: read x once; write H_1..H_L, d(logits) and dH_L..dH_1 once (the weight-gradient
// GEMMs, which contract over ALL rows, read them back in rlppo_linear_wgrad).  Weights stream from L2 through a
// 2-stage TMA ring.  In inference mode nothing but x, actions/log-probs or values touches HBM.
//
// Warp roles (320 threads, 1 CTA/SM, persistent over tiles, ONE tile in flight per CTA):
//   warp 0      TMA producer: the x tile of the NEXT tile into its own staging buffer + weight k-blocks (3-stage ring)
//   warp 1      TMEM owner; one thread issues tcgen05.mma, TMA-stores finished activation k-blocks, commits barriers
//   warps 2..9  epilogue: warp w owns TMEM lanes 32*(w%4)..+31 (rows); of every 64-column k-block of the output,
//               warps 2-5 take the lower 32 columns and warps 6-9 the upper 32.
// The activation tile (128 rows x <=256 columns bf16, 64 KB) is overwritten IN PLACE by every epilogue (the GEMM that
// read it has completed by then) and there are TWO 256-column TMEM accumulators: the epilogue of layer l releases the
// tile k-block by k-block (a_ready[kb], 8 warp arrivals each), and GEMM l+1 -- which accumulates into the OTHER
// accumulator -- starts on k-block 0 while the epilogue is still producing k-blocks 1..3.  The tensor core therefore
// trails the epilogue warps by one k-block instead of waiting for the whole tile, and the shared memory a second tile
// would need holds a deeper weight ring instead.
// History (profiles/README_r01.md): v1 kept two tiles in flight with one accumulator each and a 2-stage weight ring; its
// cycle trace showed the MMA thread taking ~4.7k cycles to issue 2k cycles of MMAs per layer (waiting for weight
// k-blocks: 64 KB in flight per SM cannot cover the L2 latency) and the epilogue warps idle 27 % of the time.
#include <type_traits>
#include <math.h>

#include "tc_common.cuh"

namespace {

using namespace rlppo;
using namespace rlppo::tc;

constexpr int MAXL = 4;
constexpr int TILE_M = 128;
constexpr int KBLK = 64;
constexpr uint32_t KB_BYTES = TILE_M * KBLK * 2;   // 16 KB: one 64-column k-block of an activation tile
constexpr uint32_t ACT_BYTES = 4 * KB_BYTES;       // 64 KB
constexpr uint32_t WST_BYTES = 256 * KBLK * 2;     // 32 KB: one k-block of a weight operand (<= 256 rows)
constexpr uint32_t MN_CHUNK = 64 * KBLK * 2;       // 8 KB: 64 k-rows x 64 n-columns of an MN-major weight operand
constexpr int MAX_NWST = 3;                        // weight ring stages of 32 KB
constexpr int kThreads = 352;
constexpr int kEpiThreads = 256;
constexpr int MAXPH = 2 * MAXL + 1;

// shared memory (offsets from the 1024-aligned base): [act 64 KB][x stage in_kb*16 KB][weight ring nwst*32 KB][misc]
constexpr uint32_t OFF_ACT = 0;
constexpr uint32_t OFF_XST = ACT_BYTES;
constexpr uint32_t BIAS_FLOATS = (MAXL + 1) * 256;                 // per net: MAXL hidden bias slots + the head slot
constexpr uint32_t MISC_BIAS = 0;                                  // 2 nets x BIAS_FLOATS floats
constexpr uint32_t MISC_ROWX = MISC_BIAS + 2 * BIAS_FLOATS * 4;    // 1280 floats: row-wise exchange planes
constexpr uint32_t ROWX_FLOATS = 1280;
constexpr uint32_t MISC_DB = MISC_ROWX + ROWX_FLOATS * 4;          // 256 floats: column sums of the value head's weight gradient
constexpr uint32_t MISC_MASK = MISC_DB + 256 * 4;                  // ReLU bit masks: [MAXL][4 k-blocks][256 threads] words
constexpr uint32_t MISC_BARS = MISC_MASK + MAXL * 4 * kEpiThreads * 4;
constexpr uint32_t MISC_BYTES = MISC_BARS + 384;     // 19 mbarriers + the TMEM slot + the item ring
constexpr uint32_t SMEM_LIMIT = 232448;                            // 227 KB
static_assert(ACT_BYTES + 2 * KB_BYTES + MISC_BYTES + 1024 + 3 * WST_BYTES <= SMEM_LIMIT,
              "an observation of <= 128 columns must leave room for a 3-stage weight ring (2 stages starve the MMA)");

enum { PH_FWD = 0, PH_FWD_VALUE = 1, PH_HEAD = 2, PH_DGRAD = 3, PH_VALUE_BWD = 4 };
constexpr uint8_t NO_STORE = 0xFF;

struct alignas(16) PhaseDesc {   // one 16-byte word: the duo kernel keeps the table in shared memory and reads a phase with one load
    uint8_t kind;       // PH_*
    uint8_t layer;      // FWD: hidden index (0-based) of the layer produced; DGRAD/VALUE_BWD: hidden index whose ReLU mask applies
    uint8_t n_kb;       // k-blocks of the contraction (0: no GEMM, PH_VALUE_BWD)
    uint8_t wmap;       // index into Maps::w
    uint16_t N;         // accumulator columns = rows of the weight box (multiple of 16, <= 256)
    uint8_t out;        // index into Params::outp of the HBM copy of this phase's output (weight-gradient operand), or NO_STORE
    uint8_t smem;       // 1: the epilogue writes the activation tile (it is the next GEMM's A operand)
    uint8_t wait_kb;    // GEMM-less phase: k-blocks released by the previous epilogue (consumed for barrier parity)
    uint8_t rel_kb;     // k-blocks this phase's epilogue releases (a_ready arrivals), = k-blocks of its output tile
    uint8_t b_mn;       // 1: the weight operand is MN-major (dgrad reads W [out, in] itself: k = out rows, n = in columns,
                        // staged as N/64 chunks of 64 k-rows x 64 n-columns) -- no transposed copy of W exists
};

constexpr int MAXNET = 2;   // one launch runs the tiles of up to two nets (policy + value of the same batch)

struct alignas(64) Maps {
    CUtensorMap x;
    CUtensorMap w[MAXNET][MAXPH];
    CUtensorMap out[MAXNET][MAXPH];   // training: H_l, d(logits), dL/dH_l (weight-gradient operands), TMA-stored per k-block
};

// everything that differs between the nets of one launch
struct NetP {
    int policy;              // 1: discrete policy head, 0: value head
    int n_ph, L;
    int H[MAXL];
    PhaseDesc ph[MAXPH];
    int tail_rel_kb;         // k-blocks the last epilogue releases (consumed by the MMA thread at the end of a tile)
    const float* bias[MAXL + 1];
    float* gbias[MAXL + 1];
    // policy head
    int n_actions, out_kb;
    const float *actions, *old_logp, *adv;
    float inv_batch, clip, ent_coef;
    const float* u_inject;
    uint64_t seed, offset;
    const unsigned long long* d_offset;   // optional device counter added to `offset` (a captured graph keeps sampling fresh numbers)
    int deterministic;
    float* actions_out;
    int64_t* actions_i64_out;
    float* logp_out;
    // value head
    const float* w_head;
    const float* targets;
    float* gw_head;
    float* values_out;
    float* metrics;
};

struct Params {
    int64_t M;
    int num_tiles, in_kb, nwst;
    int n_units;                 // work units per net: tiles (fused_mlp_kernel), or pairs of tiles (fused_duo_kernel)
    int n_nets;                  // work items = n_nets * n_units: item q is unit q % n_units of net q / n_units
    NetP net[MAXNET];
    unsigned int* sched;         // [0] next item to hand out, [1] CTAs that have left (the last one zeroes both)
    uint32_t* mask_scratch;      // duo kernel: gridDim.x x 24 KB of ReLU mask words (L2-resident scratch)
};

// ---- small PTX helpers local to this kernel -------------------------------------------------------------------
__device__ __forceinline__ void tma_store_2d(const CUtensorMap* m, const void* smem_src, int c0, int c1) {
    asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];" ::"l"(
                     reinterpret_cast<uint64_t>(m)),
                 "r"(smem_u32(smem_src)), "r"(c0), "r"(c1)
                 : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_read_all() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void epi_bar_sync() { asm volatile("bar.sync 1, 256;" ::: "memory"); }

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

// lane j returns sum over the 32 lanes of v[j] (v is destroyed): a 31-shuffle reduce-scatter
__device__ __forceinline__ float warp_colsum32(float (&v)[32], int lane) {
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

// 16-column variant: lanes l and l^16 both return the sum over the 32 lanes of v[l & 15]
__device__ __forceinline__ float warp_colsum16(float (&v)[16], int lane) {
#pragma unroll
    for (int w = 8; w >= 1; w >>= 1) {
        const bool up = (lane & w) != 0;
#pragma unroll
        for (int i = 0; i < w; ++i) {
            const float send = up ? v[i] : v[i + w];
            const float keep = up ? v[i + w] : v[i];
            v[i] = keep + __shfl_xor_sync(0xffffffffu, send, w);
        }
    }
    return v[0] + __shfl_xor_sync(0xffffffffu, v[0], 16);
}

__device__ __forceinline__ float bf16_round(float x) { return bf16_bits_to_f32(f32_to_bf16_bits(x)); }
// two floats -> packed bf16x2 in ONE instruction (cvt.rn.bf16x2.f32; `lo` lands in the low half)
__device__ __forceinline__ uint32_t cvt_bf16x2(float lo, float hi) {
    uint32_t r;
    asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
    return r;
}

// max(x, 0) of two floats -> packed bf16x2 in ONE instruction (F2FP.RELU: the ReLU costs nothing)
__device__ __forceinline__ uint32_t cvt_relu_bf16x2(float lo, float hi) {
    uint32_t r;
    asm("cvt.rn.relu.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
    return r;
}

// 32 floats -> 16 packed bf16x2 words
__device__ __forceinline__ void pack32(const float (&v)[32], uint32_t (&w)[16]) {
#pragma unroll
    for (int i = 0; i < 16; ++i) w[i] = cvt_bf16x2(v[2 * i], v[2 * i + 1]);
}
__device__ __forceinline__ void pack32_relu(const float (&v)[32], uint32_t (&w)[16]) {
#pragma unroll
    for (int i = 0; i < 16; ++i) w[i] = cvt_relu_bf16x2(v[2 * i], v[2 * i + 1]);
}
__device__ __forceinline__ uint32_t prmt_b32(uint32_t a, uint32_t b, uint32_t sel) {
    uint32_t r;
    asm("prmt.b32 %0, %1, %2, %3;" : "=r"(r) : "r"(a), "r"(b), "r"(sel));
    return r;
}
// ReLU mask of 32 post-ReLU bf16 values (16 packed words, all halves >= +0) as ONE word.  The epilogue is bound by the
// ALU pipe (LOP3 / PRMT / SHF / ISETP issue every other cycle per scheduler), so the compare runs on the other pipe:
// HSET2.BF16 turns each packed pair into 0xFFFF / 0x0000 halves (h > 0), one byte permute gathers the top bytes of four of
// them (0xFF / 0x00) and one LOP3 keeps bit 7 - q of each byte for group q.  Element 4q+e lands in bit 8e + 7 - q
// (relu_mask_bit); the reference tests H > 0 on fp32, which is the same set once H is rounded to bf16.
__device__ __forceinline__ uint32_t relu_mask32(const uint32_t (&w)[16]) {
    uint32_t m[4] = {0u, 0u, 0u, 0u};
#pragma unroll
    for (int q = 0; q < 8; ++q) {
        uint32_t f0, f1;
        asm("set.gt.u32.bf16x2 %0, %1, %2;" : "=r"(f0) : "r"(w[2 * q]), "r"(0u));
        asm("set.gt.u32.bf16x2 %0, %1, %2;" : "=r"(f1) : "r"(w[2 * q + 1]), "r"(0u));
        m[q & 3] |= prmt_b32(f0, f1, 0x7531u) & (0x80808080u >> q);
    }
    return (m[0] | m[1]) | (m[2] | m[3]);
}
// w (16 packed bf16x2 words = 32 values) with the values whose ReLU mask bit is clear zeroed: group q's four bits are moved
// to the top of the four bytes by one shift (IMAD.SHL, the other pipe), a sign-replicating byte permute expands two of them
// to a 0xFFFF / 0x0000 pair, and one AND applies it -- two ALU instructions per packed word instead of a bit test and a
// select per value
__device__ __forceinline__ void apply_relu_mask32(uint32_t (&w)[16], uint32_t bits) {
#pragma unroll
    for (int q = 0; q < 8; ++q) {
        const uint32_t t = bits << q;
        w[2 * q] &= prmt_b32(t, 0u, 0x9988u);        // bytes (sign b0, sign b0, sign b1, sign b1): values 4q, 4q+1
        w[2 * q + 1] &= prmt_b32(t, 0u, 0xBBAAu);    // values 4q+2, 4q+3
    }
}
__device__ __forceinline__ constexpr int relu_mask_bit(int i) { return 8 * (i & 3) + 7 - (i >> 2); }
// 32 consecutive columns [32*chunk32, +32) of one row into a K-major SWIZZLE_128B activation tile
__device__ __forceinline__ void sts_chunk_sw128(uint8_t* buf, int row, int chunk32, const uint32_t (&w)[16]) {
    uint8_t* kb = buf + (chunk32 >> 1) * KB_BYTES + row * 128;
    const int base16 = (chunk32 & 1) * 4;
#pragma unroll
    for (int t = 0; t < 4; ++t)
        *reinterpret_cast<uint4*>(kb + (((base16 + t) ^ (row & 7)) << 4)) = make_uint4(w[4 * t], w[4 * t + 1], w[4 * t + 2], w[4 * t + 3]);
}
// 16 consecutive columns [16*chunk16, +16) of one row into a K-major SWIZZLE_128B activation tile
__device__ __forceinline__ void sts_chunk16_sw128(uint8_t* buf, int row, int chunk16, const uint32_t (&w)[8]) {
    uint8_t* kb = buf + (chunk16 >> 2) * KB_BYTES + row * 128;
    const int base16 = (chunk16 & 3) * 2;
#pragma unroll
    for (int t = 0; t < 2; ++t)
        *reinterpret_cast<uint4*>(kb + (((base16 + t) ^ (row & 7)) << 4)) = make_uint4(w[4 * t], w[4 * t + 1], w[4 * t + 2], w[4 * t + 3]);
}

struct EpiCtx {
    uint8_t* act;
    float* s_bias;
    float* s_rowx;
    uint32_t* s_mask;     // this thread's column of the mask planes: word (layer * 4 + kb) lives at s_mask[(layer*4+kb) * 256]
    uint64_t* a_ready;    // [4], one per k-block of the activation tile, 8 arrivals (epilogue warps)
    int lane, quarter, half, row_in_tile;
};

// This warp's part of output k-block `kb` is written and its TMEM reads for it are done: one arrival per warp; the MMA
// thread may then read that k-block as the next GEMM's A operand (and TMA-store it).
__device__ __forceinline__ void release_kb(const EpiCtx& e, int kb) {
    tc_fence_before();
    fence_proxy_async();
    __syncwarp();
    if (e.lane == 0) mbar_arrive(e.a_ready + kb);          // the store thread and the MMA thread wait on it
}

template <bool TRAIN>
__global__ void __launch_bounds__(kThreads, 1) fused_mlp_kernel(const __grid_constant__ Maps maps, const Params p) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
    uint8_t* act = smem + OFF_ACT;
    uint8_t* xst = smem + OFF_XST;
    uint8_t* wring = xst + p.in_kb * KB_BYTES;
    uint8_t* misc = wring + p.nwst * WST_BYTES;
    float* s_bias = reinterpret_cast<float*>(misc + MISC_BIAS);
    float* s_rowx = reinterpret_cast<float*>(misc + MISC_ROWX);
    float* s_db = reinterpret_cast<float*>(misc + MISC_DB);
    uint32_t* s_mask = reinterpret_cast<uint32_t*>(misc + MISC_MASK);
    uint64_t* wfull = reinterpret_cast<uint64_t*>(misc + MISC_BARS);
    uint64_t* wempty = wfull + MAX_NWST;
    uint64_t* x_full = wempty + MAX_NWST;   // [1]
    uint64_t* x_free = x_full + 1;          // [1]
    uint64_t* a_ready = x_free + 1;         // [4]
    uint64_t* acc_full = a_ready + 4;       // [2]: one per accumulator
    uint64_t* st_done = acc_full + 2;       // [1]: the TMA stores of a phase's output have finished reading shared memory
    uint64_t* tile_full = st_done + 1;      // [2]: the producer has published the CTA's next tile index
    uint64_t* tile_empty = tile_full + 2;   // [2]: every consumer role has read it
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tile_empty + 2);
    volatile int* tile_ring = reinterpret_cast<volatile int*>(tmem_slot + 1);   // [2]

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (threadIdx.x == 0) {
        tma_prefetch_desc(&maps.x);
        for (int i = 0; i < MAX_NWST; ++i) {
            mbar_init(&wfull[i], 1);
            mbar_init(&wempty[i], 1);
        }
        mbar_init(x_full, 1);
        mbar_init(x_free, 1);
        for (int i = 0; i < 4; ++i) mbar_init(&a_ready[i], 8);
        mbar_init(&acc_full[0], 1);
        mbar_init(&acc_full[1], 1);
        mbar_init(st_done, 1);
        const int consumers = TRAIN ? 10 : 9;           // warp 1's thread, (training) store thread, 8 epilogue warps
        for (int i = 0; i < 2; ++i) {
            mbar_init(&tile_full[i], 1);
            mbar_init(&tile_empty[i], consumers);
        }
        fence_barrier_init();
    }
    if (warp == 1) tmem_alloc(tmem_slot, 512);
    // PDL: everything above ran while the previous kernel of the stream was still draining; its outputs (x, parameters)
    // are read from here on.  All CTAs of this grid are resident, so the next kernel may be scheduled as SMs free up.
    pdl_wait();
    pdl_trigger();
    // biases (and the value head's weights) into shared memory, one table per net: slot l < L hidden biases, slot MAXL the head
    for (int i = threadIdx.x; i < p.n_nets * (int)BIAS_FLOATS; i += kThreads) {
        const int ni = i >= (int)BIAS_FLOATS ? 1 : 0;
        const NetP& np = p.net[ni];
        const int j = i - ni * (int)BIAS_FLOATS;
        const int l = j >> 8, c = j & 255;
        float b = 0.f;
        if (l < np.L) {
            if (c < np.H[l]) b = __ldg(np.bias[l] + c);
        } else if (l == MAXL) {
            if (np.policy) {
                // padding columns of the logits: a large negative bias, so exp() of them is exactly 0
                b = c < np.n_actions ? (np.bias[MAXL] != nullptr ? __ldg(np.bias[MAXL] + c) : 0.f) : -1e30f;
            } else {
                if (c < np.H[np.L - 1]) b = __ldg(np.w_head + c);
            }
        }
        s_bias[i] = b;
    }
    for (int i = threadIdx.x; i < 256; i += kThreads) s_db[i] = 0.f;
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    // Work items (net, tile) are handed out dynamically from a global counter, the first net's tiles first (the policy
    // net's: they take longest, so the launch ends on the cheaper value tiles): 2 x 391 items over 148 CTAs instead of two
    // launches of 391 tiles that each end on a third, 64 %-full round.  The producer thread fetches the next item one
    // ahead and publishes it to the other roles through a two-slot ring; -1 ends the CTA.

    if (warp == 0) {
        // ===================== TMA producer =====================
        if (lane == 0) {
            uint32_t ws = 0, wpar = 0;
            for (int it = 0;; ++it) {
                const int slot = it & 1;
                mbar_wait(&tile_empty[slot], ((it >> 1) & 1) ^ 1);
                int q = (int)atomicAdd(p.sched, 1u);
                if (q >= p.n_nets * p.n_units) q = -1;
                tile_ring[slot] = q;
                mbar_arrive(&tile_full[slot]);
                if (q < 0) break;
                const int ni = q >= p.n_units ? 1 : 0;
                const int tile = q - ni * p.n_units;
                const NetP& np = p.net[ni];
                mbar_wait(x_free, (it & 1) ^ 1);          // GEMM 0 of the previous tile has read the staging buffer
                mbar_expect_tx(x_full, p.in_kb * KB_BYTES);
                for (int kb = 0; kb < p.in_kb; ++kb)
                    tma_load_2d(&maps.x, x_full, xst + kb * KB_BYTES, kb * KBLK, tile * TILE_M);
                for (int ph = 0; ph < np.n_ph; ++ph) {
                    const PhaseDesc& d = np.ph[ph];
                    for (int kb = 0; kb < d.n_kb; ++kb) {
                        mbar_wait(&wempty[ws], wpar ^ 1);
                        mbar_expect_tx(&wfull[ws], (uint32_t)d.N * 128u);
                        uint8_t* dst = wring + ws * WST_BYTES;
                        if (d.b_mn) {
                            for (int c = 0; c < (d.N >> 6); ++c)
                                tma_load_2d(&maps.w[ni][d.wmap], &wfull[ws], dst + c * MN_CHUNK, c * 64, kb * KBLK);
                        } else {
                            tma_load_2d(&maps.w[ni][d.wmap], &wfull[ws], dst, kb * KBLK, 0);
                        }
                        if (++ws == (uint32_t)p.nwst) {
                            ws = 0;
                            wpar ^= 1;
                        }
                    }
                }
            }
        }
    } else if (warp == 1) {
        // ===================== MMA issuer =====================
        if (lane == 0) {
            uint32_t ws = 0, wpar = 0;
            uint32_t g = 0;                        // GEMMs issued so far: GEMM g accumulates into accumulator g & 1
            uint32_t apar = 0;                     // bit kb: parity of a_ready[kb] to wait for next (registers, not a local array)
            for (int it = 0;; ++it) {
                mbar_wait(&tile_full[it & 1], (it >> 1) & 1);
                const int q = tile_ring[it & 1];
                mbar_arrive(&tile_empty[it & 1]);
                if (q < 0) break;
                const NetP& np = p.net[q >= p.n_units ? 1 : 0];
#pragma unroll 1
                for (int ph = 0; ph < np.n_ph; ++ph) {
                    const PhaseDesc& d = np.ph[ph];
                    if (d.n_kb > 0) {
                        const uint32_t idesc = umma_idesc_bf16(TILE_M, d.N, 0, d.b_mn);
                        const uint32_t d_tmem = tmem_base + (g & 1u) * 256u;
                        for (int kb = 0; kb < d.n_kb; ++kb) {
                            uint32_t a_addr;
                            if (ph == 0) {
                                if (kb == 0) {
                                    mbar_wait(x_full, it & 1);
                                    tc_fence_after();
                                }
                                a_addr = smem_u32(xst + kb * KB_BYTES);
                            } else {
                                mbar_wait(&a_ready[kb], (apar >> kb) & 1u);   // k-block kb of the previous epilogue's output
                                apar ^= 1u << kb;
                                tc_fence_after();
                                a_addr = smem_u32(act + kb * KB_BYTES);
                            }
                            mbar_wait(&wfull[ws], wpar);
                            tc_fence_after();
                            const uint32_t b_addr = smem_u32(wring + ws * WST_BYTES);
#pragma unroll
                            for (int k = 0; k < KBLK / 16; ++k) {
                                const uint64_t ad = umma_smem_desc(a_addr + k * 32, 16, 1024);
                                const uint64_t bd = d.b_mn ? umma_smem_desc(b_addr + k * (16 * 128), MN_CHUNK, 1024)
                                                           : umma_smem_desc(b_addr + k * 32, 16, 1024);
                                umma_bf16(d_tmem, ad, bd, idesc, (kb | k) != 0 ? 1u : 0u);
                            }
                            umma_commit(&wempty[ws]);
                            if (++ws == (uint32_t)p.nwst) {
                                ws = 0;
                                wpar ^= 1;
                            }
                        }
                        if (ph == 0) umma_commit(x_free);      // the staging buffer can take the next tile's x
                        umma_commit(&acc_full[g & 1u]);
                        ++g;
                    } else {
                        // GEMM-less phase (value net: dL/dH_L from the accumulator of the last forward GEMM, still in
                        // TMEM): consume the previous epilogue's releases, then hand the SAME accumulator back
                        for (int kb = 0; kb < d.wait_kb; ++kb) {
                            mbar_wait(&a_ready[kb], (apar >> kb) & 1u);
                            apar ^= 1u << kb;
                        }
                        mbar_arrive(&acc_full[(g - 1u) & 1u]);
                    }
                }
                // tail: the last epilogue's releases (barrier parity; also: every epilogue warp is done with both
                // accumulators and the activation tile before the next tile's first GEMM / epilogue touch them)
                for (int kb = 0; kb < np.tail_rel_kb; ++kb) {
                    mbar_wait(&a_ready[kb], (apar >> kb) & 1u);
                    apar ^= 1u << kb;
                }
            }
        }
    } else if (warp == 10) {
        // ===================== store thread (training) =====================
        // Every k-block an epilogue releases is TMA-stored from the activation tile to its HBM tensor (weight-gradient
        // operand); st_done[kb] tells the epilogue warps when the store has finished READING shared memory, i.e. when the
        // next epilogue may overwrite that k-block in place.  The MMA thread never waits for stores.
        if (TRAIN && lane == 0) {
            uint32_t apar = 0;
            for (int it = 0;; ++it) {
                mbar_wait(&tile_full[it & 1], (it >> 1) & 1);
                const int q = tile_ring[it & 1];
                mbar_arrive(&tile_empty[it & 1]);
                if (q < 0) break;
                const int ni = q >= p.n_units ? 1 : 0;
                const int tile = q - ni * p.n_units;
                const NetP& np = p.net[ni];
#pragma unroll 1
                for (int ph = 0; ph < np.n_ph; ++ph) {
                    const PhaseDesc& d = np.ph[ph];
                    const bool storing = d.out != NO_STORE;
                    for (int kb = 0; kb < d.rel_kb; ++kb) {
                        mbar_wait(&a_ready[kb], (apar >> kb) & 1u);
                        apar ^= 1u << kb;
                        if (!storing) continue;
                        tma_store_2d(&maps.out[ni][d.out], act + kb * KB_BYTES, kb * KBLK, tile * TILE_M);
                        bulk_commit();
                    }
                    if (d.rel_kb > 0) {
                        // ONE completion signal per phase, storing or not: the epilogue waits for it before its next phase, so
                        // it is never more than one completion of a_ready ahead of this thread (two would alias the parity).
                        // The next epilogue starts a whole GEMM (>= 1k cycles) after the last release: the reads are long done
                        if (storing) bulk_wait_read_all();
                        mbar_arrive(st_done);
                    }
                }
            }
            asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");   // all stores complete before the CTA exits
        }
    } else {
        // ===================== epilogue warps =====================
        EpiCtx e;
        e.act = act;
        e.s_bias = s_bias;
        e.s_rowx = s_rowx;
        e.s_mask = s_mask + (threadIdx.x - 64);
        e.a_ready = a_ready;
        e.lane = lane;
        e.quarter = warp & 3;
        e.half = (warp - 2) >> 2;
        e.row_in_tile = e.quarter * 32 + lane;

        float dv_keep = 0.f;   // value net: d(loss)/dv of this thread's row, kept from the forward tail
        float m0 = 0.f, m1 = 0.f, m2 = 0.f, m3 = 0.f, mrows = 0.f;   // policy metric partial sums of this thread's rows
        float vm0 = 0.f, vm1 = 0.f, vrows = 0.f;                     // value net: squared error, head bias gradient, rows
        // column sums (bias gradients, value-head weight gradient) accumulate in shared memory: lane j of a warp holds the
        // partial sum of column 32c + j over the warp's 32 rows; four warps (row quarters) add into the same word
        auto db_add = [&](int c, float v) { atomicAdd(&s_db[c * 32 + e.lane], v); };

        uint32_t g = 0;                  // mirrors the MMA thread's GEMM counter
        uint32_t fpar = 0;               // bit a: parity of acc_full[a] to wait for next
        uint32_t pend = 0;               // the previous storing phase's TMA stores have not been waited for yet
        uint32_t scnt = 0;               // parity of st_done to wait for next
        // before a phase overwrites the activation tile in place: the stores of the tile's previous contents must have read it
        auto wait_stores = [&]() {
            if (pend) {
                mbar_wait(st_done, scnt);
                scnt ^= 1u;
                pend = 0;
            }
        };
        for (int it = 0;; ++it) {
          mbar_wait(&tile_full[it & 1], (it >> 1) & 1);
          const int q = tile_ring[it & 1];
          __syncwarp();
          if (lane == 0) mbar_arrive(&tile_empty[it & 1]);
          if (q < 0) break;
          const int ni = q >= p.n_units ? 1 : 0;
          const int tile = q - ni * p.n_units;
          const NetP& np = p.net[ni];
          const float* s_bias_n = s_bias + ni * (int)BIAS_FLOATS;   // this net's bias table
          const int64_t row = (int64_t)tile * TILE_M + e.row_in_tile;
          const bool row_ok = row < p.M;
#pragma unroll 1
          for (int ph = 0; ph < np.n_ph; ++ph) {
                const PhaseDesc& d = np.ph[ph];
                uint32_t acc;
                if (d.n_kb > 0) {
                    acc = g & 1u;
                    ++g;
                } else {
                    acc = (g - 1u) & 1u;
                }
                mbar_wait(&acc_full[acc], (fpar >> acc) & 1u);
                fpar ^= 1u << acc;
                tc_fence_after();
                // the tile is overwritten in place: its last stores must have read it (and the store thread has seen every
                // release of the previous phase)
                if (TRAIN) wait_stores();
                const uint32_t trow = tmem_base + ((uint32_t)(e.quarter * 32) << 16) + acc * 256u;
                uint8_t* dst = act;      // in place: the GEMM that read this tile has completed
                const int li = d.layer;

#define RLPPO_RELEASE_KB(j) release_kb(e, j)
#define RLPPO_MASK_ST(l, kb, v) e.s_mask[((l) * 4 + (kb)) * kEpiThreads] = (v)
#define RLPPO_MASK_LD(l, kb) e.s_mask[((l) * 4 + (kb)) * kEpiThreads]
#include "fused_epilogue.inc"
#undef RLPPO_MASK_ST
#undef RLPPO_MASK_LD
#undef RLPPO_RELEASE_KB
                if (TRAIN && d.rel_kb > 0) pend = 1u;
          }
        }
        // ---- metrics (the column sums are flushed by the whole CTA below) ----
        if (TRAIN && e.half == 0) {
            for (int ni = 0; ni < p.n_nets; ++ni) {
                const NetP& np = p.net[ni];
                if (np.metrics == nullptr) continue;
                if (np.policy) {
                    const float r0 = warp_sum(m0), r1 = warp_sum(m1), r2 = warp_sum(m2), r3 = warp_sum(m3),
                                rr = warp_sum(mrows);
                    if (e.lane == 0 && rr > 0.f) {
                        atomicAdd(np.metrics + 0, r0);
                        atomicAdd(np.metrics + 1, r1);
                        atomicAdd(np.metrics + 2, r2);
                        atomicAdd(np.metrics + 3, r3);
                        atomicAdd(np.metrics + 4, rr);
                    }
                } else {
                    const float r0 = warp_sum(vm0), r1 = warp_sum(vm1), rr = warp_sum(vrows);
                    if (e.lane == 0 && rr > 0.f) {
                        atomicAdd(np.metrics + 5, r0);
                        atomicAdd(np.metrics + 6, rr);
                        if (np.gbias[MAXL] != nullptr) atomicAdd(np.gbias[MAXL], r1);
                    }
                }
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        tc_fence_after();
        tmem_dealloc(tmem_base, 512);
    }
    if (threadIdx.x == 0) {
        // every CTA has drawn its last (out-of-range) index by now: the last CTA to leave re-arms the scheduler words
        if (atomicAdd(p.sched + 1, 1u) == gridDim.x - 1) {
            p.sched[0] = 0;
            p.sched[1] = 0;
            __threadfence();
        }
    }
    if (TRAIN) {
        // flush the shared-memory column sums of the value head's weight gradient; the bias gradients of every Linear are
        // column sums of tiles the weight-gradient kernel reads anyway and are formed there (rlppo_wgrad_multi)
        for (int ni = 0; ni < p.n_nets; ++ni) {
            const NetP& np = p.net[ni];
            if (np.policy || np.gw_head == nullptr) continue;
            for (int c = threadIdx.x; c < np.H[np.L - 1]; c += kThreads) atomicAdd(np.gw_head + c, s_db[c]);
        }
    }
}

// ---------------------------------------------------------------------------------------------------------------
// fused_duo_kernel: CTA pairs with TWO tiles in flight per CTA (training).
//
// The single-tile kernel above is a chain per tile: GEMM -> epilogue -> GEMM ..., in which the tensor core waits for the
// epilogue's k-blocks and the epilogue warps wait for the GEMM's tail at every phase boundary: ~13 k of a tile's 36 k
// cycles.  Here every CTA keeps two tiles ("slots") resident, each with its own activation buffer (in place, as before) and its own 256-column TMEM accumulator, and all roles walk the same
// deterministic sequence  step n -> slot n & 1 -> that slot's next phase : while the eight epilogue warps work on one
// slot, the GEMM of the other slot's next phase runs, so MMA time, weight latency and the pair's signalling latency hide
// behind an epilogue instead of sitting between two of them.  What makes the second 64 KB buffer fit is the pair: each
// CTA stages only its N/2 half of a weight k-block (16 KB stages; both CTAs' TMA loads complete on the LEADER's barrier
// -- cp.async.bulk.tensor.cta_group::2 -- so a stage's round trip is MMA completion -> multicast commit -> TMA from L2, with
// no relay hop), the ReLU masks (24 KB for two slots) live in a per-CTA global scratch that stays in L2 (written by the
// forward epilogue, prefetched into registers before a backward epilogue waits for its accumulator; thread-local memory
// was tried and made the backward epilogues 2x slower), which buys a 5-deep ring (108.3 us per launch with three
// stages, 104.0 with five: tools/time_fused.py), and the x tile of an item is loaded straight into the slot's activation
// buffer (no staging buffer; its latency hides behind the other slot too).  A GEMM waits for the WHOLE previous epilogue
// of its slot (one barrier per slot, no k-block hand-over).
// Roles per CTA: producer (x tiles, weight halves), warp 1 = MMA issuer (leader only), eight epilogue warps, store
// thread.  Items (net, pair of tiles) are dealt out statically (see DuoWalk); a slot takes its next item when its current
// one is finished, in walk order, so every role of both CTAs replays the same assignment.
// The kernel is bound by its epilogue warps (profiles/README_r02.md section 2b): 168 registers per thread is a hard cap
// with 11 warps, and a destination register of an in-flight tcgen05.ld must never be spilled -- check STACK:0 / 16
// (cuobjdump -res-usage) after every change to fused_epilogue.inc.
// ---------------------------------------------------------------------------------------------------------------
constexpr uint32_t DUO_STAGE = WST_BYTES / 2;                      // 16 KB: this CTA's half of a weight k-block
constexpr int DUO_NST = 5;                                         // 80 KB of weight halves in flight per CTA
constexpr int DUO_MAXL = 3;                                        // hidden layers (ReLU mask words per thread: 2 slots x 3 x 4)
constexpr uint32_t DUO_OFF_RING = 2 * ACT_BYTES;
constexpr uint32_t DUO_OFF_MISC = DUO_OFF_RING + DUO_NST * DUO_STAGE;
constexpr uint32_t DUO_MISC_BARS = MISC_DB + 256 * 4;              // (the ReLU masks live in a global scratch here)
constexpr uint32_t DUO_SMEM = DUO_OFF_MISC + DUO_MISC_BARS + 256 + 2 * MAXPH * 16 + 1024;   // barriers, phase table, alignment slack
static_assert(sizeof(PhaseDesc) == 16, "one phase = one 16-byte shared-memory word");
static_assert(DUO_SMEM <= SMEM_LIMIT, "two activation tiles + a 5 x 16 KB ring + misc must fit in 227 KB");

// the walk every role of both CTAs replays: step n works on slot n & 1, one phase of that slot's current item.  The state
// is kept in scalars selected by the slot bit (arrays indexed by it lived in local memory: ~600 cycles per step).
// Items are dealt out statically: cluster c takes items c, c + n_clusters, ... (policy items first, they are the longer
// ones) -- every role derives the same sequence with no shared counter and no hand-over (the dynamic ring cost the producer
// a global atomic round trip at every item boundary, with the weight ring draining behind it).
struct DuoWalk {
    int ph0 = 0, ph1 = 0, nph0 = 0, nph1 = 0, ni0 = 0, ni1 = 0, tile0 = 0, tile1 = 0, items0 = 0, items1 = 0, fetches = 0;
    bool alive0 = true, alive1 = true;
};
#define DUO_SEL(w, f, s) ((s) ? (w).f##1 : (w).f##0)
#define DUO_SET(w, f, s, v)    \
    do {                       \
        if (s) (w).f##1 = (v); \
        else (w).f##0 = (v);   \
    } while (0)

__global__ void __launch_bounds__(kThreads, 1) fused_duo_kernel(const __grid_constant__ Maps maps, const Params p) {
    constexpr bool TRAIN = true;
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
    uint8_t* ring = smem + DUO_OFF_RING;
    uint8_t* misc = smem + DUO_OFF_MISC;
    const uint32_t rank = cluster_ctarank();
    const bool leader = rank == 0;
    float* s_bias = reinterpret_cast<float*>(misc + MISC_BIAS);
    float* s_rowx = reinterpret_cast<float*>(misc + MISC_ROWX);
    float* s_db = reinterpret_cast<float*>(misc + MISC_DB);
    uint64_t* wfull = reinterpret_cast<uint64_t*>(misc + DUO_MISC_BARS);   // [5] (leader) both halves of stage i have landed
    uint64_t* wempty = wfull + DUO_NST;      // [5] the GEMM has read stage i (multicast commit)
    uint64_t* x_full = wempty + DUO_NST;     // [2] (leader) slot s: both CTAs' x tiles have landed in act[s]
    uint64_t* x_free = x_full + 2;           // [2] slot s: the last stores of the finished item have read act[s]
    uint64_t* a_done = x_free + 2;           // [2] (leader) slot s: both CTAs' epilogue warps finished the phase (16 arrivals)
    uint64_t* acc_full = a_done + 2;         // [2] slot s: the GEMM into accumulator s is complete (multicast commit)
    uint64_t* st_done = acc_full + 2;        // [2] slot s: the store thread is through with the phase (its stores have read act[s])
    uint64_t* a_kb = st_done + 2;            // [2][4] slot s, k-block kb of the tile is written (this CTA's 8 warps): store thread
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(a_kb + 8);
    const PhaseDesc* s_ph = reinterpret_cast<const PhaseDesc*>(misc + DUO_MISC_BARS + 256);   // [2 nets][MAXPH]

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (threadIdx.x == 0) {
        tma_prefetch_desc(&maps.x);
        for (int i = 0; i < 8; ++i) mbar_init(&a_kb[i], 8);
        for (int i = 0; i < DUO_NST; ++i) {
            mbar_init(&wfull[i], 1);
            mbar_init(&wempty[i], 1);
        }
        for (int s = 0; s < 2; ++s) {
            mbar_init(&x_full[s], 1);
            mbar_init(&x_free[s], 1);
            mbar_init(&a_done[s], 16);
            mbar_init(&acc_full[s], 1);
            mbar_init(&st_done[s], 1);
        }
        fence_barrier_init();
    }
    if (warp == 1) tmem_alloc_pair(tmem_slot, 512);
    pdl_wait();
    pdl_trigger();
    for (int i = threadIdx.x; i < p.n_nets * (int)BIAS_FLOATS; i += kThreads) {
        const int ni = i >= (int)BIAS_FLOATS ? 1 : 0;
        const NetP& np = p.net[ni];
        const int j = i - ni * (int)BIAS_FLOATS;
        const int l = j >> 8, c = j & 255;
        float b = 0.f;
        if (l < np.L) {
            if (c < np.H[l]) b = __ldg(np.bias[l] + c);
        } else if (l == MAXL) {
            if (np.policy) b = c < np.n_actions ? (np.bias[MAXL] != nullptr ? __ldg(np.bias[MAXL] + c) : 0.f) : -1e30f;
            else if (c < np.H[np.L - 1]) b = __ldg(np.w_head + c);
        }
        s_bias[i] = b;
    }
    for (int i = threadIdx.x; i < 256; i += kThreads) s_db[i] = 0.f;
    for (int i = threadIdx.x; i < p.n_nets * MAXPH; i += kThreads)
        const_cast<PhaseDesc*>(s_ph)[i] = p.net[i / MAXPH].ph[i % MAXPH];
    tc_fence_before();
    __syncthreads();
    cluster_sync_all();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    const int cluster_id = (int)(blockIdx.x >> 1), n_clusters = (int)(gridDim.x >> 1);
    const int total_items = p.n_nets * p.n_units;
    const int nph_net0 = p.net[0].n_ph, nph_net1 = p.net[1].n_ph;
    // next item of this cluster for slot s: the same arithmetic in every role of both CTAs
    auto next_item = [&](DuoWalk& w, int s) -> bool {
        const int q = cluster_id + (w.fetches++) * n_clusters;
        if (q >= total_items) {
            DUO_SET(w, alive, s, false);
            return false;
        }
        const int ni = q >= p.n_units ? 1 : 0;
        DUO_SET(w, ni, s, ni);
        DUO_SET(w, tile, s, 2 * (q - ni * p.n_units) + (int)rank);
        DUO_SET(w, ph, s, 0);
        DUO_SET(w, nph, s, ni ? nph_net1 : nph_net0);
        DUO_SET(w, items, s, DUO_SEL(w, items, s) + 1);
        return true;
    };
#define DUO_WALK_BEGIN(w)                                                     \
    for (int n = 0;; ++n) {                                                   \
        const int s = n & 1;                                                  \
        if (!DUO_SEL(w, alive, s)) {                                          \
            if (!DUO_SEL(w, alive, s ^ 1)) break;                             \
            continue;                                                         \
        }                                                                     \
        if (DUO_SEL(w, ph, s) == DUO_SEL(w, nph, s) && !next_item(w, s)) {    \
            if (!DUO_SEL(w, alive, s ^ 1)) break;                             \
            continue;                                                         \
        }                                                                     \
        const int ph = DUO_SEL(w, ph, s);                                     \
        DUO_SET(w, ph, s, ph + 1);                                            \
        const int ni = DUO_SEL(w, ni, s);                                     \
        const int tile_s = DUO_SEL(w, tile, s);                               \
        const int items_s = DUO_SEL(w, items, s);                             \
        const bool last_ph = ph + 1 == DUO_SEL(w, nph, s);                    \
        const NetP& np = p.net[ni];                                           \
        const PhaseDesc d = s_ph[ni * MAXPH + ph];                            \
        (void)d; (void)np; (void)tile_s; (void)items_s; (void)last_ph;
#define DUO_WALK_END }

    if (warp == 0) {
        // ===================== producer: x tiles and this CTA's weight halves, in walk order =====================
        if (lane == 0) {
            DuoWalk w;
            uint32_t ws = 0, wpar = 0;
            DUO_WALK_BEGIN(w)
                if (ph == 0) {
                    // the item's x tile, straight into the slot's activation buffer once the previous item's stores have read
                    // it: item k of the slot (k = items_s - 1) waits for completion k - 1 of x_free
                    mbar_wait(&x_free[s], (uint32_t)(items_s & 1));
                    if (leader) mbar_expect_tx(&x_full[s], 2u * p.in_kb * KB_BYTES);      // both CTAs' tiles, counted in the leader
                    for (int kb = 0; kb < p.in_kb; ++kb)
                        tma_load_2d_leaderbar(&maps.x, &x_full[s], smem + s * ACT_BYTES + kb * KB_BYTES, kb * KBLK, tile_s * TILE_M);
                }
                const int nh = d.N >> 1;
                for (int kb = 0; kb < d.n_kb; ++kb) {
                    mbar_wait(&wempty[ws], wpar ^ 1);
                    if (leader) mbar_expect_tx(&wfull[ws], (uint32_t)d.N * 128u);      // both halves complete on the leader's barrier
                    uint8_t* dst = ring + ws * DUO_STAGE;
                    if (d.b_mn) {
                        for (int c = 0; c < (nh >> 6); ++c)
                            tma_load_2d_leaderbar(&maps.w[ni][d.wmap], &wfull[ws], dst + c * MN_CHUNK, (int)rank * nh + c * 64,
                                                  kb * KBLK);
                    } else {
                        tma_load_2d_leaderbar(&maps.w[ni][d.wmap], &wfull[ws], dst, kb * KBLK, (int)rank * nh);
                    }
                    if (++ws == DUO_NST) {
                        ws = 0;
                        wpar ^= 1;
                    }
                }
            DUO_WALK_END
        }
    } else if (warp == 1) {
        if (lane == 0 && leader) {
            // ===================== MMA issuer =====================
            DuoWalk w;
            uint32_t ws = 0, wpar = 0;
            uint32_t epi_cnt[2] = {0u, 0u};        // phases of slot s issued so far (every one ends with an epilogue)
            DUO_WALK_BEGIN(w)
                const uint32_t d_tmem = tmem_base + (uint32_t)s * 256u;
                uint8_t* act = smem + s * ACT_BYTES;
                // this slot's previous epilogue, in both CTAs (every completion of a_done[s] is waited for, in order)
                if (epi_cnt[s] > 0u) mbar_wait(&a_done[s], (epi_cnt[s] - 1u) & 1u);
                if (ph == 0) mbar_wait(&x_full[s], (items_s - 1) & 1);       // both CTAs' x tiles
                tc_fence_after();
                if (d.n_kb > 0) {
                    const uint32_t idesc = umma_idesc_bf16(2 * TILE_M, d.N, 0, d.b_mn);
                    for (int kb = 0; kb < d.n_kb; ++kb) {
                        mbar_wait(&wfull[ws], wpar);                                   // both CTAs' halves
                        tc_fence_after();
                        const uint32_t a_addr = smem_u32(act + kb * KB_BYTES);
                        const uint32_t b_addr = smem_u32(ring + ws * DUO_STAGE);
#pragma unroll
                        for (int k = 0; k < KBLK / 16; ++k) {
                            const uint64_t ad = umma_smem_desc(a_addr + k * 32, 16, 1024);
                            const uint64_t bd = d.b_mn ? umma_smem_desc(b_addr + k * (16 * 128), MN_CHUNK, 1024)
                                                       : umma_smem_desc(b_addr + k * 32, 16, 1024);
                            umma_bf16_pair(d_tmem, ad, bd, idesc, (kb | k) != 0 ? 1u : 0u);
                        }
                        umma_commit_pair(&wempty[ws]);
                        if (++ws == DUO_NST) {
                            ws = 0;
                            wpar ^= 1;
                        }
                    }
                    umma_commit_pair(&acc_full[s]);
                } else {
                    // GEMM-less phase (value net: dL/dH_L from the accumulator of the last forward GEMM, still in TMEM)
                    mbar_arrive(&acc_full[s]);
                    mbar_arrive_cta(&acc_full[s], 1);
                }
                ++epi_cnt[s];
            DUO_WALK_END
        }
    } else if (warp == 10) {
        // ===================== store thread =====================
        if (lane == 0) {
            DuoWalk w;
            uint32_t kpar = 0;                      // bit 4s + kb: parity of a_kb[s][kb] to wait for next
            DUO_WALK_BEGIN(w)
                uint8_t* act = smem + s * ACT_BYTES;
                // k-blocks are stored as the epilogue finishes them: a burst of four 16 KB stores at the end of a phase sat in
                // the TMA queue ahead of the weight loads (r02aj: the launch is 10 % shorter with the stores switched off)
                for (int kb = 0; kb < d.rel_kb; ++kb) {
                    const int b = 4 * s + kb;
                    mbar_wait(&a_kb[b], (kpar >> b) & 1u);
                    kpar ^= 1u << b;
                    if (d.out != NO_STORE) {
                        tma_store_2d(&maps.out[ni][d.out], act + kb * KB_BYTES, kb * KBLK, tile_s * TILE_M);
                        bulk_commit();
                    }
                }
                // (every phase releases at least one k-block and the last release is the epilogue's last write to the tile)
                // one completion per phase, storing or not: the epilogue waits for it before the slot's next phase, so it is
                // never two completions of a_kb ahead of this thread (that would alias their parity: the value net's
                // store-less tail phase did exactly this when the stores of the other slot were slow)
                if (d.out != NO_STORE && d.rel_kb > 0) bulk_wait_read_all();
                mbar_arrive(&st_done[s]);
                if (last_ph) mbar_arrive(&x_free[s]);      // the buffer may take the slot's next x tile
            DUO_WALK_END
            asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
        }
    } else {
        // ===================== epilogue warps =====================
        EpiCtx e;
        e.s_bias = s_bias;
        e.s_rowx = s_rowx;
        e.a_ready = nullptr;
        e.lane = lane;
        e.quarter = warp & 3;
        e.half = (warp - 2) >> 2;
        e.row_in_tile = e.quarter * 32 + lane;
        float dv_slot0 = 0.f, dv_slot1 = 0.f;
        float m0 = 0.f, m1 = 0.f, m2 = 0.f, m3 = 0.f, mrows = 0.f;
        float vm0 = 0.f, vm1 = 0.f, vrows = 0.f;
        auto db_add = [&](int c, float v) { atomicAdd(&s_db[c * 32 + e.lane], v); };
        uint32_t cnt[2] = {0u, 0u};                // phases of slot s seen so far (parity of acc_full[s])
        uint32_t pend = 0, scnt = 0;               // bit s: stores of slot s outstanding / parity of st_done[s]
        // ReLU mask words of this thread's row half, [slot][hidden layer][k-block][thread]: a per-CTA scratch in global memory
        // (24 KB, lives in L2); a backward phase fetches its four words BEFORE it waits for its accumulator
        uint32_t* mask_g = p.mask_scratch + (size_t)blockIdx.x * (2 * DUO_MAXL * 4 * kEpiThreads) + (threadIdx.x - 64);
        DuoWalk w;
        DUO_WALK_BEGIN(w)
            uint8_t* act = smem + s * ACT_BYTES;
            e.act = act;
            e.s_mask = nullptr;
            const float* s_bias_n = s_bias + ni * (int)BIAS_FLOATS;
            const int64_t row = (int64_t)tile_s * TILE_M + e.row_in_tile;
            const bool row_ok = row < p.M;
            float dv_keep = s ? dv_slot1 : dv_slot0;
            uint32_t mpre0 = 0u, mpre1 = 0u, mpre2 = 0u, mpre3 = 0u;
            if (d.kind == PH_DGRAD || d.kind == PH_VALUE_BWD) {
                const uint32_t* mp = mask_g + (s * DUO_MAXL + d.layer) * 4 * kEpiThreads;
                mpre0 = __ldcg(mp);
                mpre1 = __ldcg(mp + kEpiThreads);
                mpre2 = __ldcg(mp + 2 * kEpiThreads);
                mpre3 = __ldcg(mp + 3 * kEpiThreads);
            }
            mbar_wait(&acc_full[s], cnt[s] & 1u);
            ++cnt[s];
            tc_fence_after();
            if ((pend >> s) & 1u) {      // the slot's previous phase: its stores have read the tile, its releases were seen
                mbar_wait(&st_done[s], (scnt >> s) & 1u);
                scnt ^= 1u << s;
                pend &= ~(1u << s);
            }
            const uint32_t trow = tmem_base + ((uint32_t)(e.quarter * 32) << 16) + (uint32_t)s * 256u;
            uint8_t* dst = act;
            const int li = d.layer;
    // k-blocks are handed to the store thread in pairs: one proxy fence (it waits for the warp's shared-memory writes, a few
    // hundred cycles with two warps per scheduler) per 128 columns instead of per 64
#define RLPPO_RELEASE_KB(j)                                                  \
    do {                                                                      \
        if (((j) & 1) || (j) + 1 >= (int)d.rel_kb) {                          \
            fence_proxy_async();                                              \
            __syncwarp();                                                     \
            if (lane == 0) {                                                  \
                if ((j) & 1) mbar_arrive(&a_kb[4 * s + (j) - 1]);             \
                mbar_arrive(&a_kb[4 * s + (j)]);                              \
            }                                                                 \
        }                                                                     \
    } while (0)
#define RLPPO_MASK_ST(l, kb, v) __stcg(mask_g + ((s * DUO_MAXL + (l)) * 4 + (kb)) * kEpiThreads, (v))
#define RLPPO_MASK_LD(l, kb) ((kb) == 0 ? mpre0 : (kb) == 1 ? mpre1 : (kb) == 2 ? mpre2 : mpre3)
#include "fused_epilogue.inc"
#undef RLPPO_MASK_ST
#undef RLPPO_MASK_LD
#undef RLPPO_RELEASE_KB
            if (s) dv_slot1 = dv_keep;
            else dv_slot0 = dv_keep;
            pend |= 1u << s;
            // the whole phase is done: the tile in act[s] is complete for the slot's next GEMM and for the store thread
            // (every k-block write above was followed by its own proxy fence + release)
            tc_fence_before();
            __syncwarp();
            if (lane == 0) {
                if (leader) mbar_arrive(&a_done[s]);
                else mbar_arrive_cta(&a_done[s], 0);
            }
        DUO_WALK_END
        if (e.half == 0) {
            for (int ni = 0; ni < p.n_nets; ++ni) {
                const NetP& np = p.net[ni];
                if (np.metrics == nullptr) continue;
                if (np.policy) {
                    const float r0 = warp_sum(m0), r1 = warp_sum(m1), r2 = warp_sum(m2), r3 = warp_sum(m3),
                                rr = warp_sum(mrows);
                    if (e.lane == 0 && rr > 0.f) {
                        atomicAdd(np.metrics + 0, r0);
                        atomicAdd(np.metrics + 1, r1);
                        atomicAdd(np.metrics + 2, r2);
                        atomicAdd(np.metrics + 3, r3);
                        atomicAdd(np.metrics + 4, rr);
                    }
                } else {
                    const float r0 = warp_sum(vm0), r1 = warp_sum(vm1), rr = warp_sum(vrows);
                    if (e.lane == 0 && rr > 0.f) {
                        atomicAdd(np.metrics + 5, r0);
                        atomicAdd(np.metrics + 6, rr);
                        if (np.gbias[MAXL] != nullptr) atomicAdd(np.gbias[MAXL], r1);
                    }
                }
            }
        }
    }
#undef DUO_WALK_BEGIN
#undef DUO_WALK_END
#undef DUO_SEL
#undef DUO_SET
    tc_fence_before();
    __syncthreads();
    cluster_sync_all();
    if (warp == 1) {
        tc_fence_after();
        tmem_dealloc_pair(tmem_base, 512);
    }
    for (int ni = 0; ni < p.n_nets; ++ni) {
        const NetP& np = p.net[ni];
        if (np.policy || np.gw_head == nullptr) continue;
        for (int c = threadIdx.x; c < np.H[np.L - 1]; c += kThreads) atomicAdd(np.gw_head + c, s_db[c]);
    }
}

// ---------------------------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------------------------
int check_net(const rlppo_fused_net* net) {
    RLPPO_CHECK_ARG(net != nullptr, "null net descriptor");
    RLPPO_CHECK_ARG(net->n_hidden >= 1 && net->n_hidden <= MAXL, "fused path: 1..%d hidden layers", MAXL);
    RLPPO_CHECK_ARG(net->in_dim >= 1 && net->in_dim <= 256 && net->in_ld % 8 == 0 && net->in_ld >= net->in_dim,
                    "fused path: input width <= 256, row stride a multiple of 8");
    for (int l = 0; l < net->n_hidden; ++l)
        RLPPO_CHECK_ARG(net->hidden[l] >= 64 && net->hidden[l] <= 256 && net->hidden[l] % 64 == 0,
                        "fused path: hidden widths must be 64, 128, 192 or 256 (got %d)", net->hidden[l]);
    return RLPPO_OK;
}

// Fills net slot `ni` of a launch: phase list, tensor maps of its weights and outputs.  `n` already holds the head's
// arguments (entry points below).
template <bool TRAIN>
int build_net(bool POLICY, const rlppo_fused_net* net, int64_t M, int ni, Maps& maps, NetP& p, bool pair) {
    int rc = check_net(net);
    if (rc) return rc;
    const int L = net->n_hidden;
    p.policy = POLICY ? 1 : 0;
    p.L = L;
    for (int l = 0; l < MAXL; ++l) p.H[l] = l < L ? net->hidden[l] : 0;
    for (int l = 0; l < L; ++l) {
        p.bias[l] = net->bias[l];
        p.gbias[l] = TRAIN ? net->gbias[l] : nullptr;
        RLPPO_CHECK_ARG(net->bias[l] != nullptr, "missing bias");
    }
    p.bias[MAXL] = net->bias[L];
    p.gbias[MAXL] = TRAIN ? net->gbias[L] : nullptr;

    int nw = 0, nph = 0;
    for (int i = 0; i < MAXPH; ++i) p.ph[i] = PhaseDesc{};
    // K-major operands are boxes of N rows (a CTA pair: each CTA stages its N/2 rows); MN-major ones 64 x 64 chunks
    auto add_w = [&](const uint16_t* w, int64_t ld, int rows, int cols, int box_rows, bool mn = false) -> int {
        RLPPO_CHECK_ARG(w != nullptr && ld % 8 == 0, "missing weight operand");
        if (pair && !mn) box_rows /= 2;
        int r = make_tmap_bf16_2d(&maps.w[ni][nw], w, (uint64_t)rows, (uint64_t)cols, (uint64_t)ld, (uint32_t)box_rows);
        if (r) return r;
        ++nw;
        return RLPPO_OK;
    };
    int nout = 0;
    auto add_out = [&](uint16_t* o, int64_t ld, int cols) -> int {
        RLPPO_CHECK_ARG(o != nullptr && ld % 8 == 0 && ld >= cols, "missing activation / gradient output buffer");
        int r = make_tmap_bf16_2d(&maps.out[ni][nout], o, (uint64_t)M, (uint64_t)cols, (uint64_t)ld, TILE_M);
        if (r) return r;
        return nout++;
    };
    const int out_pad8 = POLICY ? (p.n_actions + 7) / 8 * 8 : 0;
    // the head epilogue reads the logits in 32-column chunks: the GEMM writes whole chunks (weight rows past out_pad8 are
    // out of bounds for the TMA box = zeros), so no pass ever sees a TMEM column this launch has not written
    const int head_N = POLICY ? (p.n_actions + 31) / 32 * 32 : 0;
    p.out_kb = POLICY ? (out_pad8 + KBLK - 1) / KBLK : 0;
    auto kb_of = [](int cols) { return (cols + KBLK - 1) / KBLK; };
    auto add_phase = [&](int kind, int layer, int n_kb, int N, int wmap, int out, int smem_out, int wait_kb, int rel_kb,
                         int b_mn = 0) {
        PhaseDesc& d = p.ph[nph++];
        d.kind = (uint8_t)kind;
        d.layer = (uint8_t)layer;
        d.n_kb = (uint8_t)n_kb;
        d.wmap = (uint8_t)wmap;
        d.N = (uint16_t)N;
        d.out = (uint8_t)(TRAIN && out >= 0 ? out : NO_STORE);
        d.smem = (uint8_t)smem_out;
        d.wait_kb = (uint8_t)wait_kb;
        d.rel_kb = (uint8_t)rel_kb;
        d.b_mn = (uint8_t)b_mn;
    };

    // ---- forward phases ----
    for (int l = 0; l < L; ++l) {
        const int K = l == 0 ? net->in_dim : net->hidden[l - 1];
        const int wmap = nw;
        rc = add_w(net->wq[l], net->wq_ld[l], net->hidden[l], K, net->hidden[l]);
        if (rc) return rc;
        const bool value_tail = !POLICY && l == L - 1;
        // H_l goes to HBM as a weight-gradient operand; the value net's last hidden activation is not one (its head's
        // weight gradient is formed in-kernel) and is not a GEMM operand either (the head is a register dot product)
        int out = -1;
        if (TRAIN && !value_tail) {
            out = add_out(net->h[l], net->h_ld[l], net->hidden[l]);
            if (out < 0) return out;
        }
        add_phase(value_tail ? PH_FWD_VALUE : PH_FWD, l, kb_of(K), net->hidden[l], wmap, out, value_tail ? 0 : 1, 0,
                  kb_of(net->hidden[l]));
    }
    if (POLICY) {
        const int wmap = nw;
        rc = add_w(net->wq[L], net->wq_ld[L], out_pad8, net->hidden[L - 1], head_N);
        if (rc) return rc;
        int out = -1;
        if (TRAIN) {
            out = add_out(net->dz, net->dz_ld, out_pad8);
            if (out < 0) return out;
        }
        add_phase(PH_HEAD, L, kb_of(net->hidden[L - 1]), head_N, wmap, out, TRAIN ? 1 : 0, 0, TRAIN ? p.out_kb : 0);
    }
    // k-blocks the last epilogue releases.  inference: the policy head releases nothing, the value tail H_L's k-blocks
    p.tail_rel_kb = POLICY ? 0 : kb_of(net->hidden[L - 1]);
    if (TRAIN) {
        // ---- backward data phases: dL/dH_l is written into the activation tile (the next dgrad GEMM's A operand) and
        // TMA-stored from there to HBM (weight-gradient operand) ----
        int out = add_out(net->dh[L - 1], net->dh_ld[L - 1], net->hidden[L - 1]);
        if (out < 0) return out;
        if (POLICY) {
            const int wmap = nw;
            // dL/dH_L = dz W_head: W_head [out_pad8, hidden] itself as the MN-major operand (k = its rows)
            rc = add_w(net->wq[L], net->wq_ld[L], out_pad8, net->hidden[L - 1], 64, true);
            if (rc) return rc;
            add_phase(PH_DGRAD, L - 1, p.out_kb, net->hidden[L - 1], wmap, out, 1, 0, kb_of(net->hidden[L - 1]), 1);
        } else {
            // GEMM-less phase: dL/dH_L from the accumulator of the last forward GEMM (still in TMEM)
            add_phase(PH_VALUE_BWD, L - 1, 0, net->hidden[L - 1], 0, out, 1, kb_of(net->hidden[L - 1]),
                      kb_of(net->hidden[L - 1]));
        }
        for (int l = L - 1; l >= 1; --l) {
            // produce dH (hidden index l-1) from dH (hidden index l): dH_l W_l with W_l [hidden_l, hidden_{l-1}] read as the
            // MN-major operand (the forward pass reads the same array K-major)
            const int wmap = nw;
            rc = add_w(net->wq[l], net->wq_ld[l], net->hidden[l], net->hidden[l - 1], 64, true);
            if (rc) return rc;
            out = add_out(net->dh[l - 1], net->dh_ld[l - 1], net->hidden[l - 1]);
            if (out < 0) return out;
            add_phase(PH_DGRAD, l - 1, kb_of(net->hidden[l]), net->hidden[l - 1], wmap, out, 1, 0, kb_of(net->hidden[l - 1]), 1);
        }
        p.tail_rel_kb = kb_of(net->hidden[0]);
    }
    p.n_ph = nph;
    return RLPPO_OK;
}

template <bool TRAIN>
int launch_nets_t(const rlppo_fused_net* const* nets, const bool* is_policy, int n_nets, const uint16_t* x, int64_t M,
                  Params& p, cudaStream_t s) {
    Maps maps;
    p.M = M;
    p.num_tiles = (int)((M + TILE_M - 1) / TILE_M);
    p.n_units = p.num_tiles;
    p.n_nets = n_nets;
    p.in_kb = (nets[0]->in_dim + KBLK - 1) / KBLK;
    for (int ni = 0; ni < n_nets; ++ni) {
        RLPPO_CHECK_ARG(nets[ni]->in_dim == nets[0]->in_dim && nets[ni]->in_ld == nets[0]->in_ld,
                        "nets of one launch read the same x");
        int rc = build_net<TRAIN>(is_policy[ni], nets[ni], M, ni, maps, p.net[ni], false);
        if (rc) return rc;
    }
    const rlppo_fused_net* net = nets[0];
    int rc = make_tmap_bf16_2d(&maps.x, x, (uint64_t)M, (uint64_t)net->in_dim, (uint64_t)net->in_ld, TILE_M);
    if (rc) return rc;

    // shared memory: activation tile + x staging (in_kb k-blocks) + as deep an operand ring as fits + misc
    const uint32_t fixed = ACT_BYTES + (uint32_t)p.in_kb * KB_BYTES + MISC_BYTES + 1024;
    p.nwst = (int)((SMEM_LIMIT - fixed) / WST_BYTES);
    if (p.nwst > MAX_NWST) p.nwst = MAX_NWST;
    RLPPO_CHECK_ARG(p.nwst >= 2, "fused path: shared memory budget");
    const uint32_t smem_bytes = fixed + (uint32_t)p.nwst * WST_BYTES;
    static bool configured = false;
    auto kfn = fused_mlp_kernel<TRAIN>;
    if (!configured) {
        RLPPO_CUDA(cudaFuncSetAttribute(kfn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SMEM_LIMIT));
        configured = true;
    }
    const int items = p.n_units * n_nets;
    const int grid = items < num_sms() ? items : num_sms();
    // scheduler words: a pool of self-resetting {next tile, departures} pairs, handed out round-robin so that launches that
    // may overlap (consecutive launches under PDL; launches a caller enqueues on different streams) never share a pair
    {
        constexpr int kSlots = 64;
        static unsigned int* d_sched[16] = {};
        static unsigned int next_slot[16] = {};
        int dev = 0;
        RLPPO_CUDA(cudaGetDevice(&dev));
        RLPPO_CHECK_ARG(dev >= 0 && dev < 16, "device index out of range");
        if (d_sched[dev] == nullptr) {
            RLPPO_CUDA(cudaMalloc(&d_sched[dev], kSlots * 2 * sizeof(unsigned int)));
            RLPPO_CUDA(cudaMemset(d_sched[dev], 0, kSlots * 2 * sizeof(unsigned int)));
        }
        p.sched = d_sched[dev] + 2 * (next_slot[dev]++ % kSlots);
    }
    RLPPO_CUDA(launch_pdl(kfn, dim3(grid), dim3(kThreads), smem_bytes, s, maps, p));
    return RLPPO_OK;
}

// The training launch runs as CTA pairs with two tiles in flight per CTA (fused_duo_kernel) whenever the nets allow it
// (<= 3 hidden layers of width 128 or 256); other shapes run the single-tile kernel.
bool duo_ok(const rlppo_fused_net* const* nets, int n_nets) {
    for (int ni = 0; ni < n_nets; ++ni) {
        if (nets[ni]->n_hidden > DUO_MAXL) return false;
        for (int l = 0; l < nets[ni]->n_hidden; ++l)
            if (nets[ni]->hidden[l] != 128 && nets[ni]->hidden[l] != 256) return false;
    }
    return true;
}

int launch_duo(const rlppo_fused_net* const* nets, const bool* is_policy, int n_nets, const uint16_t* x, int64_t M, Params& p,
               cudaStream_t s) {
    Maps maps;
    p.M = M;
    p.num_tiles = (int)((M + TILE_M - 1) / TILE_M);
    p.n_units = (p.num_tiles + 1) / 2;
    p.n_nets = n_nets;
    p.in_kb = (nets[0]->in_dim + KBLK - 1) / KBLK;
    for (int ni = 0; ni < n_nets; ++ni) {
        RLPPO_CHECK_ARG(nets[ni]->in_dim == nets[0]->in_dim && nets[ni]->in_ld == nets[0]->in_ld,
                        "nets of one launch read the same x");
        int rc = build_net<true>(is_policy[ni], nets[ni], M, ni, maps, p.net[ni], true);
        if (rc) return rc;
    }
    int rc = make_tmap_bf16_2d(&maps.x, x, (uint64_t)M, (uint64_t)nets[0]->in_dim, (uint64_t)nets[0]->in_ld, TILE_M);
    if (rc) return rc;
    static bool configured = false;
    if (!configured) {
        RLPPO_CUDA(cudaFuncSetAttribute(fused_duo_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SMEM_LIMIT));
        configured = true;
    }
    const int items = p.n_units * n_nets;                 // one item = one tile per CTA of a pair; two items in flight per pair
    const int pairs = num_sms() / 2;
    const int want = (items + 1) / 2;
    const int grid = 2 * (want < pairs ? want : pairs);
    // (items are dealt out statically inside the kernel: cluster c takes items c, c + grid / 2, ...)
    for (int ni = 0; ni < n_nets; ++ni)
        for (int i = 0; i < p.net[ni].n_ph; ++i)
            RLPPO_CHECK_ARG(p.net[ni].ph[i].rel_kb > 0, "duo kernel: every phase must release at least one k-block");
    p.sched = nullptr;
    {
        // four scratch areas handed out round-robin: launches a caller enqueues on different streams may overlap
        static uint32_t* d_mask[16] = {};
        static unsigned int next_area[16] = {};
        int dev = 0;
        RLPPO_CUDA(cudaGetDevice(&dev));
        const size_t area = (size_t)num_sms() * 2 * DUO_MAXL * 4 * kEpiThreads;
        if (d_mask[dev] == nullptr) RLPPO_CUDA(cudaMalloc(&d_mask[dev], 4 * area * sizeof(uint32_t)));
        p.mask_scratch = d_mask[dev] + (next_area[dev]++ % 4) * area;
    }
    RLPPO_CUDA(launch_pdl_cluster(fused_duo_kernel, dim3(grid), dim3(kThreads), (size_t)DUO_SMEM, s, 2, maps, p));
    return RLPPO_OK;
}

template <bool TRAIN>
int launch_nets(const rlppo_fused_net* const* nets, const bool* is_policy, int n_nets, const uint16_t* x, int64_t M, Params& p,
                cudaStream_t s) {
    RLPPO_CHECK_ARG(n_nets >= 1 && n_nets <= MAXNET && nets[0] != nullptr, "1..%d nets per launch", MAXNET);
    RLPPO_CHECK_ARG(M >= 1 && M < (1ll << 30) - TILE_M, "bad row count");
    for (int ni = 0; ni < n_nets; ++ni) {
        int rc = check_net(nets[ni]);
        if (rc) return rc;
    }
    if (TRAIN && duo_ok(nets, n_nets)) return launch_duo(nets, is_policy, n_nets, x, M, p, s);
    return launch_nets_t<TRAIN>(nets, is_policy, n_nets, x, M, p, s);
}

void fill_policy_train(NetP& n, int n_actions, const float* actions, const float* old_logp, const float* adv,
                       float inv_batch, float clip, float ent_coef, float* logp_out, float* metrics) {
    n.n_actions = n_actions;
    n.actions = actions; n.old_logp = old_logp; n.adv = adv;
    n.inv_batch = inv_batch; n.clip = clip; n.ent_coef = ent_coef;
    n.logp_out = logp_out; n.metrics = metrics;
}
void fill_value_train(NetP& n, const float* w_head, const float* targets, float inv_batch, float* gw_head,
                      float* values_out, float* metrics) {
    n.w_head = w_head; n.targets = targets; n.inv_batch = inv_batch; n.gw_head = gw_head;
    n.values_out = values_out; n.metrics = metrics;
}

__global__ void u64_add_kernel(unsigned long long* ctr, unsigned long long inc) { *ctr += inc; }

}  // namespace

extern "C" {

int rlppo_policy_train_fused(const rlppo_fused_net* net, const uint16_t* x, int64_t M, int n_actions,
                             const float* actions, const float* old_logp, const float* adv, float inv_batch, float clip,
                             float ent_coef, float* logp_out, float* metrics, void* stream) {
    RLPPO_REQUIRE_DEVICE();
    RLPPO_CHECK_ARG(x && actions && old_logp && adv, "null pointer");
    RLPPO_CHECK_ARG(n_actions >= 1 && n_actions <= 128, "fused path: n_actions must be in [1,128]");
    Params p{};
    fill_policy_train(p.net[0], n_actions, actions, old_logp, adv, inv_batch, clip, ent_coef, logp_out, metrics);
    const bool pol[1] = {true};
    return launch_nets<true>(&net, pol, 1, x, M, p, static_cast<cudaStream_t>(stream));
}

int rlppo_value_train_fused(const rlppo_fused_net* net, const uint16_t* x, int64_t M, const float* w_head,
                            const float* targets, float inv_batch, float* gw_head, float* values_out, float* metrics,
                            void* stream) {
    RLPPO_REQUIRE_DEVICE();
    RLPPO_CHECK_ARG(x && w_head && targets && gw_head, "null pointer");
    Params p{};
    fill_value_train(p.net[0], w_head, targets, inv_batch, gw_head, values_out, metrics);
    const bool pol[1] = {false};
    return launch_nets<true>(&net, pol, 1, x, M, p, static_cast<cudaStream_t>(stream));
}

int rlppo_policy_value_train_fused(const rlppo_fused_net* policy_net, const rlppo_fused_net* value_net, const uint16_t* x,
                                   int64_t M, int n_actions, const float* actions, const float* old_logp, const float* adv,
                                   float inv_batch, float clip, float ent_coef, float* logp_out, const float* w_head,
                                   const float* targets, float* gw_head, float* values_out, float* metrics, void* stream) {
    RLPPO_REQUIRE_DEVICE();
    RLPPO_CHECK_ARG(policy_net && value_net && x && actions && old_logp && adv && w_head && targets && gw_head, "null pointer");
    RLPPO_CHECK_ARG(n_actions >= 1 && n_actions <= 128, "fused path: n_actions must be in [1,128]");
    Params p{};
    fill_policy_train(p.net[0], n_actions, actions, old_logp, adv, inv_batch, clip, ent_coef, logp_out, metrics);
    fill_value_train(p.net[1], w_head, targets, inv_batch, gw_head, values_out, metrics);
    const rlppo_fused_net* nets[2] = {policy_net, value_net};
    const bool pol[2] = {true, false};
    return launch_nets<true>(nets, pol, 2, x, M, p, static_cast<cudaStream_t>(stream));
}

int rlppo_u64_add(uint64_t* d_counter, uint64_t inc, void* stream) {
    RLPPO_REQUIRE_DEVICE();
    RLPPO_CHECK_ARG(d_counter != nullptr, "null pointer");
    u64_add_kernel<<<1, 1, 0, static_cast<cudaStream_t>(stream)>>>(reinterpret_cast<unsigned long long*>(d_counter), inc);
    RLPPO_LAUNCH_CHECK();
    return RLPPO_OK;
}

int rlppo_policy_infer_fused(const rlppo_fused_net* net, const uint16_t* x, int64_t M, int n_actions,
                             const float* u_inject, uint64_t seed, uint64_t offset, const uint64_t* d_offset,
                             int deterministic, float* actions_out, int64_t* actions_i64_out, float* logp_out,
                             void* stream) {
    RLPPO_REQUIRE_DEVICE();
    RLPPO_CHECK_ARG(x != nullptr, "null pointer");
    RLPPO_CHECK_ARG(n_actions >= 1 && n_actions <= 128, "fused path: n_actions must be in [1,128]");
    Params p{};
    NetP& n = p.net[0];
    n.n_actions = n_actions;
    n.u_inject = u_inject; n.seed = seed; n.offset = offset; n.deterministic = deterministic;
    n.d_offset = reinterpret_cast<const unsigned long long*>(d_offset);
    n.actions_out = actions_out; n.actions_i64_out = actions_i64_out; n.logp_out = logp_out;
    const bool pol[1] = {true};
    return launch_nets<false>(&net, pol, 1, x, M, p, static_cast<cudaStream_t>(stream));
}

int rlppo_value_infer_fused(const rlppo_fused_net* net, const uint16_t* x, int64_t M, const float* w_head,
                            float* values_out, void* stream) {
    RLPPO_REQUIRE_DEVICE();
    RLPPO_CHECK_ARG(x && w_head && values_out, "null pointer");
    Params p{};
    p.net[0].w_head = w_head; p.net[0].values_out = values_out;
    const bool pol[1] = {false};
    return launch_nets<false>(&net, pol, 1, x, M, p, static_cast<cudaStream_t>(stream));
}
}
