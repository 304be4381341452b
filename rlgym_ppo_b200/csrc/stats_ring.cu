// Welford running statistics, the experience ring (append / gather) and bf16 operand preparation.
// All of these are HBM-bound byte movers: coalesced, vectorised where rows are 16-byte aligned, grids sized
// from the row count.  Reference semantics: running_stats.py:30-69, experience_buffer.py:17-37,82-102.
#include "common.cuh"

namespace {

// ---- Welford ------------------------------------------------------------------------------------------
// One thread per statistic dimension, samples applied strictly in order (running_stats.py:37-46).
template <bool F64>
__global__ void welford_kernel(float* mean, float* m2, int64_t* count, const void* samples, int64_t n, int dim,
                               float* std_out, float* mean_out) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= dim) return;
    const int64_t c0 = *count;
    float mu = mean[j], s2 = m2[j];
    int64_t c = c0;
    if (F64) {
        const double* x = static_cast<const double*>(samples);
        for (int64_t i = 0; i < n; ++i) {
            const int64_t cc = c;
            c += 1;
            const double delta = x[i * dim + j] - (double)mu;
            const double delta_n = delta / (double)c;
            mu = (float)((double)mu + delta_n);
            s2 = (float)((double)s2 + delta * delta_n * (double)cc);
        }
    } else {
        const float* x = static_cast<const float*>(samples);
        for (int64_t i = 0; i < n; ++i) {
            const int64_t cc = c;
            c += 1;
            const float delta = __fsub_rn(x[i * dim + j], mu);
            const float delta_n = __fdiv_rn(delta, (float)c);
            mu = __fadd_rn(mu, delta_n);
            s2 = __fadd_rn(s2, __fmul_rn(__fmul_rn(delta, delta_n), (float)cc));
        }
    }
    mean[j] = mu;
    m2[j] = s2;
    if (std_out) {  // running_stats.py:60-69
        float sd = 1.f;
        if (c >= 2) {
            float var = __fdiv_rn(s2, (float)(c - 1));
            if (var == 0.f) var = 1.f;
            sd = __fsqrt_rn(var);
        }
        std_out[j] = sd;
    }
    if (mean_out) mean_out[j] = (c >= 2) ? mu : 0.f;  // :54-58
    __syncthreads();
    if (j == 0) *count = c;  // single block when dim <= 1024 (checked on the host)
}

// A count next to an f32 array, as NumPy 2 converts a Python int there: to double, then to float.
__device__ __forceinline__ float count_to_f32(int64_t c) { return __double2float_rn(__ll2double_rn(c)); }

// Chan's parallel merge of n_others Welford states into (mean, m2, count), others applied in order: the reference's
// increment_from_serialized_other (running_stats.py:71-98) with its evaluation order, f32 round-to-nearest throughout.
// Other i is the block at others + i * stride: [count i64 | mean f32[dim] | m2 f32[dim] | ...].  One block; threads
// stride over dim.
__global__ void welford_merge_kernel(float* mean, float* m2, int64_t* count, const unsigned char* __restrict__ others,
                                     int64_t stride, int n_others, int dim, float* std_out, float* mean_out) {
    const int64_t c0 = *count;
    int64_t c = c0;
    for (int j = threadIdx.x; j < dim; j += blockDim.x) {
        float mu = mean[j], s2 = m2[j];
        c = c0;
        for (int i = 0; i < n_others; ++i) {
            const unsigned char* blk = others + (int64_t)i * stride;
            const int64_t oc = *reinterpret_cast<const int64_t*>(blk);
            if (oc == 0) continue;
            const float omu = reinterpret_cast<const float*>(blk + 8)[j];
            const float os2 = reinterpret_cast<const float*>(blk + 8)[dim + j];
            const int64_t cn = c + oc;
            const float fc = count_to_f32(c), fo = count_to_f32(oc), fn = count_to_f32(cn);
            const float delta = __fsub_rn(omu, mu);
            const float d2 = __fmul_rn(delta, delta);
            const float mu_n = __fdiv_rn(__fadd_rn(__fmul_rn(fc, mu), __fmul_rn(fo, omu)), fn);
            s2 = __fadd_rn(__fadd_rn(s2, os2), __fdiv_rn(__fmul_rn(__fmul_rn(d2, fc), fo), fn));
            mu = mu_n;
            c = cn;
        }
        mean[j] = mu;
        m2[j] = s2;
        if (std_out) {  // as welford_kernel
            float sd = 1.f;
            if (c >= 2) {
                float var = __fdiv_rn(s2, (float)(c - 1));
                if (var == 0.f) var = 1.f;
                sd = __fsqrt_rn(var);
            }
            std_out[j] = sd;
        }
        if (mean_out) mean_out[j] = (c >= 2) ? mu : 0.f;
    }
    __syncthreads();  // every thread has read *count
    if (threadIdx.x == 0) {
        c = c0;
        for (int i = 0; i < n_others; ++i) c += *reinterpret_cast<const int64_t*>(others + (int64_t)i * stride);
        *count = c;
    }
}

// ---- ring append ----------------------------------------------------------------------------------------
template <bool F64>
__global__ void ring_append_kernel(float* ring, int64_t ring_ld, uint16_t* ring_bf16, int64_t bf16_ld,
                                   int64_t capacity, int64_t phys_first, const void* src, int64_t src_ld,
                                   int64_t n_rows, int width) {
    // one warp per row (rows are 1 or obs_dim wide); scalar rows are handled by the flat variant below
    const int64_t row = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (row >= n_rows) return;
    const int lane = threadIdx.x & 31;
    int64_t phys = phys_first + row;
    if (phys >= capacity) phys -= capacity;
    for (int c = lane; c < (ring_bf16 ? (int)bf16_ld : width); c += 32) {
        float x = 0.f;
        if (c < width)
            x = F64 ? (float)static_cast<const double*>(src)[row * src_ld + c]
                    : static_cast<const float*>(src)[row * src_ld + c];
        if (c < width) ring[phys * ring_ld + c] = x;
        if (ring_bf16) ring_bf16[phys * bf16_ld + c] = rlppo::f32_to_bf16_bits(x);
    }
}

template <bool F64>
__global__ void ring_append_flat_kernel(float* ring, int64_t capacity, int64_t phys_first, const void* src,
                                        int64_t n_rows) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_rows) return;
    int64_t phys = phys_first + i;
    if (phys >= capacity) phys -= capacity;
    ring[phys] = F64 ? (float)static_cast<const double*>(src)[i] : static_cast<const float*>(src)[i];
}

// All fields of one submit in ONE launch: blockIdx.y = field, 64 rows per block.  Wide fields are copied as a flat run
// of elements (64 rows x width, contiguous in the source and -- away from the wrap -- in the ring): every thread has four
// independent loads in flight before its first store.  d_state (optional) = device int64[2] {start, size} of the ring:
// the append position is then (start + size) % capacity, read on the device, so a captured CUDA graph follows the ring.
constexpr int kMaxAppendFields = 12;
struct AppendFields {
    rlppo_append_field f[kMaxAppendFields];
};
__device__ __forceinline__ float append_load(const rlppo_append_field& f, int64_t row, int c) {
    return f.src_is_f64 ? (float)__ldg(static_cast<const double*>(f.src) + row * f.src_ld + c)
                        : __ldg(static_cast<const float*>(f.src) + row * f.src_ld + c);
}
__global__ void __launch_bounds__(256)
ring_append_fields_kernel(AppendFields fs, int64_t capacity, int64_t phys_first, const int64_t* __restrict__ d_state,
                          int64_t n_rows) {
    if (d_state != nullptr) phys_first = (__ldg(d_state) + __ldg(d_state + 1)) % capacity;
    const rlppo_append_field& f = fs.f[blockIdx.y];
    const int64_t row0 = (int64_t)blockIdx.x * 64;
    const int rows = (int)min((int64_t)64, n_rows - row0);
    if (rows <= 0) return;
    int64_t phys0 = phys_first + row0;
    if (phys0 >= capacity) phys0 -= capacity;
    const int wrap = (int)min((int64_t)rows, capacity - phys0);   // rows [wrap, rows) continue at physical row 0
    if (f.width == 1 && f.ring_bf16 == nullptr) {
        if ((int)threadIdx.x < rows) {
            const int r = threadIdx.x;
            const int64_t phys = r < wrap ? phys0 + r : (int64_t)(r - wrap);
            f.ring[phys * f.ring_ld] = append_load(f, row0 + r, 0);
        }
        return;
    }
    const int W = f.width;
    const int total = rows * W;
    const float inv_w = 1.0f / (float)W;
    for (int e0 = threadIdx.x; e0 < total; e0 += 1024) {
        float x[4];
        int r[4], c[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int e = e0 + u * 256;
            if (e < total) {
                r[u] = (int)(((float)e + 0.5f) * inv_w);   // exact: e < 2^18, W <= 4096 (checked on the host)
                c[u] = e - r[u] * W;
                x[u] = append_load(f, row0 + r[u], c[u]);
            }
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int e = e0 + u * 256;
            if (e < total) {
                const int64_t phys = r[u] < wrap ? phys0 + r[u] : (int64_t)(r[u] - wrap);
                f.ring[phys * f.ring_ld + c[u]] = x[u];
                if (f.ring_bf16) f.ring_bf16[phys * f.bf16_ld + c[u]] = rlppo::f32_to_bf16_bits(x[u]);
            }
        }
    }
    if (f.ring_bf16 != nullptr && f.bf16_ld > W) {   // zero padding of the bf16 rows
        const int pad = (int)f.bf16_ld - W;
        for (int e = threadIdx.x; e < rows * pad; e += 256) {
            const int r = e / pad, c = W + (e - r * pad);
            const int64_t phys = r < wrap ? phys0 + r : (int64_t)(r - wrap);
            f.ring_bf16[phys * f.bf16_ld + c] = 0;
        }
    }
}
// {start, size} <- state after appending n_rows (the host mirrors the same arithmetic, experience_buffer.py)
__global__ void ring_advance_kernel(int64_t* state, int64_t n_rows, int64_t capacity) {
    const int64_t start = state[0], size = state[1];
    const int64_t over = size + n_rows > capacity ? size + n_rows - capacity : 0;
    state[0] = (start + over) % capacity;
    state[1] = size + n_rows > capacity ? capacity : size + n_rows;
}

// ---- gather ---------------------------------------------------------------------------------------------
// Eight samples per warp: lane = 4 * sample + part.  Part q fetches scalar field q of its sample and the 16-byte
// vectors q, q+4, q+8, ... of its observation row, so every lane has several independent loads in flight behind the one
// dependent index load (one warp per sample kept 12 of 32 lanes busy with a single 16-byte load each: 0.9 TB/s at
// example sizes, latency-bound).
__global__ void gather_kernel(const float* __restrict__ actions, const float* __restrict__ logp,
                              const float* __restrict__ values, const float* __restrict__ adv,
                              const float* __restrict__ states, int64_t states_ld,
                              const uint16_t* __restrict__ states_bf16, int64_t bf16_ld, int obs_dim,
                              int64_t capacity, int64_t start, const int64_t* __restrict__ d_start,
                              const int64_t* __restrict__ idx, int64_t B,
                              float* __restrict__ out_actions, float* __restrict__ out_logp,
                              float* __restrict__ out_values, float* __restrict__ out_adv,
                              float* __restrict__ out_states, uint16_t* __restrict__ out_states_bf16) {
    const int lane = threadIdx.x & 31;
    const int q = lane & 3;
    const int64_t b = ((int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5)) * 8 + (lane >> 2);
    rlppo::pdl_wait();   // launched with the PDL attribute: the rings / the permutation may come from the previous kernel
    if (b >= B) return;
    if (d_start != nullptr) start = __ldg(d_start);   // device-resident ring origin: lets a captured graph follow the ring
    int64_t phys = start + __ldg(idx + b);
    if (phys >= capacity) phys -= capacity;
    {
        const float* src = q == 0 ? actions : (q == 1 ? logp : (q == 2 ? values : adv));
        float* dst = q == 0 ? out_actions : (q == 1 ? out_logp : (q == 2 ? out_values : out_adv));
        if (dst != nullptr) dst[b] = __ldg(src + phys);
    }
    if (out_states_bf16) {
        // rows are bf16_ld*2 bytes, bf16_ld % 8 == 0 -> 16-byte vectors
        const uint4* s = reinterpret_cast<const uint4*>(states_bf16 + phys * bf16_ld);
        uint4* o = reinterpret_cast<uint4*>(out_states_bf16 + b * bf16_ld);
        const int nvec = (int)(bf16_ld >> 3);
        int c = q;
        for (; c + 8 < nvec; c += 12) {                // three independent loads in flight
            const uint4 v0 = __ldg(s + c), v1 = __ldg(s + c + 4), v2 = __ldg(s + c + 8);
            o[c] = v0;
            o[c + 4] = v1;
            o[c + 8] = v2;
        }
        for (; c < nvec; c += 4) o[c] = __ldg(s + c);
    }
    if (out_states) {
        const float* s = states + phys * states_ld;
        float* o = out_states + b * (int64_t)obs_dim;
        for (int c = q; c < obs_dim; c += 4) o[c] = __ldg(s + c);
    }
}

// ---- f32 rows -> padded bf16 rows -------------------------------------------------------------------------
// One thread per 8 output columns (one 16-byte store); the eight source floats are consecutive, so a warp reads 256
// consecutive floats of the source and writes 512 consecutive bytes.  (Round 1: one thread per ELEMENT with a 64-bit
// divide for the row index -- 27 us for the 50 000 x 89 rollout, 1 TB/s; ncu showed the LSU issue-bound on 2-byte stores.)
template <bool STANDARDIZE>
__global__ void rows_to_bf16_kernel(const float* __restrict__ src, int64_t src_ld, int64_t n_rows, int width,
                                    const float* __restrict__ mean, const float* __restrict__ stdv, float clip,
                                    uint16_t* __restrict__ dst, int64_t dst_ld, float* __restrict__ dst_f32,
                                    int64_t dst_f32_ld) {
    const int groups = (int)(dst_ld >> 3);                 // dst_ld % 8 == 0 (checked on the host)
    const int64_t total = n_rows * groups;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total;
         i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t row = i / groups;
        const int c0 = (int)(i - row * groups) * 8;
        const float* s = src + row * src_ld + c0;
        float x[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            float v = 0.f;
            if (c0 + j < width) {
                v = __ldg(s + j);
                if (STANDARDIZE) {  // batched_agent_manager.py:303-315
                    v = __fdiv_rn(__fsub_rn(v, __ldg(mean + c0 + j)), __ldg(stdv + c0 + j));
                    v = fminf(fmaxf(v, -clip), clip);
                    if (dst_f32 != nullptr) dst_f32[row * dst_f32_ld + c0 + j] = v;
                }
            }
            x[j] = v;
        }
        uint4 o;
        o.x = rlppo::pack_bf16x2(x[0], x[1]);
        o.y = rlppo::pack_bf16x2(x[2], x[3]);
        o.z = rlppo::pack_bf16x2(x[4], x[5]);
        o.w = rlppo::pack_bf16x2(x[6], x[7]);
        *reinterpret_cast<uint4*>(dst + row * dst_ld + c0) = o;
    }
}

__global__ void weight_to_bf16_kernel(const float* __restrict__ w, int out_f, int in_f, uint16_t* __restrict__ wq,
                                      int64_t wq_ld, int out_pad, uint16_t* __restrict__ wt, int64_t wt_ld,
                                      int in_pad) {
    // tile transpose through shared memory so both outputs are written coalesced
    __shared__ float tile[32][33];
    const int o0 = blockIdx.y * 32, i0 = blockIdx.x * 32;
    for (int r = threadIdx.y; r < 32; r += blockDim.y) {
        const int o = o0 + r, i = i0 + threadIdx.x;
        const float x = (o < out_f && i < in_f) ? w[(int64_t)o * in_f + i] : 0.f;
        tile[r][threadIdx.x] = x;
        if (o < out_pad && i < wq_ld) wq[(int64_t)o * wq_ld + i] = rlppo::f32_to_bf16_bits(x);
    }
    if (wt == nullptr) return;
    __syncthreads();
    for (int r = threadIdx.y; r < 32; r += blockDim.y) {
        const int i = i0 + r, o = o0 + threadIdx.x;
        if (i < in_pad && o < wt_ld) wt[(int64_t)i * wt_ld + o] = rlppo::f32_to_bf16_bits(tile[threadIdx.x][r]);
    }
}


// ---- split ("fp32-exact") operands: f32 -> hi / mid / lo bf16 parts side by side (rlppo_split in rlppo.h) ----------
// part 0 = bf16(x), part q = bf16(x - part_0 - ... - part_{q-1}); three parts carry 24 significand bits.
template <bool STANDARDIZE>
__global__ void rows_split_kernel(const float* __restrict__ src, int64_t src_ld, int64_t n_rows, int width,
                                  const float* __restrict__ mean, const float* __restrict__ stdv, float clip,
                                  uint16_t* __restrict__ dst, int64_t dst_ld, int parts, int64_t pstride) {
    const int64_t total = n_rows * pstride;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total;
         i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t row = i / pstride;
        const int c = (int)(i - row * pstride);
        float x = 0.f;
        if (c < width) {
            x = __ldg(src + row * src_ld + c);
            if (STANDARDIZE) {  // batched_agent_manager.py:303-315
                x = __fdiv_rn(__fsub_rn(x, __ldg(mean + c)), __ldg(stdv + c));
                x = fminf(fmaxf(x, -clip), clip);
            }
        }
        for (int q = 0; q < parts; ++q) {
            const uint16_t b = rlppo::f32_to_bf16_bits(x);
            dst[row * dst_ld + q * pstride + c] = b;
            x -= rlppo::bf16_bits_to_f32(b);
        }
    }
}

__global__ void weight_split_kernel(const float* __restrict__ w, int out_f, int in_f, uint16_t* __restrict__ wq,
                                    int64_t wq_ld, int q_parts, int64_t q_pstride, int out_rows,
                                    uint16_t* __restrict__ wt, int64_t wt_ld, int t_parts, int64_t t_pstride, int in_rows) {
    __shared__ float tile[32][33];
    const int o0 = blockIdx.y * 32, i0 = blockIdx.x * 32;
    for (int r = threadIdx.y; r < 32; r += blockDim.y) {
        const int o = o0 + r, i = i0 + threadIdx.x;
        float x = (o < out_f && i < in_f) ? w[(int64_t)o * in_f + i] : 0.f;
        tile[r][threadIdx.x] = x;
        if (wq != nullptr && o < out_rows && i < q_pstride) {
            for (int q = 0; q < q_parts; ++q) {
                const uint16_t b = rlppo::f32_to_bf16_bits(x);
                wq[(int64_t)o * wq_ld + q * q_pstride + i] = b;
                x -= rlppo::bf16_bits_to_f32(b);
            }
        }
    }
    if (wt == nullptr) return;
    __syncthreads();
    for (int r = threadIdx.y; r < 32; r += blockDim.y) {
        const int i = i0 + r, o = o0 + threadIdx.x;
        if (i < in_rows && o < t_pstride) {
            float x = tile[threadIdx.x][r];
            for (int q = 0; q < t_parts; ++q) {
                const uint16_t b = rlppo::f32_to_bf16_bits(x);
                wt[(int64_t)i * wt_ld + q * t_pstride + o] = b;
                x -= rlppo::bf16_bits_to_f32(b);
            }
        }
    }
}

}  // namespace

extern "C" {

int rlppo_welford_update(float* mean, float* m2, int64_t* count, const void* samples, int samples_are_f64,
                         int64_t n, int dim, float* std_out, float* mean_out, void* stream) {
    RLPPO_REQUIRE_DEVICE();
    RLPPO_CHECK_ARG(mean && m2 && count && (samples || n == 0), "null pointer");
    RLPPO_CHECK_ARG(dim >= 1 && dim <= 1024 && n >= 0, "dim must be in [1,1024]");
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    const int threads = ((dim + 31) / 32) * 32;
    if (samples_are_f64)
        welford_kernel<true><<<1, threads, 0, s>>>(mean, m2, count, samples, n, dim, std_out, mean_out);
    else
        welford_kernel<false><<<1, threads, 0, s>>>(mean, m2, count, samples, n, dim, std_out, mean_out);
    RLPPO_LAUNCH_CHECK();
    return RLPPO_OK;
}

int rlppo_welford_merge(float* mean, float* m2, int64_t* count, const void* others, int64_t other_stride_bytes,
                        int n_others, int dim, float* std_out, float* mean_out, void* stream) {
    RLPPO_REQUIRE_DEVICE();
    RLPPO_CHECK_ARG(mean && m2 && count && (others || n_others == 0), "null pointer");
    RLPPO_CHECK_ARG(dim >= 1 && n_others >= 0, "dim must be >= 1 and n_others >= 0");
    RLPPO_CHECK_ARG(n_others == 0 || (other_stride_bytes >= 8 + 8 * (int64_t)dim && other_stride_bytes % 8 == 0 &&
                                      (reinterpret_cast<uintptr_t>(others) & 7) == 0),
                    "other blocks: stride must hold [count | mean | m2] and keep the i64 counts 8-byte aligned");
    const int threads = (int)min((int64_t)1024, ((int64_t)dim + 31) / 32 * 32);
    welford_merge_kernel<<<1, threads, 0, static_cast<cudaStream_t>(stream)>>>(
        mean, m2, count, static_cast<const unsigned char*>(others), other_stride_bytes, n_others, dim, std_out, mean_out);
    RLPPO_LAUNCH_CHECK();
    return RLPPO_OK;
}

int rlppo_ring_append(float* ring, int64_t ring_ld, uint16_t* ring_bf16, int64_t bf16_ld, int64_t capacity,
                      int64_t phys_first, const void* src, int src_is_f64, int64_t src_ld, int64_t n_rows, int width,
                      void* stream) {
    RLPPO_REQUIRE_DEVICE();
    RLPPO_CHECK_ARG(ring && src && capacity > 0 && n_rows >= 0 && n_rows <= capacity && width >= 1, "bad argument");
    RLPPO_CHECK_ARG(phys_first >= 0 && phys_first < capacity, "phys_first out of range");
    RLPPO_CHECK_ARG(!ring_bf16 || (bf16_ld >= width && bf16_ld % 8 == 0), "bf16_ld must be >= width and %% 8 == 0");
    if (n_rows == 0) return RLPPO_OK;
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    if (width == 1 && ring_ld == 1 && src_ld == 1 && !ring_bf16) {
        const int threads = 256;
        const unsigned blocks = (unsigned)((n_rows + threads - 1) / threads);
        if (src_is_f64) ring_append_flat_kernel<true><<<blocks, threads, 0, s>>>(ring, capacity, phys_first, src, n_rows);
        else ring_append_flat_kernel<false><<<blocks, threads, 0, s>>>(ring, capacity, phys_first, src, n_rows);
    } else {
        const int threads = 256, rows_per_block = threads / 32;
        const unsigned blocks = (unsigned)((n_rows + rows_per_block - 1) / rows_per_block);
        if (src_is_f64)
            ring_append_kernel<true><<<blocks, threads, 0, s>>>(ring, ring_ld, ring_bf16, bf16_ld, capacity, phys_first,
                                                                src, src_ld, n_rows, width);
        else
            ring_append_kernel<false><<<blocks, threads, 0, s>>>(ring, ring_ld, ring_bf16, bf16_ld, capacity, phys_first,
                                                                 src, src_ld, n_rows, width);
    }
    RLPPO_LAUNCH_CHECK();
    return RLPPO_OK;
}

static int append_fields_impl(const rlppo_append_field* h_fields, int n_fields, int64_t capacity, int64_t phys_first,
                              int64_t* d_state, int64_t n_rows, cudaStream_t s) {
    RLPPO_CHECK_ARG(h_fields && n_fields >= 1 && n_fields <= kMaxAppendFields, "1..%d fields", kMaxAppendFields);
    RLPPO_CHECK_ARG(capacity > 0 && n_rows >= 0 && n_rows <= capacity && phys_first >= 0 && phys_first < capacity,
                    "bad ring position");
    if (n_rows == 0) return RLPPO_OK;
    AppendFields fs;
    for (int i = 0; i < n_fields; ++i) {
        const rlppo_append_field& f = h_fields[i];
        RLPPO_CHECK_ARG(f.ring && f.src && f.width >= 1 && f.width <= 4096 && f.ring_ld >= 1 && f.src_ld >= 1,
                        "bad field %d", i);
        RLPPO_CHECK_ARG(!f.ring_bf16 || (f.bf16_ld >= f.width && f.bf16_ld % 8 == 0), "field %d: bad bf16_ld", i);
        fs.f[i] = f;
    }
    dim3 grid((unsigned)((n_rows + 63) / 64), (unsigned)n_fields);
    ring_append_fields_kernel<<<grid, 256, 0, s>>>(fs, capacity, phys_first, d_state, n_rows);
    RLPPO_LAUNCH_CHECK();
    if (d_state != nullptr) {
        ring_advance_kernel<<<1, 1, 0, s>>>(d_state, n_rows, capacity);
        RLPPO_LAUNCH_CHECK();
    }
    return RLPPO_OK;
}

int rlppo_ring_append_fields(const rlppo_append_field* h_fields, int n_fields, int64_t capacity, int64_t phys_first,
                             int64_t n_rows, void* stream) {
    RLPPO_REQUIRE_DEVICE();
    return append_fields_impl(h_fields, n_fields, capacity, phys_first, nullptr, n_rows, static_cast<cudaStream_t>(stream));
}

int rlppo_ring_append_fields_dev(const rlppo_append_field* h_fields, int n_fields, int64_t capacity, int64_t* d_state,
                                 int64_t n_rows, void* stream) {
    RLPPO_REQUIRE_DEVICE();
    RLPPO_CHECK_ARG(d_state != nullptr, "null ring state");
    return append_fields_impl(h_fields, n_fields, capacity, 0, d_state, n_rows, static_cast<cudaStream_t>(stream));
}

int rlppo_gather_batch(const float* actions, const float* logp, const float* values, const float* adv,
                       const float* states, int64_t states_ld, const uint16_t* states_bf16, int64_t bf16_ld,
                       int obs_dim, int64_t capacity, int64_t start, const int64_t* d_start, const int64_t* idx,
                       int64_t B, float* out_actions, float* out_logp, float* out_values, float* out_adv,
                       float* out_states, uint16_t* out_states_bf16, void* stream) {
    RLPPO_REQUIRE_DEVICE();
    RLPPO_CHECK_ARG(idx && capacity > 0 && start >= 0 && start < capacity && B >= 0, "bad argument");
    RLPPO_CHECK_ARG(!out_actions || actions, "actions ring missing");
    RLPPO_CHECK_ARG(!out_logp || logp, "log_probs ring missing");
    RLPPO_CHECK_ARG(!out_values || values, "values ring missing");
    RLPPO_CHECK_ARG(!out_adv || adv, "advantages ring missing");
    RLPPO_CHECK_ARG(!out_states || states, "states ring missing");
    RLPPO_CHECK_ARG(!out_states_bf16 || (states_bf16 && bf16_ld % 8 == 0), "bf16 states ring missing / ld %% 8");
    if (B == 0) return RLPPO_OK;
    // 128-thread CTAs of <= 48 registers: one fits on an SM BESIDE a persistent fused-MLP CTA (352 threads x 168 registers leave
    // 6400), so a gather launched on a second stream runs under the previous step's kernels (ppo_learner._learn_body)
    const int threads = 128, per_block = threads / 32 * 8;      // eight samples per warp
    const unsigned blocks = (unsigned)((B + per_block - 1) / per_block);
    RLPPO_CUDA(rlppo::launch_pdl(gather_kernel, dim3(blocks), dim3(threads), 0, static_cast<cudaStream_t>(stream), actions,
                                 logp, values, adv, states, states_ld, states_bf16, bf16_ld, obs_dim, capacity, start,
                                 d_start, idx, B, out_actions, out_logp, out_values, out_adv, out_states, out_states_bf16));
    return RLPPO_OK;
}

int rlppo_rows_to_bf16(const float* src, int64_t src_ld, int64_t n_rows, int width, const float* mean,
                       const float* stdv, float clip, uint16_t* dst, int64_t dst_ld, float* dst_f32, int64_t dst_f32_ld,
                       void* stream) {
    RLPPO_REQUIRE_DEVICE();
    RLPPO_CHECK_ARG(src && dst && dst_ld >= width && n_rows >= 0, "bad argument");
    RLPPO_CHECK_ARG((mean == nullptr) == (stdv == nullptr), "mean and std go together");
    RLPPO_CHECK_ARG(mean || !dst_f32, "dst_f32 holds standardised rows: it needs mean and std");
    RLPPO_CHECK_ARG(dst_ld % 8 == 0 && (reinterpret_cast<uintptr_t>(dst) & 15) == 0,
                    "bf16 rows: dst_ld must be a multiple of 8 and dst 16-byte aligned");
    if (n_rows == 0) return RLPPO_OK;
    const int64_t total = n_rows * (dst_ld / 8);
    const unsigned blocks = (unsigned)min((int64_t)rlppo::num_sms() * 16, (total + 255) / 256);
    RLPPO_CHECK_ARG(!dst_f32 || dst_f32_ld >= width, "dst_f32_ld must be >= width");
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    if (mean == nullptr)
        rows_to_bf16_kernel<false><<<blocks, 256, 0, s>>>(src, src_ld, n_rows, width, nullptr, nullptr, 0.f, dst, dst_ld,
                                                          nullptr, 0);
    else
        rows_to_bf16_kernel<true><<<blocks, 256, 0, s>>>(src, src_ld, n_rows, width, mean, stdv, clip, dst, dst_ld, dst_f32,
                                                         dst_f32_ld);
    RLPPO_LAUNCH_CHECK();
    return RLPPO_OK;
}

int rlppo_weight_to_bf16(const float* w, int out_f, int in_f, uint16_t* wq, int64_t wq_ld, int out_pad, uint16_t* wt,
                         int64_t wt_ld, int in_pad, void* stream) {
    RLPPO_REQUIRE_DEVICE();
    RLPPO_CHECK_ARG(w && wq && out_f >= 1 && in_f >= 1 && wq_ld >= in_f && out_pad >= out_f, "bad argument");
    RLPPO_CHECK_ARG(!wt || (wt_ld >= out_f && in_pad >= in_f), "bad transposed operand shape");
    // cover the padded extents of both outputs
    const int cols = (int)max((int64_t)max(in_pad, in_f), wq_ld);
    const int rows = (int)max((int64_t)out_pad, wt ? wt_ld : (int64_t)0);
    dim3 grid((cols + 31) / 32, (rows + 31) / 32), block(32, 8);
    weight_to_bf16_kernel<<<grid, block, 0, static_cast<cudaStream_t>(stream)>>>(w, out_f, in_f, wq, wq_ld, out_pad, wt,
                                                                                 wt_ld, in_pad);
    RLPPO_LAUNCH_CHECK();
    return RLPPO_OK;
}

int rlppo_rows_split_bf16(const float* src, int64_t src_ld, int64_t n_rows, int width, const float* mean,
                          const float* stdv, float clip, uint16_t* dst, int64_t dst_ld, int parts, int64_t pstride,
                          void* stream) {
    RLPPO_REQUIRE_DEVICE();
    RLPPO_CHECK_ARG(src && dst && n_rows >= 0 && parts >= 1 && parts <= 3 && pstride >= width &&
                        dst_ld >= (int64_t)parts * pstride, "bad argument");
    RLPPO_CHECK_ARG((mean == nullptr) == (stdv == nullptr), "mean and std go together");
    if (n_rows == 0) return RLPPO_OK;
    const int64_t total = n_rows * pstride;
    const unsigned blocks = (unsigned)min((int64_t)rlppo::num_sms() * 16, (total + 255) / 256);
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    if (mean != nullptr)
        rows_split_kernel<true><<<blocks, 256, 0, s>>>(src, src_ld, n_rows, width, mean, stdv, clip, dst, dst_ld, parts, pstride);
    else
        rows_split_kernel<false><<<blocks, 256, 0, s>>>(src, src_ld, n_rows, width, nullptr, nullptr, 0.f, dst, dst_ld, parts,
                                                        pstride);
    RLPPO_LAUNCH_CHECK();
    return RLPPO_OK;
}

int rlppo_weight_split_bf16(const float* w, int out_f, int in_f, uint16_t* wq, int64_t wq_ld, int q_parts,
                            int64_t q_pstride, int out_rows, uint16_t* wt, int64_t wt_ld, int t_parts, int64_t t_pstride,
                            int in_rows, void* stream) {
    RLPPO_REQUIRE_DEVICE();
    RLPPO_CHECK_ARG(w && out_f >= 1 && in_f >= 1 && (wq || wt), "bad argument");
    RLPPO_CHECK_ARG(!wq || (q_parts >= 1 && q_parts <= 3 && q_pstride >= in_f && wq_ld >= (int64_t)q_parts * q_pstride &&
                            out_rows >= out_f), "bad forward operand shape");
    RLPPO_CHECK_ARG(!wt || (t_parts >= 1 && t_parts <= 3 && t_pstride >= out_f && wt_ld >= (int64_t)t_parts * t_pstride &&
                            in_rows >= in_f), "bad transposed operand shape");
    const int cols = (int)max((int64_t)(wt ? in_rows : in_f), wq ? q_pstride : (int64_t)0);
    const int rows = (int)max((int64_t)(wq ? out_rows : out_f), wt ? t_pstride : (int64_t)0);
    dim3 grid((cols + 31) / 32, (rows + 31) / 32), block(32, 8);
    weight_split_kernel<<<grid, block, 0, static_cast<cudaStream_t>(stream)>>>(w, out_f, in_f, wq, wq_ld, q_parts, q_pstride,
                                                                               out_rows, wt, wt_ld, t_parts, t_pstride, in_rows);
    RLPPO_LAUNCH_CHECK();
    return RLPPO_OK;
}
}
