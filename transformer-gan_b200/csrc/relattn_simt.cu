// Relative-position attention core, SIMT (FFMA) implementation.
//
// This is the fp32-mode path (1e-4 parity with the reference's fp32 arithmetic), the path for single-token
// decode shapes (Q = 1: GAN sampling loop, generation) and the fallback for shapes the tcgen05 kernel does not
// take.  The relative shift (mem_transformer.py:133-147) and the causal / same_length / reset mask
// (mem_transformer.py:495-547) are index arithmetic:  p(i, j) = j + Q - 1 - i,  no [B,Q,K] tensor exists.
//
// Forward: one warp per (b, n, i) query row, lanes stride over the keys with a private online softmax and a
// private output accumulator, merged across the warp at the end.
// Backward: three atomic-free passes that each recompute the scores:
//   rows  : warp per (b, n, i)  -> dq, delta, (du, dvb: one atomic per column per block)
//   keys  : warp per (b, n, j)  -> dk, dv
//   rel   : warp per (n, p)     -> dr  (the inverse rel-shift: a gather along the anti-diagonal i - j = const)
#include "common.cuh"

namespace {
constexpr int HS = TGAN_HS;  // 64
constexpr int WARPS = 4;

struct AttnArgs {
    int B, N, Q, M, K, msl, same_length;
    float scale, drop_scale;
    uint32_t thresh;  // 16-bit threshold (0 = dropout off)
    uint32_t key;
    const int32_t* key_start;  // forward only: per-sequence key floor (common.cuh: key_floor), NULL = off
    int64_t key_base;
};

template <typename T>
__device__ __forceinline__ float dot_row(const float* __restrict__ a, const T* __restrict__ row) {
    float s = 0.f;
#pragma unroll
    for (int c = 0; c < HS / 8; ++c) {
        float x[8];
        load8(row + 8 * c, x);
#pragma unroll
        for (int t = 0; t < 8; ++t) s = fmaf(a[8 * c + t], x[t], s);
    }
    return s;
}
// s = a . x + b . y
template <typename T>
__device__ __forceinline__ float dot_row2(const float* __restrict__ a, const T* __restrict__ x,
                                          const float* __restrict__ b, const T* __restrict__ y) {
    float s = 0.f;
#pragma unroll
    for (int c = 0; c < HS / 8; ++c) {
        float xv[8], yv[8];
        load8(x + 8 * c, xv);
        load8(y + 8 * c, yv);
#pragma unroll
        for (int t = 0; t < 8; ++t) s = fmaf(a[8 * c + t], xv[t], fmaf(b[8 * c + t], yv[t], s));
    }
    return s;
}

__device__ __forceinline__ bool attn_masked(int i, int j, int b_reset, const AttnArgs& a) {
    if (j > i + a.M) return true;
    if (a.same_length && j <= i - a.msl) return true;
    if (b_reset && j < a.M) return true;
    return false;
}

__device__ __forceinline__ bool drop_keep_ij(const AttnArgs& a, int bn, int i, int j) {
    if (!a.thresh) return true;
    return attn_drop_keep(attn_drop_rowkey(step_fold(a.key), (uint32_t)(bn * a.Q + i)), j, a.thresh);
}

// ------------------------------------------------------------------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(WARPS * 32)
relattn_fwd_simt(const T* __restrict__ q, int64_t ldq, const T* __restrict__ k, const T* __restrict__ v,
                 int64_t ldkv, const T* __restrict__ r, int64_t ldr, const float* __restrict__ u,
                 const float* __restrict__ vb, const uint8_t* __restrict__ reset, T* __restrict__ out, int64_t ldo,
                 float* __restrict__ lse, AttnArgs a) {
    __shared__ float s_qu[WARPS][HS], s_qv[WARPS][HS];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int i = blockIdx.x * WARPS + warp;
    const int bn = blockIdx.y, b = bn / a.N, n = bn % a.N;
    if (i >= a.Q) return;  // no block-wide barrier below
    const int64_t row = (int64_t)i * a.B + b;
    for (int d = lane; d < HS; d += 32) {
        float qd = to_f(q[row * ldq + n * HS + d]);
        s_qu[warp][d] = qd + u[n * HS + d];
        s_qv[warp][d] = qd + vb[n * HS + d];
    }
    __syncwarp();
    int jlo = 0, jhi = min(a.K - 1, i + a.M);
    if (a.same_length) jlo = max(0, i - a.msl + 1);
    jlo = max(jlo, min(key_floor(reset, a.key_start, a.key_base, b, a.M, a.K), i + a.M));
    float m = -INFINITY, l = 0.f, acc[HS];
#pragma unroll
    for (int d = 0; d < HS; ++d) acc[d] = 0.f;
    for (int j = jlo + lane; j <= jhi; j += 32) {
        const int p = j + a.Q - 1 - i;
        const T* kr = k + ((int64_t)j * a.B + b) * ldkv + n * HS;
        const T* rr = r + (int64_t)p * ldr + n * HS;
        float s = dot_row2(s_qu[warp], kr, s_qv[warp], rr) * a.scale;
        float mn = fmaxf(m, s);
        float corr = (m == -INFINITY) ? 0.f : expf(m - mn);
        float pe = expf(s - mn);
        l = l * corr + pe;
        float pw = drop_keep_ij(a, bn, i, j) ? pe * a.drop_scale : 0.f;
        const T* vr = v + ((int64_t)j * a.B + b) * ldkv + n * HS;
#pragma unroll
        for (int c = 0; c < HS / 8; ++c) {
            float x[8];
            load8(vr + 8 * c, x);
#pragma unroll
            for (int t = 0; t < 8; ++t) acc[8 * c + t] = fmaf(pw, x[t], acc[8 * c + t] * corr);
        }
        m = mn;
    }
    const float m_all = warp_max(m);
    const float f = (m == -INFINITY) ? 0.f : expf(m - m_all);
    const float l_all = warp_sum(l * f);
    const float inv = l_all > 0.f ? 1.f / l_all : 0.f;
    float o0 = 0.f, o1 = 0.f;
#pragma unroll
    for (int d = 0; d < HS; ++d) {
        float t = warp_sum(acc[d] * f);
        if (d == lane) o0 = t;
        if (d == lane + 32) o1 = t;
    }
    out[row * ldo + n * HS + lane] = from_f<T>(o0 * inv);
    out[row * ldo + n * HS + lane + 32] = from_f<T>(o1 * inv);
    if (lane == 0) lse[(int64_t)bn * a.Q + i] = l_all > 0.f ? m_all + logf(l_all) : -INFINITY;
}

// ------------------------------------------------------------------------------------------------------------
// Forward for decode-sized calls (Q <= DECODE_Q): one CTA per (query row, sequence, head), its DECODE_WARPS warps split
// the keys in 32-key chunks ("flash decoding").  Score phase: lane = key (each lane streams its own 128-byte k / r
// rows); value phase: lane = two head dims (the chunk's probabilities are broadcast with shuffles and every v row is
// one coalesced 128-byte warp load), so a lane carries 2 accumulators instead of 64 and nothing is reduced across
// lanes at the end.  The warps' partial (max, sum, out) triples meet in shared memory.
// The generic kernel above runs ONE warp per (row, sequence, head): at Q = 1 that is 13 % occupancy and a 64-way
// warp reduction per row -- the decode step then sits ~7x above the time the K/V cache stream needs.
constexpr int DECODE_Q = 8, DECODE_WARPS = 8;
__device__ __forceinline__ float2 load2(const float* p) { return *reinterpret_cast<const float2*>(p); }
__device__ __forceinline__ float2 load2(const bf16* p) {
    return __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(p));
}
template <typename T>
__global__ void __launch_bounds__(DECODE_WARPS * 32)
relattn_fwd_decode(const T* __restrict__ q, int64_t ldq, const T* __restrict__ k, const T* __restrict__ v,
                   int64_t ldkv, const T* __restrict__ r, int64_t ldr, const float* __restrict__ u,
                   const float* __restrict__ vb, const uint8_t* __restrict__ reset, T* __restrict__ out, int64_t ldo,
                   float* __restrict__ lse, AttnArgs a) {
    __shared__ float s_qu[HS], s_qv[HS];
    __shared__ float s_m[DECODE_WARPS], s_l[DECODE_WARPS], s_o[DECODE_WARPS][HS];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int i = blockIdx.x;
    const int bn = blockIdx.y, b = bn / a.N, n = bn % a.N;
    const int64_t row = (int64_t)i * a.B + b;
    for (int d = threadIdx.x; d < HS; d += blockDim.x) {
        const float qd = to_f(q[row * ldq + n * HS + d]);
        s_qu[d] = qd + u[n * HS + d];
        s_qv[d] = qd + vb[n * HS + d];
    }
    __syncthreads();
    int jlo = 0, jhi = min(a.K - 1, i + a.M);
    if (a.same_length) jlo = max(0, i - a.msl + 1);
    jlo = max(jlo, min(key_floor(reset, a.key_start, a.key_base, b, a.M, a.K), i + a.M));
    float m = -INFINITY, l = 0.f, acc0 = 0.f, acc1 = 0.f;  // m: warp-uniform running max; l: this lane's share of the sum
    for (int j0 = jlo + 32 * warp; j0 <= jhi; j0 += 32 * DECODE_WARPS) {
        const int j = j0 + lane;
        float s = -INFINITY;
        if (j <= jhi) {
            const T* kr = k + ((int64_t)j * a.B + b) * ldkv + n * HS;
            const T* rr = r + (int64_t)(j + a.Q - 1 - i) * ldr + n * HS;
            s = dot_row2(s_qu, kr, s_qv, rr) * a.scale;
        }
        const float mn = fmaxf(m, warp_max(s));  // finite: the chunk holds at least key j0
        const float corr = (m == -INFINITY) ? 0.f : expf(m - mn);
        const float pe = (j <= jhi) ? expf(s - mn) : 0.f;
        l = l * corr + pe;
        const float pw = (j <= jhi && drop_keep_ij(a, bn, i, j)) ? pe * a.drop_scale : 0.f;
        acc0 *= corr; acc1 *= corr;
        m = mn;
        const int nk = min(32, jhi - j0 + 1);
        const T* vbase = v + ((int64_t)j0 * a.B + b) * ldkv + n * HS + 2 * lane;
#pragma unroll 8
        for (int jj = 0; jj < nk; ++jj) {
            const float pj = __shfl_sync(0xffffffffu, pw, jj);
            const T* vr = vbase + (int64_t)jj * a.B * ldkv;
            const float2 vv = load2(vr);
            acc0 = fmaf(pj, vv.x, acc0);
            acc1 = fmaf(pj, vv.y, acc1);
        }
    }
    const float lw = warp_sum(l);
    if (lane == 0) { s_m[warp] = m; s_l[warp] = lw; }
    s_o[warp][2 * lane] = acc0;
    s_o[warp][2 * lane + 1] = acc1;
    __syncthreads();
    if (warp == 0) {
        float m_all = -INFINITY;
#pragma unroll
        for (int w = 0; w < DECODE_WARPS; ++w) m_all = fmaxf(m_all, s_m[w]);
        float l_all = 0.f, o0 = 0.f, o1 = 0.f;
#pragma unroll
        for (int w = 0; w < DECODE_WARPS; ++w) {
            const float f = (s_m[w] == -INFINITY) ? 0.f : expf(s_m[w] - m_all);
            l_all = fmaf(s_l[w], f, l_all);
            o0 = fmaf(s_o[w][2 * lane], f, o0);
            o1 = fmaf(s_o[w][2 * lane + 1], f, o1);
        }
        const float inv = l_all > 0.f ? 1.f / l_all : 0.f;
        out[row * ldo + n * HS + 2 * lane] = from_f<T>(o0 * inv);
        out[row * ldo + n * HS + 2 * lane + 1] = from_f<T>(o1 * inv);
        if (lane == 0) lse[(int64_t)bn * a.Q + i] = l_all > 0.f ? m_all + logf(l_all) : -INFINITY;
    }
}

// ------------------------------------------------------------------------------------------------------------
// backward pass 1: per query row -> dq, delta, du, dvb
template <typename T>
__global__ void __launch_bounds__(WARPS * 32)
relattn_bwd_rows_simt(const T* __restrict__ q, int64_t ldq, const T* __restrict__ k, const T* __restrict__ v,
                      int64_t ldkv, const T* __restrict__ r, int64_t ldr, const float* __restrict__ u,
                      const float* __restrict__ vb, const uint8_t* __restrict__ reset, const T* __restrict__ out,
                      const T* __restrict__ dout, int64_t ldo, const float* __restrict__ lse,
                      float* __restrict__ delta, T* __restrict__ dq, float* __restrict__ du,
                      float* __restrict__ dvb, AttnArgs a) {
    __shared__ float s_qu[WARPS][HS], s_qv[WARPS][HS], s_do[WARPS][HS];
    __shared__ float s_du[HS], s_dvb[HS];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int i = blockIdx.x * WARPS + warp;
    const int bn = blockIdx.y, b = bn / a.N, n = bn % a.N;
    for (int d = threadIdx.x; d < HS; d += blockDim.x) { s_du[d] = 0.f; s_dvb[d] = 0.f; }
    __syncthreads();
    if (i < a.Q) {
        const int64_t row = (int64_t)i * a.B + b;
        float dl = 0.f;
        for (int d = lane; d < HS; d += 32) {
            float qd = to_f(q[row * ldq + n * HS + d]);
            s_qu[warp][d] = qd + u[n * HS + d];
            s_qv[warp][d] = qd + vb[n * HS + d];
            float g = to_f(dout[row * ldo + n * HS + d]);
            s_do[warp][d] = g;
            dl += g * to_f(out[row * ldo + n * HS + d]);
        }
        dl = warp_sum(dl);
        __syncwarp();
        const float L = lse[(int64_t)bn * a.Q + i];
        if (lane == 0) delta[(int64_t)bn * a.Q + i] = dl;
        int jlo = 0, jhi = min(a.K - 1, i + a.M);
        if (a.same_length) jlo = max(0, i - a.msl + 1);
        if (reset && reset[b]) jlo = max(jlo, a.M);
        float acck[HS], accr[HS];
#pragma unroll
        for (int d = 0; d < HS; ++d) { acck[d] = 0.f; accr[d] = 0.f; }
        for (int j = jlo + lane; j <= jhi; j += 32) {
            const int p = j + a.Q - 1 - i;
            const T* kr = k + ((int64_t)j * a.B + b) * ldkv + n * HS;
            const T* rr = r + (int64_t)p * ldr + n * HS;
            const T* vr = v + ((int64_t)j * a.B + b) * ldkv + n * HS;
            float s = dot_row2(s_qu[warp], kr, s_qv[warp], rr) * a.scale;
            float pr = expf(s - L);
            float dp = dot_row(s_do[warp], vr);
            dp = drop_keep_ij(a, bn, i, j) ? dp * a.drop_scale : 0.f;
            float ds = pr * (dp - dl) * a.scale;
#pragma unroll
            for (int c = 0; c < HS / 8; ++c) {
                float x[8], y[8];
                load8(kr + 8 * c, x);
                load8(rr + 8 * c, y);
#pragma unroll
                for (int t = 0; t < 8; ++t) {
                    acck[8 * c + t] = fmaf(ds, x[t], acck[8 * c + t]);
                    accr[8 * c + t] = fmaf(ds, y[t], accr[8 * c + t]);
                }
            }
        }
        float k0 = 0.f, k1 = 0.f, r0 = 0.f, r1 = 0.f;
#pragma unroll
        for (int d = 0; d < HS; ++d) {
            float tk = warp_sum(acck[d]), tr = warp_sum(accr[d]);
            if (d == lane) { k0 = tk; r0 = tr; }
            if (d == lane + 32) { k1 = tk; r1 = tr; }
        }
        dq[row * ldq + n * HS + lane] = from_f<T>(k0 + r0);
        dq[row * ldq + n * HS + lane + 32] = from_f<T>(k1 + r1);
        atomicAdd(&s_du[lane], k0); atomicAdd(&s_du[lane + 32], k1);
        atomicAdd(&s_dvb[lane], r0); atomicAdd(&s_dvb[lane + 32], r1);
    }
    __syncthreads();
    for (int d = threadIdx.x; d < HS; d += blockDim.x) {
        atomicAdd(&du[n * HS + d], s_du[d]);
        atomicAdd(&dvb[n * HS + d], s_dvb[d]);
    }
}

// backward pass 2 for decode-sized calls (Q <= SMALLQ): one THREAD per key row.  The warp-per-key kernel below spreads
// the query rows over the lanes and pays 128 warp reductions per key whatever Q is -- at Q = 1 (every Gumbel sampling
// step of the GAN phase) that is ~1500 instructions per key for 200 FMAs of work.  Here lane = key: the (q + bias) /
// dout rows sit in shared memory, each thread streams its own k / v / r rows (full 128-byte lines), keeps its
// dS / P~ column in shared memory and writes dk / dv with 16-byte stores.  No cross-lane traffic at all.
constexpr int SMALLQ = 16;
template <typename T>
__global__ void __launch_bounds__(WARPS * 32)
relattn_bwd_keys_smallq(const T* __restrict__ q, int64_t ldq, const T* __restrict__ k, const T* __restrict__ v,
                        int64_t ldkv, const T* __restrict__ r, int64_t ldr, const float* __restrict__ u,
                        const float* __restrict__ vb, const uint8_t* __restrict__ reset,
                        const T* __restrict__ dout, int64_t ldo, const float* __restrict__ lse,
                        const float* __restrict__ delta, T* __restrict__ dk, T* __restrict__ dv, int64_t lddkv,
                        AttnArgs a) {
    __shared__ float s_qu[SMALLQ][HS], s_qv[SMALLQ][HS], s_do[SMALLQ][HS], s_L[SMALLQ], s_dl[SMALLQ];
    __shared__ float s_ds[SMALLQ][WARPS * 32], s_pw[SMALLQ][WARPS * 32];
    const int bn = blockIdx.y, b = bn / a.N, n = bn % a.N;
    for (int idx = threadIdx.x; idx < a.Q * HS; idx += blockDim.x) {
        const int i = idx / HS, d = idx % HS;
        const int64_t row = (int64_t)i * a.B + b;
        const float x = to_f(q[row * ldq + n * HS + d]);
        s_qu[i][d] = x + u[n * HS + d];
        s_qv[i][d] = x + vb[n * HS + d];
        s_do[i][d] = to_f(dout[row * ldo + n * HS + d]);
    }
    for (int i = threadIdx.x; i < a.Q; i += blockDim.x) {
        s_L[i] = lse[(int64_t)bn * a.Q + i];
        s_dl[i] = delta[(int64_t)bn * a.Q + i];
    }
    __syncthreads();
    const int j = blockIdx.x * (WARPS * 32) + threadIdx.x;
    if (j >= a.K) return;
    const int64_t krow = (int64_t)j * a.B + b;
    const T* kr = k + krow * ldkv + n * HS;
    const T* vr = v + krow * ldkv + n * HS;
    int ilo = max(0, j - a.M), ihi = a.Q - 1;
    if (a.same_length) ihi = min(ihi, j + a.msl - 1);
    if (reset && reset[b] && j < a.M) ihi = -1;
    // phase 1: dS and the dropped probability of every (query, this key) pair -> thread-private shared-memory columns
    for (int i = ilo; i <= ihi; ++i) {
        const T* rr = r + (int64_t)(j + a.Q - 1 - i) * ldr + n * HS;
        float s = 0.f, dp = 0.f;
#pragma unroll
        for (int c = 0; c < HS / 8; ++c) {
            float kk[8], yy[8], vv[8];
            load8(kr + 8 * c, kk);
            load8(rr + 8 * c, yy);
            load8(vr + 8 * c, vv);
#pragma unroll
            for (int t = 0; t < 8; ++t) {
                const int d = 8 * c + t;
                s = fmaf(s_qu[i][d], kk[t], fmaf(s_qv[i][d], yy[t], s));
                dp = fmaf(s_do[i][d], vv[t], dp);
            }
        }
        const float pr = expf(s * a.scale - s_L[i]);
        const bool keep = drop_keep_ij(a, bn, i, j);
        dp = keep ? dp * a.drop_scale : 0.f;
        s_pw[i][threadIdx.x] = keep ? pr * a.drop_scale : 0.f;
        s_ds[i][threadIdx.x] = pr * (dp - s_dl[i]) * a.scale;
    }
    // phase 2: dk_j = sum_i dS_ij (q_i + u), dv_j = sum_i P~_ij dout_i, eight columns at a time
    T* dkr = dk + krow * lddkv + n * HS;
    T* dvr = dv + krow * lddkv + n * HS;
#pragma unroll
    for (int c = 0; c < HS / 8; ++c) {
        float ak[8], av[8];
#pragma unroll
        for (int t = 0; t < 8; ++t) { ak[t] = 0.f; av[t] = 0.f; }
        for (int i = ilo; i <= ihi; ++i) {
            const float ds = s_ds[i][threadIdx.x], pw = s_pw[i][threadIdx.x];
#pragma unroll
            for (int t = 0; t < 8; ++t) {
                ak[t] = fmaf(ds, s_qu[i][8 * c + t], ak[t]);
                av[t] = fmaf(pw, s_do[i][8 * c + t], av[t]);
            }
        }
        store8(dkr + 8 * c, ak);
        store8(dvr + 8 * c, av);
    }
}

// backward pass 2: per key row -> dk, dv
template <typename T>
__global__ void __launch_bounds__(WARPS * 32)
relattn_bwd_keys_simt(const T* __restrict__ q, int64_t ldq, const T* __restrict__ k, const T* __restrict__ v,
                      int64_t ldkv, const T* __restrict__ r, int64_t ldr, const float* __restrict__ u,
                      const float* __restrict__ vb, const uint8_t* __restrict__ reset,
                      const T* __restrict__ dout, int64_t ldo, const float* __restrict__ lse,
                      const float* __restrict__ delta, T* __restrict__ dk, T* __restrict__ dv, int64_t lddkv,
                      AttnArgs a) {
    __shared__ float s_k[WARPS][HS], s_v[WARPS][HS], s_u[HS], s_vb[HS];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int j = blockIdx.x * WARPS + warp;
    const int bn = blockIdx.y, b = bn / a.N, n = bn % a.N;
    for (int d = threadIdx.x; d < HS; d += blockDim.x) { s_u[d] = u[n * HS + d]; s_vb[d] = vb[n * HS + d]; }
    __syncthreads();
    if (j >= a.K) return;
    const int64_t krow = (int64_t)j * a.B + b;
    for (int d = lane; d < HS; d += 32) {
        s_k[warp][d] = to_f(k[krow * ldkv + n * HS + d]);
        s_v[warp][d] = to_f(v[krow * ldkv + n * HS + d]);
    }
    __syncwarp();
    int ilo = max(0, j - a.M), ihi = a.Q - 1;
    if (a.same_length) ihi = min(ihi, j + a.msl - 1);
    if (reset && reset[b] && j < a.M) ihi = -1;
    float acck[HS], accv[HS];
#pragma unroll
    for (int d = 0; d < HS; ++d) { acck[d] = 0.f; accv[d] = 0.f; }
    for (int i = ilo + lane; i <= ihi; i += 32) {
        const int64_t row = (int64_t)i * a.B + b;
        const int p = j + a.Q - 1 - i;
        const T* qr = q + row * ldq + n * HS;
        const T* rr = r + (int64_t)p * ldr + n * HS;
        const T* dor = dout + row * ldo + n * HS;
        float s = 0.f, dp = 0.f;
#pragma unroll
        for (int c = 0; c < HS / 8; ++c) {
            float x[8], y[8], g[8];
            load8(qr + 8 * c, x);
            load8(rr + 8 * c, y);
            load8(dor + 8 * c, g);
#pragma unroll
            for (int t = 0; t < 8; ++t) {
                int d = 8 * c + t;
                s = fmaf(x[t] + s_u[d], s_k[warp][d], fmaf(x[t] + s_vb[d], y[t], s));
                dp = fmaf(g[t], s_v[warp][d], dp);
            }
        }
        const float L = lse[(int64_t)bn * a.Q + i], dl = delta[(int64_t)bn * a.Q + i];
        float pr = expf(s * a.scale - L);
        bool keep = drop_keep_ij(a, bn, i, j);
        float pw = keep ? pr * a.drop_scale : 0.f;
        dp = keep ? dp * a.drop_scale : 0.f;
        float ds = pr * (dp - dl) * a.scale;
#pragma unroll
        for (int c = 0; c < HS / 8; ++c) {
            float x[8], g[8];
            load8(qr + 8 * c, x);
            load8(dor + 8 * c, g);
#pragma unroll
            for (int t = 0; t < 8; ++t) {
                int d = 8 * c + t;
                acck[d] = fmaf(ds, x[t] + s_u[d], acck[d]);
                accv[d] = fmaf(pw, g[t], accv[d]);
            }
        }
    }
    float k0 = 0.f, k1 = 0.f, v0 = 0.f, v1 = 0.f;
#pragma unroll
    for (int d = 0; d < HS; ++d) {
        float tk = warp_sum(acck[d]), tv = warp_sum(accv[d]);
        if (d == lane) { k0 = tk; v0 = tv; }
        if (d == lane + 32) { k1 = tk; v1 = tv; }
    }
    dk[krow * lddkv + n * HS + lane] = from_f<T>(k0);
    dk[krow * lddkv + n * HS + lane + 32] = from_f<T>(k1);
    dv[krow * lddkv + n * HS + lane] = from_f<T>(v0);
    dv[krow * lddkv + n * HS + lane + 32] = from_f<T>(v1);
}

// backward pass 3: per relative position -> dr[p] = scale * sum_{b,i} dS[b,i,j=p-Q+1+i] (q_i + vb)
template <typename T>
__global__ void __launch_bounds__(WARPS * 32)
relattn_bwd_rel_simt(const T* __restrict__ q, int64_t ldq, const T* __restrict__ k, const T* __restrict__ v,
                     int64_t ldkv, const T* __restrict__ r, int64_t ldr, const float* __restrict__ u,
                     const float* __restrict__ vb, const uint8_t* __restrict__ reset, const T* __restrict__ dout,
                     int64_t ldo, const float* __restrict__ lse, const float* __restrict__ delta,
                     float* __restrict__ dr, int64_t lddr, AttnArgs a) {
    __shared__ float s_r[WARPS][HS], s_u[HS], s_vb[HS];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int p = blockIdx.x * WARPS + warp;
    const int n = blockIdx.y;
    for (int d = threadIdx.x; d < HS; d += blockDim.x) { s_u[d] = u[n * HS + d]; s_vb[d] = vb[n * HS + d]; }
    __syncthreads();
    if (p >= a.K) return;
    for (int d = lane; d < HS; d += 32) s_r[warp][d] = to_f(r[(int64_t)p * ldr + n * HS + d]);
    __syncwarp();
    float acc[HS];
#pragma unroll
    for (int d = 0; d < HS; ++d) acc[d] = 0.f;
    const int total = a.B * a.Q;
    for (int idx = lane; idx < total; idx += 32) {
        const int b = idx / a.Q, i = idx % a.Q;
        const int j = p - a.Q + 1 + i;
        if (j < 0 || j >= a.K) continue;
        if (attn_masked(i, j, reset ? reset[b] : 0, a)) continue;
        const int bn = b * a.N + n;
        const int64_t row = (int64_t)i * a.B + b, krow = (int64_t)j * a.B + b;
        const T* qr = q + row * ldq + n * HS;
        const T* kr = k + krow * ldkv + n * HS;
        const T* vr = v + krow * ldkv + n * HS;
        const T* dor = dout + row * ldo + n * HS;
        float s = 0.f, dp = 0.f;
#pragma unroll
        for (int c = 0; c < HS / 8; ++c) {
            float x[8], y[8], g[8], w[8];
            load8(qr + 8 * c, x);
            load8(kr + 8 * c, y);
            load8(dor + 8 * c, g);
            load8(vr + 8 * c, w);
#pragma unroll
            for (int t = 0; t < 8; ++t) {
                int d = 8 * c + t;
                s = fmaf(x[t] + s_u[d], y[t], fmaf(x[t] + s_vb[d], s_r[warp][d], s));
                dp = fmaf(g[t], w[t], dp);
            }
        }
        const float L = lse[(int64_t)bn * a.Q + i], dl = delta[(int64_t)bn * a.Q + i];
        float pr = expf(s * a.scale - L);
        dp = drop_keep_ij(a, bn, i, j) ? dp * a.drop_scale : 0.f;
        float ds = pr * (dp - dl) * a.scale;
#pragma unroll
        for (int c = 0; c < HS / 8; ++c) {
            float x[8];
            load8(qr + 8 * c, x);
#pragma unroll
            for (int t = 0; t < 8; ++t) acc[8 * c + t] = fmaf(ds, x[t] + s_vb[8 * c + t], acc[8 * c + t]);
        }
    }
    float r0 = 0.f, r1 = 0.f;
#pragma unroll
    for (int d = 0; d < HS; ++d) {
        float t = warp_sum(acc[d]);
        if (d == lane) r0 = t;
        if (d == lane + 32) r1 = t;
    }
    dr[(int64_t)p * lddr + n * HS + lane] = r0;
    dr[(int64_t)p * lddr + n * HS + lane + 32] = r1;
}

AttnArgs make_args(int B, int N, int Q, int M, int msl, int same_length, float scale, float drop_p, uint64_t seed,
                   uint64_t site) {
    AttnArgs a;
    a.B = B; a.N = N; a.Q = Q; a.M = M; a.K = M + Q; a.msl = msl; a.same_length = same_length; a.scale = scale;
    a.drop_scale = drop_p > 0.f ? 1.f / (1.f - drop_p) : 1.f;
    a.thresh = drop_p > 0.f ? dropout_thresh16(drop_p) : 0u;
    a.key = dropout_key(seed, site);
    a.key_start = nullptr;
    a.key_base = 0;
    return a;
}
}  // namespace

int tgan_relattn_fwd_simt(int dtype, const void* q, int64_t ldq, const void* k, const void* v, int64_t ldkv,
                          const void* r, int64_t ldr, const float* u, const float* vb, const uint8_t* reset,
                          const int32_t* key_start, int64_t key_base, void* out, int64_t ldo, float* lse, int B, int N,
                          int Q, int M, int msl, int same_length, float scale, float drop_p, uint64_t seed, uint64_t site,
                          cudaStream_t st) {
    AttnArgs a = make_args(B, N, Q, M, msl, same_length, scale, drop_p, seed, site);
    a.key_start = key_start;
    a.key_base = key_base;
    const bool vec_ok = ((((uintptr_t)k | (uintptr_t)v | (uintptr_t)r) & 31) == 0) && ldkv % 8 == 0 && ldr % 8 == 0;
    if (Q == 1 && vec_ok && ((((uintptr_t)q | (uintptr_t)out | (uintptr_t)u | (uintptr_t)vb) & 31) == 0) && ldq % 8 == 0 &&
        ldo % 8 == 0)
        return tgan_relattn_fwd_decode1(dtype, q, ldq, k, v, ldkv, r, ldr, u, vb, reset, key_start, key_base, out, ldo,
                                        lse, B, N, M, msl, same_length, scale, drop_p, seed, site, st);
    if (Q <= DECODE_Q && vec_ok) {
        dim3 gd(Q, B * N);
        if (dtype == TGAN_F32)
            relattn_fwd_decode<float><<<gd, DECODE_WARPS * 32, 0, st>>>((const float*)q, ldq, (const float*)k, (const float*)v,
                                                                         ldkv, (const float*)r, ldr, u, vb, reset,
                                                                         (float*)out, ldo, lse, a);
        else
            relattn_fwd_decode<bf16><<<gd, DECODE_WARPS * 32, 0, st>>>((const bf16*)q, ldq, (const bf16*)k, (const bf16*)v,
                                                                        ldkv, (const bf16*)r, ldr, u, vb, reset,
                                                                        (bf16*)out, ldo, lse, a);
        TGAN_COUNT_LAUNCH();
        TGAN_LAUNCH_OK();
        return 0;
    }
    dim3 grid(ceil_div(Q, WARPS), B * N);
    if (dtype == TGAN_F32)
        relattn_fwd_simt<float><<<grid, WARPS * 32, 0, st>>>((const float*)q, ldq, (const float*)k, (const float*)v,
                                                              ldkv, (const float*)r, ldr, u, vb, reset, (float*)out,
                                                              ldo, lse, a);
    else
        relattn_fwd_simt<bf16><<<grid, WARPS * 32, 0, st>>>((const bf16*)q, ldq, (const bf16*)k, (const bf16*)v, ldkv,
                                                             (const bf16*)r, ldr, u, vb, reset, (bf16*)out, ldo, lse,
                                                             a);
    TGAN_COUNT_LAUNCH();
    TGAN_LAUNCH_OK();
    return 0;
}

template <typename T>
static int bwd_launch(const void* q, int64_t ldq, const void* k, const void* v, int64_t ldkv, const void* r,
                      int64_t ldr, const float* u, const float* vb, const uint8_t* reset, const void* out,
                      const void* dout, int64_t ldo, const float* lse, float* delta, void* dq, void* dk, void* dv,
                      int64_t lddkv, float* dr, int64_t lddr, float* du, float* dvb, const AttnArgs& a,
                      cudaStream_t st) {
    dim3 g1(ceil_div(a.Q, WARPS), a.B * a.N);
    relattn_bwd_rows_simt<T><<<g1, WARPS * 32, 0, st>>>((const T*)q, ldq, (const T*)k, (const T*)v, ldkv, (const T*)r,
                                                         ldr, u, vb, reset, (const T*)out, (const T*)dout, ldo, lse,
                                                         delta, (T*)dq, du, dvb, a);
    TGAN_COUNT_LAUNCH();
    TGAN_LAUNCH_OK();
    const bool vec_ok = ((((uintptr_t)k | (uintptr_t)v | (uintptr_t)r | (uintptr_t)dk | (uintptr_t)dv) & 31) == 0) &&
                        ldkv % 8 == 0 && ldr % 8 == 0 && lddkv % 8 == 0;
    if (a.Q <= SMALLQ && vec_ok) {
        dim3 g2(ceil_div(a.K, WARPS * 32), a.B * a.N);
        relattn_bwd_keys_smallq<T><<<g2, WARPS * 32, 0, st>>>((const T*)q, ldq, (const T*)k, (const T*)v, ldkv,
                                                               (const T*)r, ldr, u, vb, reset, (const T*)dout, ldo, lse,
                                                               delta, (T*)dk, (T*)dv, lddkv, a);
    } else {
        dim3 g2(ceil_div(a.K, WARPS), a.B * a.N);
        relattn_bwd_keys_simt<T><<<g2, WARPS * 32, 0, st>>>((const T*)q, ldq, (const T*)k, (const T*)v, ldkv, (const T*)r,
                                                             ldr, u, vb, reset, (const T*)dout, ldo, lse, delta, (T*)dk,
                                                             (T*)dv, lddkv, a);
    }
    TGAN_COUNT_LAUNCH();
    TGAN_LAUNCH_OK();
    dim3 g3(ceil_div(a.K, WARPS), a.N);
    relattn_bwd_rel_simt<T><<<g3, WARPS * 32, 0, st>>>((const T*)q, ldq, (const T*)k, (const T*)v, ldkv, (const T*)r,
                                                        ldr, u, vb, reset, (const T*)dout, ldo, lse, delta, dr, lddr,
                                                        a);
    TGAN_COUNT_LAUNCH();
    TGAN_LAUNCH_OK();
    return 0;
}

int tgan_relattn_bwd_simt(int dtype, const void* q, int64_t ldq, const void* k, const void* v, int64_t ldkv,
                          const void* r, int64_t ldr, const float* u, const float* vb, const uint8_t* reset,
                          const void* out, const void* dout, int64_t ldo, const float* lse, float* delta, void* dq,
                          void* dk, void* dv, int64_t lddkv, float* dr, int64_t lddr, float* du, float* dvb, int B,
                          int N, int Q, int M, int msl, int same_length, float scale, float drop_p, uint64_t seed,
                          uint64_t site, cudaStream_t st) {
    const uintptr_t al = (uintptr_t)q | (uintptr_t)k | (uintptr_t)v | (uintptr_t)r | (uintptr_t)out | (uintptr_t)dout |
                         (uintptr_t)dq | (uintptr_t)dk | (uintptr_t)dv | (uintptr_t)u | (uintptr_t)vb;
    if (Q == 1 && (al & 31) == 0 && ldq % 8 == 0 && ldkv % 8 == 0 && ldr % 8 == 0 && ldo % 8 == 0 && lddkv % 8 == 0 &&
        lddr % 4 == 0)
        // `delta` doubles as the dS scratch of the fused single-token backward: B * N * (M + 1) floats (tgan_b200.h)
        return tgan_relattn_bwd_decode1(dtype, q, ldq, k, v, ldkv, r, ldr, u, vb, reset, out, dout, ldo, lse, delta, dq,
                                        dk, dv, lddkv, dr, lddr, du, dvb, B, N, M, msl, same_length, scale, drop_p, seed,
                                        site, st, 0);
    AttnArgs a = make_args(B, N, Q, M, msl, same_length, scale, drop_p, seed, site);
    if (dtype == TGAN_F32)
        return bwd_launch<float>(q, ldq, k, v, ldkv, r, ldr, u, vb, reset, out, dout, ldo, lse, delta, dq, dk, dv,
                                 lddkv, dr, lddr, du, dvb, a, st);
    return bwd_launch<bf16>(q, ldq, k, v, ldkv, r, ldr, u, vb, reset, out, dout, ldo, lse, delta, dq, dk, dv, lddkv,
                            dr, lddr, du, dvb, a, st);
}

int tgan_set_step_ctr_relattn_simt(const void* p) { return tgan_set_step_ctr_local(p); }
