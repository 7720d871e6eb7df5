// Shared device/host helpers for libtgan_b200 (sm_100a only).
#pragma once
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/tgan_b200.h"

typedef __nv_bfloat16 bf16;

// ---- error plumbing (thread-local message, int return codes) -------------------------------------------
void tgan_set_error(const char* fmt, ...);

#define TGAN_CHECK_ARG(cond, ...)          \
    do {                                   \
        if (!(cond)) {                     \
            tgan_set_error(__VA_ARGS__);   \
            return 1;                      \
        }                                  \
    } while (0)

#define TGAN_CUDA_OK(expr)                                                                    \
    do {                                                                                      \
        cudaError_t _e = (expr);                                                              \
        if (_e != cudaSuccess) {                                                              \
            tgan_set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, \
                           __LINE__);                                                         \
            return 2;                                                                         \
        }                                                                                     \
    } while (0)

#define TGAN_LAUNCH_OK() TGAN_CUDA_OK(cudaGetLastError())

// every kernel launch of the library is counted (bench.py reports it as gpu_launches)
extern unsigned long long g_tgan_launches;
#define TGAN_COUNT_LAUNCH() (++g_tgan_launches)

// ---- element access ---------------------------------------------------------------------------------------
__device__ __forceinline__ float to_f(float x) { return x; }
__device__ __forceinline__ float to_f(bf16 x) { return __bfloat162float(x); }
template <typename T> __device__ __forceinline__ T from_f(float x);
template <> __device__ __forceinline__ float from_f<float>(float x) { return x; }
template <> __device__ __forceinline__ bf16 from_f<bf16>(float x) { return __float2bfloat16_rn(x); }

// 8 consecutive elements (16-byte aligned for bf16, 32-byte for float) -> 8 floats
__device__ __forceinline__ void load8(const float* p, float* o) {
    float4 a = *reinterpret_cast<const float4*>(p), b = *reinterpret_cast<const float4*>(p + 4);
    o[0] = a.x; o[1] = a.y; o[2] = a.z; o[3] = a.w; o[4] = b.x; o[5] = b.y; o[6] = b.z; o[7] = b.w;
}
__device__ __forceinline__ void load8(const bf16* p, float* o) {
    uint4 r = *reinterpret_cast<const uint4*>(p);
    const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&r);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        float2 f = __bfloat1622float2(h[i]);
        o[2 * i] = f.x; o[2 * i + 1] = f.y;
    }
}
__device__ __forceinline__ void store8(float* p, const float* v) {
    *reinterpret_cast<float4*>(p) = make_float4(v[0], v[1], v[2], v[3]);
    *reinterpret_cast<float4*>(p + 4) = make_float4(v[4], v[5], v[6], v[7]);
}
__device__ __forceinline__ void store8(bf16* p, const float* v) {
    uint4 r;
    __nv_bfloat162* h = reinterpret_cast<__nv_bfloat162*>(&r);
#pragma unroll
    for (int i = 0; i < 4; ++i) h[i] = __floats2bfloat162_rn(v[2 * i], v[2 * i + 1]);
    *reinterpret_cast<uint4*>(p) = r;
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}

// ---- Philox4x32-10 (stateless; keyed by seed, counter = (site, element index / 4)) -----------------------
struct Philox4 {
    uint32_t x, y, z, w;
};
__host__ __device__ __forceinline__ uint32_t mulhi32(uint32_t a, uint32_t b) {
#ifdef __CUDA_ARCH__
    return __umulhi(a, b);
#else
    return (uint32_t)(((uint64_t)a * b) >> 32);
#endif
}
__host__ __device__ __forceinline__ Philox4 philox4x32_10(uint64_t seed, uint64_t site, uint64_t idx) {
    uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32);
    uint32_t c0 = (uint32_t)idx, c1 = (uint32_t)(idx >> 32), c2 = (uint32_t)site, c3 = (uint32_t)(site >> 32);
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        uint32_t hi0 = mulhi32(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
        uint32_t hi1 = mulhi32(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
        uint32_t n0 = hi1 ^ c1 ^ k0, n1 = lo1, n2 = hi0 ^ c3 ^ k1, n3 = lo0;
        c0 = n0; c1 = n1; c2 = n2; c3 = n3;
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
    Philox4 o = {c0, c1, c2, c3};
    return o;
}
// ---- dropout masks: stateless counter hash (lowbias32 finaliser over (seed, site, element index)) ----------
// Bit-parity with torch's dropout stream is impossible by construction, so the mask generator is chosen for
// cost: ~10 integer ops per element, any element can be regenerated independently in the backward pass.
__host__ __device__ __forceinline__ uint32_t mix32(uint32_t x) {
    x ^= x >> 16; x *= 0x7feb352du; x ^= x >> 15; x *= 0x846ca68bu; x ^= x >> 16;
    return x;
}
__host__ __device__ __forceinline__ uint32_t dropout_key(uint64_t seed, uint64_t site) {
    return mix32((uint32_t)seed ^ mix32((uint32_t)(seed >> 32) ^ mix32((uint32_t)site ^ mix32((uint32_t)(site >> 32) + 0x9E3779B9u))));
}
// one hash decides a PAIR of consecutive elements (16 random bits each): halves the integer work per element.
__host__ __device__ __forceinline__ uint32_t dropout_hash_pair(uint32_t key, uint64_t pair) {
    return mix32(((uint32_t)pair * 0x9E3779B1u) ^ ((uint32_t)(pair >> 32) * 0x85EBCA77u) ^ key);
}
__host__ __device__ __forceinline__ bool dropout_keep_k(uint32_t key, uint64_t e, uint32_t thresh16) {
    const uint32_t h = dropout_hash_pair(key, e >> 1);
    return ((e & 1) ? (h >> 16) : (h & 0xffffu)) >= thresh16;  // thresh16 = p * 2^16
}
// ---- device-side step counter --------------------------------------------------------------------------------
// A replayed CUDA graph repeats its kernel arguments, so (seed, site) alone would repeat the dropout masks every
// step.  tgan_set_step_counter() registers one device uint32 that the trainer bumps once per optimizer step
// (on the stream, e.g. as the first node of the captured step); every mask key folds its current value in.  The
// forward and the backward of one step read the same value, so they regenerate identical masks.  NULL = off.
// (one copy of the pointer per translation unit: the library is built without relocatable device code)
static __device__ const uint32_t* d_tgan_step_ctr = nullptr;
__device__ __forceinline__ uint32_t step_fold(uint32_t key) {
    const uint32_t* c = d_tgan_step_ctr;
    return c ? mix32(key ^ (__ldg(c) * 0x9E3779B1u)) : key;
}
__device__ __forceinline__ uint64_t step_fold_site(uint64_t site) {
    const uint32_t* c = d_tgan_step_ctr;
    return c ? site ^ ((uint64_t)__ldg(c) << 40) : site;
}
static inline int tgan_set_step_ctr_local(const void* dev_ptr) {
    return (int)cudaMemcpyToSymbol(d_tgan_step_ctr, &dev_ptr, sizeof(dev_ptr));
}
int tgan_set_step_ctr_gemm_simt(const void*);
int tgan_set_step_ctr_gemm_tc(const void*);
int tgan_set_step_ctr_relattn_simt(const void*);
int tgan_set_step_ctr_relattn_decode(const void*);
int tgan_set_step_ctr_bert(const void*);
int tgan_set_step_ctr_sampling(const void*);
int tgan_set_step_ctr_relattn_fwd_tc(const void*);
int tgan_set_step_ctr_relattn_bwd_tc(const void*);

__device__ __forceinline__ bool dropout_keep(uint64_t seed, uint64_t site, uint64_t e, uint32_t thresh16) {
    return dropout_keep_k(step_fold(dropout_key(seed, site)), e, thresh16);
}
// keep bits for the 8 consecutive elements e0 .. e0+7
__host__ __device__ __forceinline__ uint32_t dropout_keep8_k(uint32_t key, uint64_t e0, uint32_t thresh16) {
    uint32_t m = 0;
    if ((e0 & 1) == 0) {
#pragma unroll
        for (int t = 0; t < 4; ++t) {
            const uint32_t h = dropout_hash_pair(key, (e0 >> 1) + t);
            m |= (uint32_t)((h & 0xffffu) >= thresh16) << (2 * t);
            m |= (uint32_t)((h >> 16) >= thresh16) << (2 * t + 1);
        }
    } else {
#pragma unroll
        for (int t = 0; t < 8; ++t) m |= (uint32_t)dropout_keep_k(key, e0 + t, thresh16) << t;
    }
    return m;
}
__device__ __forceinline__ uint32_t dropout_keep8(uint64_t seed, uint64_t site, uint64_t e0, uint32_t thresh16) {
    return dropout_keep8_k(step_fold(dropout_key(seed, site)), e0, thresh16);
}
// attention-probability dropout: one hash yields the keep decisions of a pair of adjacent keys (16 bits each);
// the per-row key is hashed once per query row.  Shared by the SIMT and the tcgen05 attention kernels so that
// both generate identical masks.
__host__ __device__ __forceinline__ uint32_t attn_drop_rowkey(uint32_t key, uint32_t bn_row) {
    return mix32(key ^ (bn_row * 0x9E3779B1u));
}
// three-instruction finaliser (IMAD.WIDE, LOP3, IMAD): fold the 64-bit product of the Weyl-stepped row key, multiply
// again.  Measured on 4096 rows x 1152 keys at p = 0.1: lag / row correlations of the keep bits <= 1e-3 (the
// xor-shift / multiply / xor-shift finaliser it replaces: 6e-3), at 3 instead of 5 integer instructions per key pair.
__host__ __device__ __forceinline__ uint32_t attn_mixlite(uint32_t x) {
    const uint64_t p = (uint64_t)x * 0x9E3779B1u;
    return ((uint32_t)(p >> 32) ^ (uint32_t)p) * 0x7feb352du;
}
__host__ __device__ __forceinline__ uint32_t attn_drop_pair(uint32_t rowkey, uint32_t j_pair) {
    return attn_mixlite(rowkey + j_pair * 0x85EBCA77u);
}
__host__ __device__ __forceinline__ bool attn_drop_keep(uint32_t rowkey, int j, uint32_t thresh16) {
    uint32_t h = attn_drop_pair(rowkey, (uint32_t)j >> 1);
    return ((j & 1) ? (h >> 16) : (h & 0xffffu)) >= thresh16;
}
__host__ __device__ __forceinline__ uint32_t dropout_thresh16(float p) {
    double t = (double)p * 65536.0 + 0.5;
    if (t < 0) t = 0;
    if (t > 65535.0) t = 65535.0;
    return (uint32_t)t;
}
__device__ __forceinline__ float fast_exp2(float x) {
    float y;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
// every dropout site uses 16-bit thresholds (p quantised to 2^-16)
__host__ __device__ __forceinline__ uint32_t dropout_thresh(float p) { return dropout_thresh16(p); }

static inline int ceil_div(int64_t a, int64_t b) { return (int)((a + b - 1) / b); }

// Per-sequence key floor of the attention forward: floor_b = max(reset[b] ? M : 0, key_start[b] - key_base), clamped to
// [0, K].  Query row i of sequence b masks the keys j < min(floor_b, i + M) (tgan_b200.h, tgan_relattn_fwd_ragged);
// with key_start == NULL this is the reset rule, min(M, i + M) = M.  Computed once per sequence and CTA / warp.
__device__ __forceinline__ int key_floor(const uint8_t* reset, const int32_t* key_start, int64_t key_base, int b, int M,
                                         int K) {
    int f = (reset && reset[b]) ? M : 0;
    if (key_start) {
        const int64_t s = (int64_t)key_start[b] - key_base;
        f = max(f, (int)(s < 0 ? 0 : (s > K ? K : s)));
    }
    return f;
}

// ---- internal entry points shared between translation units ----------------------------------------------
int tgan_gemm_simt(int dtype_ab, int dtype_c, int transA, int transB, int M, int N, int K, const void* A,
                   int64_t lda, const void* B, int64_t ldb, void* C, int64_t ldc, const float* bias, const void* aux,
                   int64_t ldaux, int flags, float alpha, float drop_p, uint64_t seed, uint64_t site,
                   cudaStream_t st);
// returns -1 when the shape / layout is not eligible for the tcgen05 kernel (caller falls back or errors)
int tgan_gemm_tc(int dtype_c, int transA, int transB, int M, int N, int K, const void* A, int64_t lda,
                 const void* B, int64_t ldb, void* C, int64_t ldc, const float* bias, const void* aux,
                 int64_t ldaux, int flags, float alpha, float drop_p, uint64_t seed, uint64_t site, int force,
                 cudaStream_t st);
// key_start / key_base: the per-sequence key floor (key_floor above); key_start = NULL switches it off
int tgan_relattn_fwd_simt(int dtype, const void* q, int64_t ldq, const void* k, const void* v, int64_t ldkv,
                          const void* r, int64_t ldr, const float* u, const float* vb, const uint8_t* reset,
                          const int32_t* key_start, int64_t key_base, void* out, int64_t ldo, float* lse, int B, int N,
                          int Q, int M, int msl, int same_length, float scale, float drop_p, uint64_t seed, uint64_t site,
                          cudaStream_t st);
int tgan_relattn_bwd_simt(int dtype, const void* q, int64_t ldq, const void* k, const void* v, int64_t ldkv,
                          const void* r, int64_t ldr, const float* u, const float* vb, const uint8_t* reset,
                          const void* out, const void* dout, int64_t ldo, const float* lse, float* delta, void* dq,
                          void* dk, void* dv, int64_t lddkv, float* dr, int64_t lddr, float* du, float* dvb, int B,
                          int N, int Q, int M, int msl, int same_length, float scale, float drop_p, uint64_t seed,
                          uint64_t site, cudaStream_t st);
// single-token (Q = 1) kernels (relattn_decode.cu); scratch = fp32 [B * N * (M + 1)]
int tgan_relattn_fwd_decode1(int dtype, const void* q, int64_t ldq, const void* k, const void* v, int64_t ldkv,
                             const void* r, int64_t ldr, const float* u, const float* vb, const uint8_t* reset,
                             const int32_t* key_start, int64_t key_base, void* out, int64_t ldo, float* lse, int B, int N,
                             int M, int msl, int same_length, float scale, float drop_p, uint64_t seed, uint64_t site,
                             cudaStream_t st);
int tgan_relattn_bwd_decode1(int dtype, const void* q, int64_t ldq, const void* k, const void* v, int64_t ldkv,
                             const void* r, int64_t ldr, const float* u, const float* vb, const uint8_t* reset,
                             const void* out, const void* dout, int64_t ldo, const float* lse, float* scratch, void* dq,
                             void* dk, void* dv, int64_t lddkv, float* dr, int64_t lddr, float* du, float* dvb, int B,
                             int N, int M, int msl, int same_length, float scale, float drop_p, uint64_t seed,
                             uint64_t site, cudaStream_t st, int phase);
// BERT attention tiles on mma.sync (bert_attn_mma.cu): bf16, T <= 64, d_head a multiple of 16 <= 64
int tgan_bert_attn_fwd_mma(const void* qkv, int64_t ldq, void* ctx, int64_t ldc, float* lse, int B, int heads, int T, int dh,
                           float drop_p, uint64_t seed, uint64_t site, cudaStream_t st);
int tgan_bert_attn_bwd_mma(const void* qkv, int64_t ldq, const void* dctx, int64_t ldc, const float* lse, void* dqkv,
                           int64_t lddq, int B, int heads, int T, int dh, float drop_p, uint64_t seed, uint64_t site,
                           cudaStream_t st);
int tgan_bert_attn_jvp_mma(const void* qkv, int64_t ldq, const void* qkvd, int64_t ldqd, const float* lse, void* ctxd,
                           int64_t ldc, int B, int heads, int T, int dh, float drop_p, uint64_t seed, uint64_t site,
                           cudaStream_t st);
// tcgen05 attention (bf16 only); return -1 when the shape is not eligible
int tgan_relattn_fwd_tc(const void* q, int64_t ldq, const void* k, const void* v, int64_t ldkv, const void* r,
                        int64_t ldr, const float* u, const float* vb, const uint8_t* reset, const int32_t* key_start,
                        int64_t key_base, void* out, int64_t ldo, float* lse, int B, int N, int Q, int M, int msl,
                        int same_length, float scale, float drop_p, uint64_t seed, uint64_t site, cudaStream_t st);
int tgan_relattn_bwd_tc(const void* q, int64_t ldq, const void* k, const void* v, int64_t ldkv, const void* r,
                        int64_t ldr, const float* u, const float* vb, const uint8_t* reset, const void* out,
                        const void* dout, int64_t ldo, const float* lse, float* delta, void* dq, void* dk, void* dv,
                        int64_t lddkv, float* dr, int64_t lddr, float* du, float* dvb, int B, int N, int Q, int M,
                        int msl, int same_length, float scale, float drop_p, uint64_t seed, uint64_t site,
                        cudaStream_t st);

// epilogue shared by both GEMM kernels: acc -> (alpha) -> +bias -> relu -> relu-mask -> dropout -> +aux
struct EpiParams {
    const float* bias;
    const void* aux;
    int64_t ldaux;
    int flags;
    float alpha;
    float drop_scale;      // 1/(1-p)
    uint32_t drop_thresh;  // p * 2^16
    uint32_t drop_key;     // dropout_key(seed, site)
    int aux_is_f32;        // aux element type when the flag says so (TGAN_EPI_AUX_F32)
};
