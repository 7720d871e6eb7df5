// Public entry points of the relative-position attention core: dispatch between the tcgen05 kernels
// (relattn_tc.cu, bf16, training shapes) and the SIMT kernels (relattn_simt.cu: fp32 mode, decode shapes).
#include "common.cuh"

// One implementation behind both forward entry points; key_start = NULL is tgan_relattn_fwd.
static int relattn_fwd_impl(int dtype, const void* q, int64_t ldq, const void* k, const void* v, int64_t ldkv,
                            const void* r, int64_t ldr, const float* u, const float* vb, const uint8_t* reset,
                            const int32_t* key_start, int64_t key_base, void* out, int64_t ldo, float* lse, int B, int N,
                            int Q, int M, int msl, int same_length, float scale, float drop_p, uint64_t seed,
                            uint64_t site, int impl, void* stream) {
    cudaStream_t st = (cudaStream_t)stream;
    TGAN_CHECK_ARG(B > 0 && N > 0 && Q > 0 && M >= 0, "tgan_relattn_fwd: bad dims");
    TGAN_CHECK_ARG(ldq % 8 == 0 && ldkv % 8 == 0 && ldr % 8 == 0 && ldo % 8 == 0, "tgan_relattn_fwd: ld must be multiples of 8");
    if (impl != TGAN_IMPL_SIMT && dtype == TGAN_BF16) {
        int rc = tgan_relattn_fwd_tc(q, ldq, k, v, ldkv, r, ldr, u, vb, reset, key_start, key_base, out, ldo, lse, B, N,
                                     Q, M, msl, same_length, scale, drop_p, seed, site, st);
        if (rc >= 0) return rc;
        if (impl == TGAN_IMPL_TC) return 3;
    } else if (impl == TGAN_IMPL_TC) {
        tgan_set_error("tgan_relattn_fwd: tcgen05 path needs bf16");
        return 3;
    }
    return tgan_relattn_fwd_simt(dtype, q, ldq, k, v, ldkv, r, ldr, u, vb, reset, key_start, key_base, out, ldo, lse, B,
                                 N, Q, M, msl, same_length, scale, drop_p, seed, site, st);
}

extern "C" int tgan_relattn_fwd(int dtype, const void* q, int64_t ldq, const void* k, const void* v, int64_t ldkv,
                                const void* r, int64_t ldr, const float* u, const float* vb, const uint8_t* reset,
                                void* out, int64_t ldo, float* lse, int B, int N, int Q, int M, int msl,
                                int same_length, float scale, float drop_p, uint64_t seed, uint64_t site, int impl,
                                void* stream) {
    return relattn_fwd_impl(dtype, q, ldq, k, v, ldkv, r, ldr, u, vb, reset, nullptr, 0, out, ldo, lse, B, N, Q, M, msl,
                            same_length, scale, drop_p, seed, site, impl, stream);
}

extern "C" int tgan_relattn_fwd_ragged(int dtype, const void* q, int64_t ldq, const void* k, const void* v,
                                       int64_t ldkv, const void* r, int64_t ldr, const float* u, const float* vb,
                                       const uint8_t* reset, void* out, int64_t ldo, float* lse, int B, int N, int Q,
                                       int M, int msl, int same_length, float scale, float drop_p, uint64_t seed,
                                       uint64_t site, int impl, void* stream, const int32_t* key_start,
                                       int64_t key_base) {
    return relattn_fwd_impl(dtype, q, ldq, k, v, ldkv, r, ldr, u, vb, reset, key_start, key_base, out, ldo, lse, B, N, Q,
                            M, msl, same_length, scale, drop_p, seed, site, impl, stream);
}

extern "C" int tgan_relattn_bwd(int dtype, const void* q, int64_t ldq, const void* k, const void* v, int64_t ldkv,
                                const void* r, int64_t ldr, const float* u, const float* vb, const uint8_t* reset,
                                const void* out, const void* dout, int64_t ldo, const float* lse, float* delta,
                                void* dq, void* dk, void* dv, int64_t lddkv, float* dr, int64_t lddr, float* du,
                                float* dvb, int B, int N, int Q, int M, int msl, int same_length, float scale,
                                float drop_p, uint64_t seed, uint64_t site, int impl, void* stream) {
    cudaStream_t st = (cudaStream_t)stream;
    TGAN_CHECK_ARG(B > 0 && N > 0 && Q > 0 && M >= 0, "tgan_relattn_bwd: bad dims");
    TGAN_CHECK_ARG(ldq % 8 == 0 && ldkv % 8 == 0 && ldr % 8 == 0 && ldo % 8 == 0 && lddkv % 8 == 0,
                   "tgan_relattn_bwd: ld must be multiples of 8");
    if (impl != TGAN_IMPL_SIMT && dtype == TGAN_BF16) {
        int rc = tgan_relattn_bwd_tc(q, ldq, k, v, ldkv, r, ldr, u, vb, reset, out, dout, ldo, lse, delta, dq, dk, dv,
                                     lddkv, dr, lddr, du, dvb, B, N, Q, M, msl, same_length, scale, drop_p, seed, site,
                                     st);
        if (rc >= 0) return rc;
        if (impl == TGAN_IMPL_TC) return 3;
    } else if (impl == TGAN_IMPL_TC) {
        tgan_set_error("tgan_relattn_bwd: tcgen05 path needs bf16");
        return 3;
    }
    return tgan_relattn_bwd_simt(dtype, q, ldq, k, v, ldkv, r, ldr, u, vb, reset, out, dout, ldo, lse, delta, dq, dk,
                                 dv, lddkv, dr, lddr, du, dvb, B, N, Q, M, msl, same_length, scale, drop_p, seed, site,
                                 st);
}
