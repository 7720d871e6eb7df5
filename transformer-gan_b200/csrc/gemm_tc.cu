// tcgen05 GEMM for sm_100a: C[M,N] = epi(opA(A) * opB(B)), bf16 operands, fp32 accumulation in TMEM.
//
// Persistent, warp-specialised kernel (one CTA per SM, 192 threads):
//   warp 0      TMA producer: cp.async.bulk.tensor tiles (128-byte swizzle) into a STAGES-deep shared-memory ring
//   warp 1      MMA issuer: one thread issues tcgen05.mma (M=128, N=BN, K=16) per 16-wide k slice, commits the
//               stage back to the producer (tcgen05.commit -> mbarrier) and the finished tile to the epilogue
//   warps 2..9  epilogue: tcgen05.ld the 128 x BN fp32 accumulator (double-buffered in TMEM, 2 x BN columns), apply
//               alpha / bias / ReLU / ReLU-mask / dropout / residual with the flag set fixed at COMPILE time for the
//               combinations the layer stack uses (a run-time-flag epilogue is branch- and I-cache-bound: 5300 vs
//               500 clocks per tile), stage [32 rows][128 bytes] boxes in swizzled shared memory and let the copy
//               engine write them (TMA store; TMA reduce-add for gradient accumulation and split-K partial sums).
//               Operands the copy engine cannot address (unaligned rows, bf16 accumulation) take a direct path.
// Operand layouts: K-major (row-major [rows, K]) or MN-major (row-major [K, rows]); both are read by TMA with
// the same 64 x 64-element swizzled boxes and described to the tensor core through the UMMA descriptors.
// Used for every dense contraction of the path: QKV / R / O projections, FFN, logits, and all dgrad / wgrad.
#include <string.h>

#include "tc_common.cuh"

namespace tc {

static EncodeTiledFn g_encode = nullptr;
EncodeTiledFn get_encode_fn() {
    if (g_encode) return g_encode;
    void* fn = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres) != cudaSuccess ||
        qres != cudaDriverEntryPointSuccess)
        return nullptr;
    g_encode = (EncodeTiledFn)fn;
    return g_encode;
}

int make_tmap_2d(CUtensorMap* m, const void* base, uint64_t rows, uint64_t cols, uint64_t ld, uint32_t box_rows,
                 uint32_t box_cols) {
    EncodeTiledFn enc = get_encode_fn();
    if (!enc) { tgan_set_error("cuTensorMapEncodeTiled entry point not available"); return 2; }
    cuuint64_t dims[2] = {cols, rows};
    cuuint64_t strides[1] = {ld * 2};
    cuuint32_t box[2] = {box_cols, box_rows};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), dims, strides, box, estr,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
        tgan_set_error("cuTensorMapEncodeTiled(2d) failed: %d (rows %llu cols %llu ld %llu)", (int)r,
                       (unsigned long long)rows, (unsigned long long)cols, (unsigned long long)ld);
        return 2;
    }
    return 0;
}

int make_tmap_2d_dt(CUtensorMap* m, const void* base, uint64_t rows, uint64_t cols, uint64_t ld, uint32_t box_rows,
                    uint32_t box_cols, int is_f32) {
    EncodeTiledFn enc = get_encode_fn();
    if (!enc) { tgan_set_error("cuTensorMapEncodeTiled entry point not available"); return 2; }
    const uint64_t esz = is_f32 ? 4 : 2;
    cuuint64_t dims[2] = {cols, rows};
    cuuint64_t strides[1] = {ld * esz};
    cuuint32_t box[2] = {box_cols, box_rows};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = enc(m, is_f32 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2,
                     const_cast<void*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                     CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
        tgan_set_error("cuTensorMapEncodeTiled(2d, %s) failed: %d (rows %llu cols %llu ld %llu)", is_f32 ? "f32" : "bf16",
                       (int)r, (unsigned long long)rows, (unsigned long long)cols, (unsigned long long)ld);
        return 2;
    }
    return 0;
}

int make_tmap_3d(CUtensorMap* m, const void* base, uint64_t d0, uint64_t d1, uint64_t d2, uint64_t stride1,
                 uint64_t stride2, uint32_t b0, uint32_t b1, uint32_t b2) {
    EncodeTiledFn enc = get_encode_fn();
    if (!enc) { tgan_set_error("cuTensorMapEncodeTiled entry point not available"); return 2; }
    cuuint64_t dims[3] = {d0, d1, d2};
    cuuint64_t strides[2] = {stride1 * 2, stride2 * 2};
    cuuint32_t box[3] = {b0, b1, b2};
    cuuint32_t estr[3] = {1, 1, 1};
    CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, const_cast<void*>(base), dims, strides, box, estr,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
        tgan_set_error("cuTensorMapEncodeTiled(3d) failed: %d", (int)r);
        return 2;
    }
    return 0;
}

int sm_count() {
    static int n = 0;
    if (n == 0) {
        int dev = 0;
        cudaGetDevice(&dev);
        if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) n = 148;
    }
    return n;
}
}  // namespace tc

namespace {
using namespace tc;

constexpr int BM = 128, BK = 64;
constexpr int EPI_WARPS = 8;
constexpr int NUM_THREADS = 64 + 32 * EPI_WARPS;  // warp 0 TMA, warp 1 MMA, warps 2..9 epilogue
constexpr int A_BYTES = BM * BK * 2;  // 16 KB
constexpr int EPI_ATOMIC = 1 << 20;   // internal: split-K partial sums are added with red.global.add (fp32 C)
constexpr int EPI_VEC = 1 << 21;      // internal: C / aux rows are 16-byte aligned -> 8-wide vector accesses
constexpr int EPI_BIAS_VEC = 1 << 22; // internal: bias pointer is 16-byte aligned
constexpr int EPI_TMA = 1 << 23;      // internal: C leaves through shared memory + TMA store (reduce-add for ACCUM / split-K)
constexpr int EPI_ALPHA = 1 << 24;    // internal: alpha != 1
constexpr int STAGE_BYTES = 32 * 128; // one epilogue warp's staging box: 32 rows x 128 bytes, 128-byte swizzle

template <int BN> struct Cfg {
    static constexpr int STAGES = BN == 256 ? 4 : 6;
    static constexpr int B_BYTES = BN * BK * 2;
    static constexpr int SMEM = STAGES * (A_BYTES + B_BYTES) + EPI_WARPS * STAGE_BYTES + 8 * (2 * STAGES + 4) + 16 + 1024;
    static_assert(SMEM <= 232448, "shared memory budget");
};

__device__ __forceinline__ void red_add_f32x4(float* addr, const float* v) {
    asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(addr), "f"(v[0]), "f"(v[1]), "f"(v[2]), "f"(v[3])
                 : "memory");
}

// Final values (before ACCUM) of the 8 consecutive columns col .. col+7 of output row `row`; nv <= 8 of them exist.
// thread = TMEM lane = output row, so aux / bias accesses are row-contiguous 16/32-byte vectors.
__device__ __forceinline__ void epi_values8(float* v, const uint32_t* regs, int64_t row, int col, int nv, int64_t ldc,
                                            const EpiParams& ep, uint32_t dkey) {
    const int flags = ep.flags;
#pragma unroll
    for (int t = 0; t < 8; ++t) v[t] = __uint_as_float(regs[t]) * ep.alpha;
    if ((flags & EPI_VEC) && nv == 8) {
        if (flags & TGAN_EPI_BIAS) {
            float b[8];
            if (flags & EPI_BIAS_VEC) load8(ep.bias + col, b);
            else {
#pragma unroll
                for (int t = 0; t < 8; ++t) b[t] = __ldg(ep.bias + col + t);
            }
#pragma unroll
            for (int t = 0; t < 8; ++t) v[t] += b[t];
        }
        if (flags & TGAN_EPI_RELU) {
#pragma unroll
            for (int t = 0; t < 8; ++t) v[t] = fmaxf(v[t], 0.f);
        }
        float a[8];
        if (flags & (TGAN_EPI_MASK_POS | TGAN_EPI_ADD_AUX)) {
            if (ep.aux_is_f32) load8((const float*)ep.aux + row * ep.ldaux + col, a);
            else load8((const bf16*)ep.aux + row * ep.ldaux + col, a);
        }
        if (flags & TGAN_EPI_MASK_POS) {
#pragma unroll
            for (int t = 0; t < 8; ++t) v[t] = a[t] > 0.f ? v[t] : 0.f;
        }
        if (flags & TGAN_EPI_DROPOUT) {
            const uint32_t keep = dropout_keep8_k(dkey, (uint64_t)row * ldc + col, ep.drop_thresh);
#pragma unroll
            for (int t = 0; t < 8; ++t) v[t] = ((keep >> t) & 1) ? v[t] * ep.drop_scale : 0.f;
        }
        if (flags & TGAN_EPI_ADD_AUX) {
#pragma unroll
            for (int t = 0; t < 8; ++t) v[t] += a[t];
        }
    } else {
#pragma unroll
        for (int t = 0; t < 8; ++t) {
            float x = 0.f;
            if (t < nv) {
                x = v[t];
                if (flags & TGAN_EPI_BIAS) x += __ldg(ep.bias + col + t);
                if (flags & TGAN_EPI_RELU) x = fmaxf(x, 0.f);
                float a = 0.f;
                if (flags & (TGAN_EPI_MASK_POS | TGAN_EPI_ADD_AUX))
                    a = ep.aux_is_f32 ? ((const float*)ep.aux)[row * ep.ldaux + col + t]
                                      : to_f(((const bf16*)ep.aux)[row * ep.ldaux + col + t]);
                if (flags & TGAN_EPI_MASK_POS) x = a > 0.f ? x : 0.f;
                if (flags & TGAN_EPI_DROPOUT)
                    x = dropout_keep_k(dkey, (uint64_t)row * ldc + col + t, ep.drop_thresh) ? x * ep.drop_scale : 0.f;
                if (flags & TGAN_EPI_ADD_AUX) x += a;
            }
            v[t] = x;
        }
    }
}

// Direct-to-global sink of one 32-column accumulator segment (operands that the copy engine cannot address:
// unaligned C rows, bf16 accumulation).  Each thread writes its own row.
template <typename TC>
__device__ __forceinline__ void epi_row32(const uint32_t* regs, int64_t row, int col0, int N, TC* __restrict__ C,
                                          int64_t ldc, const EpiParams& ep, uint32_t dkey) {
    const int flags = ep.flags;
#pragma unroll
    for (int g = 0; g < 4; ++g) {
        const int col = col0 + 8 * g;
        if (col >= N) break;
        const int nv = min(8, N - col);
        float v[8];
        epi_values8(v, regs + 8 * g, row, col, nv, ldc, ep, dkey);
        TC* cp = C + row * ldc + col;
        if ((flags & EPI_VEC) && nv == 8) {
            if (flags & EPI_ATOMIC) {
                red_add_f32x4((float*)cp, v);
                red_add_f32x4((float*)cp + 4, v + 4);
            } else {
                if (flags & TGAN_EPI_ACCUM) {
                    float c[8];
                    load8(cp, c);
#pragma unroll
                    for (int t = 0; t < 8; ++t) v[t] += c[t];
                }
                store8(cp, v);
            }
        } else {
#pragma unroll
            for (int t = 0; t < 8; ++t) {
                if (t < nv) {
                    float x = v[t];
                    if (flags & EPI_ATOMIC) atomicAdd((float*)(cp + t), x);
                    else {
                        if (flags & TGAN_EPI_ACCUM) x += to_f(cp[t]);
                        cp[t] = from_f<TC>(x);
                    }
                }
            }
        }
    }
}

// Compile-time epilogue (EPI = the public flag bits that apply + EPI_ALPHA): vector-aligned operands, N % 8 == 0, bf16
// aux.  The hot shapes of the layer stack all take this path; no per-flag branches, no scalar tail.
template <int EPI>
__device__ __forceinline__ void epi_values8_ct(float* v, const uint32_t* regs, int64_t row, int col, int64_t ldc,
                                               const EpiParams& ep, uint32_t dkey) {
#pragma unroll
    for (int t = 0; t < 8; ++t) v[t] = (EPI & EPI_ALPHA) ? __uint_as_float(regs[t]) * ep.alpha : __uint_as_float(regs[t]);
    if constexpr ((EPI & TGAN_EPI_BIAS) != 0) {
        float b[8];
        load8(ep.bias + col, b);
#pragma unroll
        for (int t = 0; t < 8; ++t) v[t] += b[t];
    }
    if constexpr ((EPI & TGAN_EPI_RELU) != 0) {
#pragma unroll
        for (int t = 0; t < 8; ++t) v[t] = fmaxf(v[t], 0.f);
    }
    float a[8];
    if constexpr ((EPI & (TGAN_EPI_MASK_POS | TGAN_EPI_ADD_AUX)) != 0) load8((const bf16*)ep.aux + row * ep.ldaux + col, a);
    if constexpr ((EPI & TGAN_EPI_MASK_POS) != 0) {
#pragma unroll
        for (int t = 0; t < 8; ++t) v[t] = a[t] > 0.f ? v[t] : 0.f;
    }
    if constexpr ((EPI & TGAN_EPI_DROPOUT) != 0) {
        const uint32_t keep = dropout_keep8_k(dkey, (uint64_t)row * ldc + col, ep.drop_thresh);
#pragma unroll
        for (int t = 0; t < 8; ++t) v[t] = ((keep >> t) & 1) ? v[t] * ep.drop_scale : 0.f;
    }
    if constexpr ((EPI & TGAN_EPI_ADD_AUX) != 0) {
#pragma unroll
        for (int t = 0; t < 8; ++t) v[t] += a[t];
    }
}

// Shared-memory sink: the 32-column segment of row r (0..31 inside this warp's staging tile) goes into the
// 128-byte-swizzled [32 rows][128 bytes] box that the TMA store / reduce reads.  seg = index of the 32-column
// segment inside the box (bf16: 0 or 1, fp32: 0).
template <typename TC, int EPI>
__device__ __forceinline__ void epi_row32_smem(const uint32_t* regs, int64_t row, int r, int col0, int seg, int N,
                                               uint8_t* stage, int64_t ldc, const EpiParams& ep, uint32_t dkey) {
#pragma unroll
    for (int g = 0; g < 4; ++g) {
        const int col = col0 + 8 * g;
        float v[8];
        if constexpr (EPI >= 0) {
            epi_values8_ct<EPI>(v, regs + 8 * g, row, col, ldc, ep, dkey);  // N % 8 == 0: a started segment is whole groups
        } else {
            const int nv = max(0, min(8, N - col));
            if (nv > 0) epi_values8(v, regs + 8 * g, row, col, nv, ldc, ep, dkey);
            else {
#pragma unroll
                for (int t = 0; t < 8; ++t) v[t] = 0.f;
            }
        }
        if constexpr (sizeof(TC) == 2) {
            store8(reinterpret_cast<bf16*>(stage + sw128_off(r, 4 * seg + g)), v);
        } else {
            *reinterpret_cast<float4*>(stage + sw128_off(r, 2 * g)) = make_float4(v[0], v[1], v[2], v[3]);
            *reinterpret_cast<float4*>(stage + sw128_off(r, 2 * g + 1)) = make_float4(v[4], v[5], v[6], v[7]);
        }
    }
}

// work item w -> (output tile, K split).  Consecutive CTAs share the A row block (tiles of one m are adjacent).
struct Work {
    int m0, n0, kb0, kb1;
};
template <int BN>
__device__ __forceinline__ Work get_work(int w, int num_tiles, int tiles_n, int nk, int kb_per_split) {
    const int tile = w % num_tiles, split = w / num_tiles;
    Work r;
    r.m0 = (tile / tiles_n) * BM;
    r.n0 = (tile % tiles_n) * BN;
    r.kb0 = split * kb_per_split;
    r.kb1 = min(nk, r.kb0 + kb_per_split);
    return r;
}

// EPI >= 0: compile-time epilogue (see epi_values8_ct; always the TMA sink); EPI = -1: run-time flags, either sink
template <int BN, bool A_MN, bool B_MN, typename TC, int EPI>
__global__ void __launch_bounds__(NUM_THREADS, 1)
gemm_tc_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
               const __grid_constant__ CUtensorMap tmC, TC* __restrict__ C, int64_t ldc, int M, int N, int K, int splits,
               int kb_per_split, EpiParams ep) {
    constexpr int STAGES = Cfg<BN>::STAGES;
    constexpr int B_BYTES = Cfg<BN>::B_BYTES;
    extern __shared__ uint8_t smem_raw[];
    const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
    const uint32_t sA = base, sB = base + STAGES * A_BYTES;
    const uint32_t sStage = sB + STAGES * B_BYTES;  // 1024-byte aligned: EPI_WARPS staging boxes
    const uint32_t sBar = sStage + EPI_WARPS * STAGE_BYTES;
    const uint32_t full0 = sBar, empty0 = sBar + 8 * STAGES, tfull0 = sBar + 16 * STAGES, tempty0 = tfull0 + 16;
    const uint32_t sTmemPtr = tempty0 + 16;
    uint8_t* gen_base = smem_raw + (base - smem_u32(smem_raw));
    volatile uint32_t* tmem_ptr_gen = reinterpret_cast<volatile uint32_t*>(gen_base + (sTmemPtr - base));

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int tiles_n = (N + BN - 1) / BN, tiles_m = (M + BM - 1) / BM;
    const int num_tiles = tiles_m * tiles_n;
    const int num_work = num_tiles * splits;
    const int nk = (K + BK - 1) / BK;

    if (threadIdx.x == 0) {
        for (int s = 0; s < STAGES; ++s) { mbar_init(full0 + 8 * s, 1); mbar_init(empty0 + 8 * s, 1); }
        for (int a = 0; a < 2; ++a) { mbar_init(tfull0 + 8 * a, 1); mbar_init(tempty0 + 8 * a, EPI_WARPS); }
        fence_barrier_init();
    }
    if (warp == 0 && lane == 0) {
        tma_prefetch_desc(&tmA); tma_prefetch_desc(&tmB);
        if (EPI >= 0 || (ep.flags & EPI_TMA)) tma_prefetch_desc(&tmC);
    }
    if (warp == 1) tmem_alloc(sTmemPtr, 2 * BN);
    tcgen05_fence_before();
    __syncthreads();
    tcgen05_fence_after();
    const uint32_t tmem_base = *tmem_ptr_gen;

    if (warp == 0) {
        // ===================== TMA producer =====================
        if (lane == 0) {
            int s = 0; uint32_t ph = 0;
            for (int w = blockIdx.x; w < num_work; w += gridDim.x) {
                const Work wk = get_work<BN>(w, num_tiles, tiles_n, nk, kb_per_split);
                for (int kb = wk.kb0; kb < wk.kb1; ++kb) {
                    mbar_wait(empty0 + 8 * s, ph ^ 1);
                    const uint32_t fb = full0 + 8 * s;
                    mbar_expect_tx(fb, A_BYTES + B_BYTES);
                    const uint32_t a_dst = sA + s * A_BYTES, b_dst = sB + s * B_BYTES;
                    if (!A_MN) tma_load_2d(a_dst, &tmA, fb, kb * BK, wk.m0);
                    else {
#pragma unroll
                        for (int bx = 0; bx < BM / 64; ++bx) tma_load_2d(a_dst + bx * 8192, &tmA, fb, wk.m0 + 64 * bx, kb * BK);
                    }
                    if (!B_MN) tma_load_2d(b_dst, &tmB, fb, kb * BK, wk.n0);
                    else {
#pragma unroll
                        for (int bx = 0; bx < BN / 64; ++bx) tma_load_2d(b_dst + bx * 8192, &tmB, fb, wk.n0 + 64 * bx, kb * BK);
                    }
                    if (++s == STAGES) { s = 0; ph ^= 1; }
                }
            }
        }
    } else if (warp == 1) {
        // ===================== MMA issuer =====================
        // The whole warp runs the loop (converged waits); one elected lane issues.  Descriptors are built once per
        // operand and advanced by adding to the 14-bit start-address field, so each tcgen05.mma costs a few uniform ops.
        constexpr uint32_t idesc = umma_idesc_bf16(BM, BN, A_MN ? 1 : 0, B_MN ? 1 : 0);
        const uint64_t da0 = A_MN ? umma_smem_desc(sA, 8192, 1024) : umma_smem_desc(sA, 16, 1024);
        const uint64_t db0 = B_MN ? umma_smem_desc(sB, 8192, 1024) : umma_smem_desc(sB, 16, 1024);
        constexpr uint32_t a_kstep = (A_MN ? 2048 : 32) >> 4, b_kstep = (B_MN ? 2048 : 32) >> 4;
        int s = 0; uint32_t ph = 0; int it = 0;
        for (int w = blockIdx.x; w < num_work; w += gridDim.x, ++it) {
            const Work wk = get_work<BN>(w, num_tiles, tiles_n, nk, kb_per_split);
            const int as = it & 1; const uint32_t aph = (it >> 1) & 1;
            mbar_wait(tempty0 + 8 * as, aph ^ 1);
            tcgen05_fence_after();
            const uint32_t d_tmem = tmem_base + as * BN;
            for (int kb = wk.kb0; kb < wk.kb1; ++kb) {
                mbar_wait(full0 + 8 * s, ph);
                tcgen05_fence_after();
                if (elect_one()) {
                    const uint64_t da = da0 + (uint64_t)((s * A_BYTES) >> 4), db = db0 + (uint64_t)((s * B_BYTES) >> 4);
#pragma unroll
                    for (int k = 0; k < BK / 16; ++k)
                        umma_bf16(d_tmem, da + k * a_kstep, db + k * b_kstep, idesc, (kb != wk.kb0 || k != 0) ? 1u : 0u);
                    umma_commit(empty0 + 8 * s);  // frees the smem stage once these MMAs have read it
                    if (kb == wk.kb1 - 1) umma_commit(tfull0 + 8 * as);  // accumulator complete -> epilogue
                }
                __syncwarp();
                if (++s == STAGES) { s = 0; ph ^= 1; }
            }
        }
    } else {
        // ===================== epilogue warps =====================
        // warp w may only touch TMEM lanes 32*(w%4) .. +31; the two warps sharing a lane quarter split the columns.
        // TMA path: each warp stages a [32 rows][128 bytes] box in shared memory (swizzled) and lets the copy engine
        // write (or reduce-add) full 128-byte lines; the direct path stores row-strided 16-byte vectors itself.
        const int eq = warp & 3, eh = (warp - 2) >> 2;
        constexpr int BOXC = 128 / (int)sizeof(TC);  // columns per staging box (bf16: 64, fp32: 32)
        const uint32_t dkey = step_fold(ep.drop_key);
        const bool use_tma = EPI >= 0 || (ep.flags & EPI_TMA) != 0;
        const bool reduce = (ep.flags & (EPI_ATOMIC | TGAN_EPI_ACCUM)) != 0;
        uint8_t* stage = gen_base + (sStage - base) + (warp - 2) * STAGE_BYTES;
        const uint32_t stage_u32 = sStage + (warp - 2) * STAGE_BYTES;
        bool pending = false;  // a bulk store issued by this warp may still be reading the staging box
        int it = 0;
        for (int w = blockIdx.x; w < num_work; w += gridDim.x, ++it) {
            const Work wk = get_work<BN>(w, num_tiles, tiles_n, nk, kb_per_split);
            const int as = it & 1; const uint32_t aph = (it >> 1) & 1;
            mbar_wait(tfull0 + 8 * as, aph);
            tcgen05_fence_after();
            const int row0 = wk.m0 + 32 * eq;
            const int64_t row = row0 + lane;
            if (use_tma) {
#pragma unroll 1
                for (int b0 = eh * (BN / 2); b0 < (eh + 1) * (BN / 2); b0 += BOXC) {
                    if (wk.n0 + b0 >= N) break;  // warp-uniform
#pragma unroll
                    for (int seg = 0; seg < BOXC / 32; ++seg) {
                        const int c0 = b0 + 32 * seg;
                        if (wk.n0 + c0 >= N) break;  // warp-uniform; the rest of the box is clipped by the tensor map
                        uint32_t regs[32];
                        tmem_ld32(tmem_base + as * BN + c0 + ((uint32_t)(32 * eq) << 16), regs);
                        tmem_ld_wait();
                        if (seg == 0 && pending) {
                            if (lane == 0) tma_store_wait_read();
                            __syncwarp();
                            pending = false;
                        }
                        if (row < M) epi_row32_smem<TC, EPI>(regs, row, lane, wk.n0 + c0, seg, N, stage, ldc, ep, dkey);
                    }
                    fence_proxy_async_smem();
                    __syncwarp();
                    if (lane == 0) {
                        if (reduce) tma_reduce_add_2d(&tmC, stage_u32, wk.n0 + b0, row0);
                        else tma_store_2d(&tmC, stage_u32, wk.n0 + b0, row0);
                        tma_store_commit();
                    }
                    pending = true;
                }
            } else if constexpr (EPI < 0) {
#pragma unroll 1
                for (int c0 = eh * (BN / 2); c0 < (eh + 1) * (BN / 2); c0 += 32) {
                    if (wk.n0 + c0 >= N) break;  // warp-uniform
                    uint32_t regs[32];
                    tmem_ld32(tmem_base + as * BN + c0 + ((uint32_t)(32 * eq) << 16), regs);
                    tmem_ld_wait();
                    if (row < M) epi_row32<TC>(regs, row, wk.n0 + c0, N, C, ldc, ep, dkey);
                }
            }
            tcgen05_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(tempty0 + 8 * as);
        }
        if (pending && lane == 0) tma_store_wait_all();
    }
    tcgen05_fence_before();
    __syncthreads();
    if (warp == 1) {
        tcgen05_fence_after();
        tmem_dealloc(tmem_base, 2 * BN);
    }
}

// ============================================================================================================
// 2-CTA variant (tcgen05 cta_group::2): a CTA pair on one TPC computes a 256 x 256 tile.  Each CTA stages its own 128
// rows of A and its own 128-row HALF of the B tile; one tcgen05.mma (M = 256) issued by the leader reads both CTAs'
// shared memory and writes each CTA's 128 x 256 accumulator into that CTA's TMEM.  Per CTA and k-block the L2 -> SM
// traffic drops from 48 KB (A 16 + B 32) to 32 KB: the 1-CTA kernel on the K = 512 projections is bound by exactly
// that stream (9 GB at ~13 TB/s for the K/V projection).  nn.Linear layout only (A, B K-major), compile-time
// epilogues only (TMA sink).
// ============================================================================================================
constexpr int STAGES2 = 5;
constexpr int B2_BYTES = 128 * BK * 2;  // this CTA's half of the 256-row B tile
constexpr int SMEM2 = STAGES2 * (A_BYTES + B2_BYTES) + EPI_WARPS * STAGE_BYTES + 8 * (2 * STAGES2 + 4) + 16 + 1024;
static_assert(SMEM2 <= 232448, "shared memory budget");

__device__ __forceinline__ uint32_t cluster_ctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// shared::cluster address of `saddr` (a shared::cta address of this CTA) in the CTA of rank `rank`
__device__ __forceinline__ uint32_t mapa_u32(uint32_t saddr, uint32_t rank) {
    uint32_t r;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(saddr), "r"(rank));
    return r;
}
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_addr) {
    asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
// TMA load whose completion bytes are signalled on an mbarrier that may live in the PEER CTA (the pair leader's)
__device__ __forceinline__ void tma_load_2d_2sm(uint32_t dst, const CUtensorMap* m, uint32_t bar_cluster, int c0, int c1) {
    asm volatile(
        "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(dst),
        "l"(m), "r"(bar_cluster), "r"(c0), "r"(c1)
        : "memory");
}
__device__ __forceinline__ void umma_bf16_2sm(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc,
                                              uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(d_tmem),
        "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
        : "memory");
}
// arrive (once the MMAs issued so far have completed) on the mbarrier at this offset in BOTH CTAs of the pair
__device__ __forceinline__ void umma_commit_2sm(uint32_t bar) {
    asm volatile(
        "tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(bar),
        "h"((uint16_t)3)
        : "memory");
}
__device__ __forceinline__ void tmem_alloc_2sm(uint32_t dst_smem, uint32_t ncols) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(dst_smem), "r"(ncols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc_2sm(uint32_t taddr, uint32_t ncols) {
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}

template <typename TC, int EPI>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(NUM_THREADS, 1)
gemm_tc2_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                const __grid_constant__ CUtensorMap tmC, int64_t ldc, int M, int N, int K, EpiParams ep) {
    static_assert(EPI >= 0, "2-CTA kernel: compile-time epilogues only");
    constexpr int BN2 = 256, BM2 = 256;
    extern __shared__ uint8_t smem_raw[];
    const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
    const uint32_t sA = base, sB = base + STAGES2 * A_BYTES;
    const uint32_t sStage = sB + STAGES2 * B2_BYTES;
    const uint32_t sBar = sStage + EPI_WARPS * STAGE_BYTES;
    const uint32_t full0 = sBar, empty0 = sBar + 8 * STAGES2, tfull0 = sBar + 16 * STAGES2, tempty0 = tfull0 + 16;
    const uint32_t sTmemPtr = tempty0 + 16;
    uint8_t* gen_base = smem_raw + (base - smem_u32(smem_raw));
    volatile uint32_t* tmem_ptr_gen = reinterpret_cast<volatile uint32_t*>(gen_base + (sTmemPtr - base));

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t rank = cluster_ctarank();
    const int pair = blockIdx.x >> 1, npairs = gridDim.x >> 1;
    const int tiles_n = (N + BN2 - 1) / BN2, tiles_m = (M + BM2 - 1) / BM2;
    const int num_tiles = tiles_m * tiles_n;
    const int nk = (K + BK - 1) / BK;

    if (threadIdx.x == 0) {
        for (int s = 0; s < STAGES2; ++s) { mbar_init(full0 + 8 * s, 1); mbar_init(empty0 + 8 * s, 1); }
        for (int a = 0; a < 2; ++a) { mbar_init(tfull0 + 8 * a, 1); mbar_init(tempty0 + 8 * a, 2 * EPI_WARPS); }
        fence_barrier_init();
    }
    if (warp == 0 && lane == 0) { tma_prefetch_desc(&tmA); tma_prefetch_desc(&tmB); tma_prefetch_desc(&tmC); }
    if (warp == 1) tmem_alloc_2sm(sTmemPtr, 2 * BN2);
    tcgen05_fence_before();
    __syncthreads();
    cluster_sync_all();  // both CTAs' barriers are initialised before anyone signals across the pair
    tcgen05_fence_after();
    const uint32_t tmem_base = *tmem_ptr_gen;

    if (warp == 0) {
        // ===================== TMA producer (both CTAs; completion bytes land on the LEADER's full barrier) =====================
        if (lane == 0) {
            int s = 0; uint32_t ph = 0;
            for (int t = pair; t < num_tiles; t += npairs) {
                const int m0 = (t / tiles_n) * BM2 + 128 * (int)rank, n0 = (t % tiles_n) * BN2 + 128 * (int)rank;
                for (int kb = 0; kb < nk; ++kb) {
                    mbar_wait(empty0 + 8 * s, ph ^ 1);
                    const uint32_t fb = mapa_u32(full0 + 8 * s, 0);
                    if (rank == 0) mbar_expect_tx(full0 + 8 * s, 2 * (A_BYTES + B2_BYTES));
                    tma_load_2d_2sm(sA + s * A_BYTES, &tmA, fb, kb * BK, m0);
                    tma_load_2d_2sm(sB + s * B2_BYTES, &tmB, fb, kb * BK, n0);
                    if (++s == STAGES2) { s = 0; ph ^= 1; }
                }
            }
        }
    } else if (warp == 1) {
        // ===================== MMA issuer (leader CTA only) =====================
        if (rank == 0) {
            constexpr uint32_t idesc = umma_idesc_bf16(BM2, BN2, 0, 0);
            const uint64_t da0 = umma_smem_desc(sA, 16, 1024), db0 = umma_smem_desc(sB, 16, 1024);
            int s = 0; uint32_t ph = 0; int it = 0;
            for (int t = pair; t < num_tiles; t += npairs, ++it) {
                const int as = it & 1; const uint32_t aph = (it >> 1) & 1;
                mbar_wait(tempty0 + 8 * as, aph ^ 1);  // the epilogue warps of BOTH CTAs have drained this accumulator
                tcgen05_fence_after();
                const uint32_t d_tmem = tmem_base + as * BN2;
                for (int kb = 0; kb < nk; ++kb) {
                    mbar_wait(full0 + 8 * s, ph);
                    tcgen05_fence_after();
                    if (elect_one()) {
                        const uint64_t da = da0 + (uint64_t)((s * A_BYTES) >> 4), db = db0 + (uint64_t)((s * B2_BYTES) >> 4);
#pragma unroll
                        for (int k = 0; k < BK / 16; ++k) umma_bf16_2sm(d_tmem, da + 2 * k, db + 2 * k, idesc, (kb | k) ? 1u : 0u);
                        umma_commit_2sm(empty0 + 8 * s);
                        if (kb == nk - 1) umma_commit_2sm(tfull0 + 8 * as);
                    }
                    __syncwarp();
                    if (++s == STAGES2) { s = 0; ph ^= 1; }
                }
            }
        }
    } else {
        // ===================== epilogue warps (each CTA drains its own 128 x 256 accumulator) =====================
        const int eq = warp & 3, eh = (warp - 2) >> 2;
        constexpr int BOXC = 128 / (int)sizeof(TC);
        const uint32_t dkey = step_fold(ep.drop_key);
        const bool reduce = (ep.flags & (EPI_ATOMIC | TGAN_EPI_ACCUM)) != 0;
        uint8_t* stage = gen_base + (sStage - base) + (warp - 2) * STAGE_BYTES;
        const uint32_t stage_u32 = sStage + (warp - 2) * STAGE_BYTES;
        const uint32_t tempty_leader = mapa_u32(tempty0, 0);
        bool pending = false;
        int it = 0;
        for (int t = pair; t < num_tiles; t += npairs, ++it) {
            const int m0 = (t / tiles_n) * BM2 + 128 * (int)rank, n0 = (t % tiles_n) * BN2;
            const int as = it & 1; const uint32_t aph = (it >> 1) & 1;
            mbar_wait(tfull0 + 8 * as, aph);
            tcgen05_fence_after();
            const int row0 = m0 + 32 * eq;
            const int64_t row = row0 + lane;
#pragma unroll 1
            for (int b0 = eh * (BN2 / 2); b0 < (eh + 1) * (BN2 / 2); b0 += BOXC) {
                if (n0 + b0 >= N) break;
#pragma unroll
                for (int seg = 0; seg < BOXC / 32; ++seg) {
                    const int c0 = b0 + 32 * seg;
                    if (n0 + c0 >= N) break;
                    uint32_t regs[32];
                    tmem_ld32(tmem_base + as * BN2 + c0 + ((uint32_t)(32 * eq) << 16), regs);
                    tmem_ld_wait();
                    if (seg == 0 && pending) {
                        if (lane == 0) tma_store_wait_read();
                        __syncwarp();
                        pending = false;
                    }
                    if (row < M) epi_row32_smem<TC, EPI>(regs, row, lane, n0 + c0, seg, N, stage, ldc, ep, dkey);
                }
                fence_proxy_async_smem();
                __syncwarp();
                if (lane == 0) {
                    if (reduce) tma_reduce_add_2d(&tmC, stage_u32, n0 + b0, row0);
                    else tma_store_2d(&tmC, stage_u32, n0 + b0, row0);
                    tma_store_commit();
                }
                pending = true;
            }
            tcgen05_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive_cluster(tempty_leader + 8 * as);
        }
        if (pending && lane == 0) tma_store_wait_all();
    }
    tcgen05_fence_before();
    __syncthreads();
    cluster_sync_all();  // the leader's MMAs read the peer's shared memory: nobody leaves before both are done
    if (warp == 1) {
        tcgen05_fence_after();
        tmem_dealloc_2sm(tmem_base, 2 * BN2);
    }
}

template <typename TC, int EPI>
int launch_tc2(const CUtensorMap& tmA, const CUtensorMap& tmB, const CUtensorMap& tmC, int64_t ldc, int M, int N, int K,
               const EpiParams& ep, cudaStream_t st) {
    auto kern = gemm_tc2_kernel<TC, EPI>;
    static bool attr_set = false;
    if (!attr_set) {
        TGAN_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM2));
        attr_set = true;
    }
    const int tiles = ceil_div(M, 256) * ceil_div(N, 256);
    const int pairs = tiles < sm_count() / 2 ? tiles : sm_count() / 2;
    kern<<<2 * pairs, NUM_THREADS, SMEM2, st>>>(tmA, tmB, tmC, ldc, M, N, K, ep);  // __cluster_dims__(2, 1, 1)
    TGAN_COUNT_LAUNCH();
    TGAN_LAUNCH_OK();
    return 0;
}

#define TGAN_LAUNCH2_ARGS tmA, tmB, tmC, ldc, M, N, K, ep, st
template <typename TC>
int launch_tc2_epi(int epi_ct, const CUtensorMap& tmA, const CUtensorMap& tmB, const CUtensorMap& tmC, int64_t ldc, int M,
                   int N, int K, const EpiParams& ep, cudaStream_t st) {
    constexpr int B_ = TGAN_EPI_BIAS, R_ = TGAN_EPI_RELU, MP = TGAN_EPI_MASK_POS, AX = TGAN_EPI_ADD_AUX, DR = TGAN_EPI_DROPOUT;
    switch (epi_ct) {
        case 0: return launch_tc2<TC, 0>(TGAN_LAUNCH2_ARGS);
        case B_ | R_: return launch_tc2<TC, B_ | R_>(TGAN_LAUNCH2_ARGS);
        case B_ | R_ | DR: return launch_tc2<TC, B_ | R_ | DR>(TGAN_LAUNCH2_ARGS);
        case AX: return launch_tc2<TC, AX>(TGAN_LAUNCH2_ARGS);
        case AX | DR: return launch_tc2<TC, AX | DR>(TGAN_LAUNCH2_ARGS);
        case B_ | AX: return launch_tc2<TC, B_ | AX>(TGAN_LAUNCH2_ARGS);
        case B_ | AX | DR: return launch_tc2<TC, B_ | AX | DR>(TGAN_LAUNCH2_ARGS);
        case MP: return launch_tc2<TC, MP>(TGAN_LAUNCH2_ARGS);
        case MP | EPI_ALPHA: return launch_tc2<TC, MP | EPI_ALPHA>(TGAN_LAUNCH2_ARGS);
        default: return -1;
    }
}

template <int BN, bool A_MN, bool B_MN, typename TC, int EPI>
int launch_tc(const CUtensorMap& tmA, const CUtensorMap& tmB, const CUtensorMap& tmC, void* C, int64_t ldc, int M, int N,
              int K, int splits, const EpiParams& ep, cudaStream_t st) {
    auto kern = gemm_tc_kernel<BN, A_MN, B_MN, TC, EPI>;
    static bool attr_set = false;
    if (!attr_set) {
        TGAN_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg<BN>::SMEM));
        attr_set = true;
    }
    const int nk = ceil_div(K, BK);
    const int kb_per_split = ceil_div(nk, splits);
    splits = ceil_div(nk, kb_per_split);  // no empty split
    const int work = ceil_div(M, BM) * ceil_div(N, BN) * splits;
    const int grid = work < sm_count() ? work : sm_count();
    kern<<<grid, NUM_THREADS, Cfg<BN>::SMEM, st>>>(tmA, tmB, tmC, (TC*)C, ldc, M, N, K, splits, kb_per_split, ep);
    TGAN_COUNT_LAUNCH();
    TGAN_LAUNCH_OK();
    return 0;
}

#define TGAN_LAUNCH_ARGS tmA, tmB, tmC, C, ldc, M, N, K, splits, ep, st
// epi_ct: the compile-time epilogue key, or -1.  The fused epilogues of the layer stack only occur with the
// nn.Linear layout (A and B K-major); every layout has the plain (0) variant for projections / weight gradients.
template <int BN, typename TC>
int launch_layout(int transA, int transB, int epi_ct, const CUtensorMap& tmA, const CUtensorMap& tmB, const CUtensorMap& tmC,
                  void* C, int64_t ldc, int M, int N, int K, int splits, const EpiParams& ep, cudaStream_t st) {
    constexpr int B_ = TGAN_EPI_BIAS, R_ = TGAN_EPI_RELU, MP = TGAN_EPI_MASK_POS, AX = TGAN_EPI_ADD_AUX, DR = TGAN_EPI_DROPOUT;
    // transA = 1 -> A stored [K, M] -> MN-major A;  transB = 0 -> B stored [K, N] -> MN-major B
    if (!transA && transB) {
        switch (epi_ct) {
            case 0: return launch_tc<BN, false, false, TC, 0>(TGAN_LAUNCH_ARGS);
            case B_: return launch_tc<BN, false, false, TC, B_>(TGAN_LAUNCH_ARGS);
            case B_ | R_: return launch_tc<BN, false, false, TC, B_ | R_>(TGAN_LAUNCH_ARGS);
            case B_ | R_ | DR: return launch_tc<BN, false, false, TC, B_ | R_ | DR>(TGAN_LAUNCH_ARGS);
            case AX: return launch_tc<BN, false, false, TC, AX>(TGAN_LAUNCH_ARGS);
            case AX | DR: return launch_tc<BN, false, false, TC, AX | DR>(TGAN_LAUNCH_ARGS);
            case B_ | AX: return launch_tc<BN, false, false, TC, B_ | AX>(TGAN_LAUNCH_ARGS);
            case B_ | AX | DR: return launch_tc<BN, false, false, TC, B_ | AX | DR>(TGAN_LAUNCH_ARGS);
            case MP: return launch_tc<BN, false, false, TC, MP>(TGAN_LAUNCH_ARGS);
            case MP | EPI_ALPHA: return launch_tc<BN, false, false, TC, MP | EPI_ALPHA>(TGAN_LAUNCH_ARGS);
            default: return launch_tc<BN, false, false, TC, -1>(TGAN_LAUNCH_ARGS);
        }
    }
    if (!transA && !transB)
        return epi_ct == 0 ? launch_tc<BN, false, true, TC, 0>(TGAN_LAUNCH_ARGS) : launch_tc<BN, false, true, TC, -1>(TGAN_LAUNCH_ARGS);
    if (transA && transB)
        return epi_ct == 0 ? launch_tc<BN, true, false, TC, 0>(TGAN_LAUNCH_ARGS) : launch_tc<BN, true, false, TC, -1>(TGAN_LAUNCH_ARGS);
    return epi_ct == 0 ? launch_tc<BN, true, true, TC, 0>(TGAN_LAUNCH_ARGS) : launch_tc<BN, true, true, TC, -1>(TGAN_LAUNCH_ARGS);
}
}  // namespace

extern "C" int tgan_has_tcgen05(void) { return 1; }
int tgan_set_step_ctr_gemm_tc(const void* p) { return tgan_set_step_ctr_local(p); }

int tgan_gemm_tc(int dtype_c, int transA, int transB, int M, int N, int K, const void* A, int64_t lda, const void* B,
                 int64_t ldb, void* C, int64_t ldc, const float* bias, const void* aux, int64_t ldaux, int flags,
                 float alpha, float drop_p, uint64_t seed, uint64_t site, int force, cudaStream_t st) {
    if (M <= 0 || N <= 0) return 0;
    const bool aligned = (lda % 8 == 0) && (ldb % 8 == 0) && (((uintptr_t)A & 15) == 0) && (((uintptr_t)B & 15) == 0) && K >= 1;
    if (!aligned) {
        tgan_set_error("tgan_gemm: tcgen05 path needs 16-byte aligned operands and leading dimensions that are multiples of 8");
        return -1;
    }
    // Even a 32-row decode GEMM belongs here: one 128-row MMA tile per 128/256 output columns finishes in a few
    // microseconds, while the FFMA kernel needs ~100 us for the same rows (few CTAs, serial K loop).
    if (!force && 2.0 * M * N * K < 1.0e6) {
        tgan_set_error("tgan_gemm: problem too small for the tcgen05 path");
        return -1;
    }
    const int waste256 = ceil_div(N, 256) * 256 - N, waste128 = ceil_div(N, 128) * 128 - N;
    int BN = (waste256 <= waste128) ? 256 : 128;
    // few tiles (decode-sized GEMMs: a single-token step of the sampling chain has 4 row tiles): narrower tiles occupy
    // more SMs and halve each CTA's K loop, which is what bounds these launch-latency-sized kernels.  Long-K weight
    // gradients (plain fp32 output) keep the wide tile: they fill the SMs through split-K instead.
    const bool splittable = dtype_c == TGAN_F32 && (flags & ~(TGAN_EPI_ACCUM | TGAN_EPI_AUX_F32)) == 0;
    if (ceil_div(M, BM) * ceil_div(N, 256) * 2 <= sm_count() && (ceil_div(K, BK) < 16 || !splittable)) BN = 128;
    CUtensorMap tmA, tmB;
    int rc;
    if (!transA) rc = tc::make_tmap_2d(&tmA, A, (uint64_t)M, (uint64_t)K, (uint64_t)lda, BM, BK);
    else rc = tc::make_tmap_2d(&tmA, A, (uint64_t)K, (uint64_t)M, (uint64_t)lda, BK, 64);
    if (rc) return rc;
    if (transB) rc = tc::make_tmap_2d(&tmB, B, (uint64_t)N, (uint64_t)K, (uint64_t)ldb, BN, BK);
    else rc = tc::make_tmap_2d(&tmB, B, (uint64_t)K, (uint64_t)N, (uint64_t)ldb, BK, 64);
    if (rc) return rc;
    EpiParams ep;
    ep.bias = bias; ep.aux = aux; ep.ldaux = ldaux; ep.flags = flags; ep.alpha = alpha;
    ep.drop_scale = drop_p > 0.f ? 1.f / (1.f - drop_p) : 1.f;
    ep.drop_thresh = dropout_thresh(drop_p);
    ep.drop_key = dropout_key(seed, site);
    ep.aux_is_f32 = (flags & TGAN_EPI_AUX_F32) ? 1 : 0;
    if (drop_p <= 0.f || ep.drop_thresh == 0) ep.flags &= ~TGAN_EPI_DROPOUT;
    // vector epilogue: rows of C (and aux) start 16-byte aligned
    const int esz_c = dtype_c == TGAN_F32 ? 4 : 2;
    bool vec = (((uintptr_t)C & 15) == 0) && ((ldc * esz_c) % 16 == 0);
    if (flags & (TGAN_EPI_MASK_POS | TGAN_EPI_ADD_AUX)) {
        const int esz_a = ep.aux_is_f32 ? 4 : 2;
        vec = vec && (((uintptr_t)aux & 15) == 0) && ((ldaux * esz_a) % 16 == 0);
    }
    if (vec) ep.flags |= EPI_VEC;
    if ((flags & TGAN_EPI_BIAS) && (((uintptr_t)bias & 15) == 0)) ep.flags |= EPI_BIAS_VEC;
    // split-K: weight-gradient shapes (few output tiles, very long K) would leave most SMs idle.  Partial sums are
    // added into the fp32 output with red.global.add; without ACCUM the output is zeroed first.
    int splits = 1;
    {
        const int tiles = ceil_div(M, BM) * ceil_div(N, BN), nk = ceil_div(K, BK);
        const int plain = flags & ~(TGAN_EPI_ACCUM | TGAN_EPI_AUX_F32);
        if (dtype_c == TGAN_F32 && plain == 0 && tiles * 2 <= sm_count() && nk >= 16) {
            splits = sm_count() / tiles;
            if (splits > nk / 8) splits = nk / 8;
            if (splits < 1) splits = 1;
        }
        if (splits > 1) {
            if (!(flags & TGAN_EPI_ACCUM))
                TGAN_CUDA_OK(cudaMemset2DAsync(C, ldc * sizeof(float), 0, (size_t)N * sizeof(float), M, st));
            ep.flags = (ep.flags & ~TGAN_EPI_ACCUM) | EPI_ATOMIC;
        }
    }
    // C leaves through shared memory + TMA whenever the copy engine can address it: 16-byte aligned rows, and
    // accumulation only into fp32 (reduce-add)
    CUtensorMap tmC;
    memset(&tmC, 0, sizeof(tmC));
    const bool accum = (ep.flags & (TGAN_EPI_ACCUM | EPI_ATOMIC)) != 0;
    if (vec && ((int64_t)N * esz_c) % 16 == 0 && !(accum && dtype_c != TGAN_F32)) {
        rc = tc::make_tmap_2d_dt(&tmC, C, (uint64_t)M, (uint64_t)N, (uint64_t)ldc, 32, dtype_c == TGAN_F32 ? 32 : 64,
                                 dtype_c == TGAN_F32);
        if (rc) return rc;
        ep.flags |= EPI_TMA;
    }
    // fp32 accumulation without the TMA reduce path (unaligned C): atomics, so that it stays a reduction -- accumulating
    // GEMMs of concurrent streams may target the same rows (engine.py: weight gradients on side streams)
    if (!(ep.flags & EPI_TMA) && (ep.flags & TGAN_EPI_ACCUM) && dtype_c == TGAN_F32 &&
        (ep.flags & ~(TGAN_EPI_ACCUM | TGAN_EPI_AUX_F32 | EPI_VEC | EPI_BIAS_VEC)) == 0)
        ep.flags = (ep.flags & ~TGAN_EPI_ACCUM) | EPI_ATOMIC;
    // compile-time epilogue variant: whole 8-column groups, aligned bias, bf16 aux
    int epi_ct = -1;
    if ((ep.flags & EPI_TMA) && N % 8 == 0 && !ep.aux_is_f32 && (!(ep.flags & TGAN_EPI_BIAS) || (ep.flags & EPI_BIAS_VEC)))
        epi_ct = (ep.flags & (TGAN_EPI_BIAS | TGAN_EPI_RELU | TGAN_EPI_MASK_POS | TGAN_EPI_ADD_AUX | TGAN_EPI_DROPOUT)) |
                 (alpha != 1.0f ? EPI_ALPHA : 0);
    // 2-CTA pairs for the nn.Linear layout when there are enough 256 x 256 tiles to fill the 74 pairs
    if (!transA && transB && epi_ct >= 0 && splits == 1 && M >= 2048 &&
        ceil_div(M, 256) * ceil_div(N, 256) >= sm_count() / 2) {
        CUtensorMap tmA2, tmB2;
        rc = tc::make_tmap_2d(&tmA2, A, (uint64_t)M, (uint64_t)K, (uint64_t)lda, 128, BK);
        if (rc) return rc;
        rc = tc::make_tmap_2d(&tmB2, B, (uint64_t)N, (uint64_t)K, (uint64_t)ldb, 128, BK);
        if (rc) return rc;
        rc = dtype_c == TGAN_F32 ? launch_tc2_epi<float>(epi_ct, tmA2, tmB2, tmC, ldc, M, N, K, ep, st)
                                 : launch_tc2_epi<bf16>(epi_ct, tmA2, tmB2, tmC, ldc, M, N, K, ep, st);
        if (rc >= 0) return rc;
    }
    if (dtype_c == TGAN_F32) {
        if (BN == 256) return launch_layout<256, float>(transA, transB, epi_ct, tmA, tmB, tmC, C, ldc, M, N, K, splits, ep, st);
        return launch_layout<128, float>(transA, transB, epi_ct, tmA, tmB, tmC, C, ldc, M, N, K, splits, ep, st);
    }
    if (BN == 256) return launch_layout<256, bf16>(transA, transB, epi_ct, tmA, tmB, tmC, C, ldc, M, N, K, splits, ep, st);
    return launch_layout<128, bf16>(transA, transB, epi_ct, tmA, tmB, tmC, C, ldc, M, N, K, splits, ep, st);
}
