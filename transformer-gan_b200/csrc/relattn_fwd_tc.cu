// tcgen05 relative-position attention FORWARD for sm_100a (bf16 operands, fp32 accumulation in TMEM).
// Reference: mem_transformer.py:201-244 (attention core), :133-147 (_rel_shift), :495-547 (mask).
//
// One CTA per (batch b, head n, 128-row query tile); two CTAs are resident per SM (<= 113 KB shared memory,
// 256 TMEM columns each) so the softmax arithmetic of one overlaps the barrier waits of the other.  Seven warps:
//   warps 0..3  "row" warps: thread = query row = TMEM lane.  Rel-shift, mask, softmax, dropout.
//   warp  4     one thread issues every tcgen05.mma
//   warp  5     one thread issues the K / V tile loads (TMA)
//   warp  6     one thread issues the R chunk loads (TMA)
// Per 32-key tile t the tensor core produces, into TMEM,
//     S_t  = (q + u) K_t^T            [128 x 32]
//     G_c  = (q + v) R_c^T            [128 x 32]   for ONE new 32-wide chunk c = t + 4 of relative positions
//     O   += P_t V_t                  [128 x 64]   (A operand = P_t read from TMEM, never staged in shared memory)
// The relative shift  BD[i, j] = G[i, j + Q - 1 - i]  is a row-dependent column offset.  TMEM rows are thread
// private (thread = lane), so the shift goes through a thread-private ring of the last five G chunks kept in
// shared memory as ring[column][row] (bank = row: conflict-free for any per-row offset).  Every G element is
// computed exactly once.  No [Q, K] score / mask / shifted copy ever exists.
// The running output stays in TMEM; it is rescaled only when a row's maximum grows by more than 2^8 ("lazy"
// rescale), so the steady-state tile costs no accumulator traffic at all.
#include <cuda_fp16.h>

#include "tc_common.cuh"

namespace {
using namespace tc;

constexpr int HS = TGAN_HS;  // 64
constexpr int BQ = 128;      // query rows per CTA
constexpr int BJ = 32;       // keys per tile
constexpr int KV_STAGES = 3;
constexpr int R_STAGES = 2;
constexpr int NCHUNK = 5;                 // G chunks a tile can touch: (BQ + BJ - 1) / BJ rounded up
constexpr int RING_COLS = NCHUNK * BJ;    // 160
constexpr int NTHREADS = 224;

constexpr int TILE_BYTES = BJ * HS * 2;   // 4 KB: [32 rows][64 bf16], K-major SW128
constexpr int OFF_QU = 0;                                // [128][64] bf16, K-major SW128
constexpr int OFF_QV = OFF_QU + BQ * HS * 2;             // 16 KB
constexpr int OFF_KV = OFF_QV + BQ * HS * 2;             // KV_STAGES x (K tile + V tile)
constexpr int OFF_R = OFF_KV + KV_STAGES * 2 * TILE_BYTES;
constexpr int OFF_RING = OFF_R + R_STAGES * TILE_BYTES;  // [160][128] fp16 (thread-private G ring)
constexpr int OFF_BAR = OFF_RING + RING_COLS * BQ * 2;
constexpr int NUM_BARS = 2 * KV_STAGES + 2 * R_STAGES + 2 + 2 + 2 + 2 + 2 + 2;
constexpr int FWD_SMEM = OFF_BAR + NUM_BARS * 8 + 16 + 1024;
static_assert(FWD_SMEM <= 115712, "two CTAs per SM need <= 113 KB each");

// TMEM columns (256 allocated)
constexpr int TM_S = 0;     // 2 x 32
constexpr int TM_G = 64;    // 2 x 32
constexpr int TM_O = 128;   // 64
constexpr int TM_P = 192;   // 2 x 16 (bf16 pairs)
constexpr int TM_COLS = 256;

constexpr float RESCALE_THRESHOLD = 8.f;  // log2 units: P stays <= 2^8 between rescales

struct FwdParams {
    const bf16* q; int64_t ldq;
    bf16* out; int64_t ldo;
    float* lse;
    const float* u; const float* vb;
    const uint8_t* reset;
    const int32_t* key_start; int64_t key_base;  // per-sequence key floor (NULL: off)
    int B, N, Q, M, K, msl, same_length;
    float scale_log2;  // scale * log2(e)
    float drop_scale; uint32_t drop_thresh; uint32_t drop_key;
};

__global__ void __launch_bounds__(NTHREADS, 2)
relattn_fwd_tc_kernel(const __grid_constant__ CUtensorMap tmK, const __grid_constant__ CUtensorMap tmV,
                      const __grid_constant__ CUtensorMap tmR, FwdParams p) {
    extern __shared__ uint8_t smem_raw[];
    const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
    uint8_t* gbase = smem_raw + (base - smem_u32(smem_raw));
    const uint32_t sQu = base + OFF_QU, sQv = base + OFF_QV, sKV = base + OFF_KV, sR = base + OFF_R;
    __half* ring = reinterpret_cast<__half*>(gbase + OFF_RING);
    const uint32_t bar0 = base + OFF_BAR;
    // barrier map
    const uint32_t kv_full = bar0, kv_empty = kv_full + 8 * KV_STAGES, r_full = kv_empty + 8 * KV_STAGES,
                   r_empty = r_full + 8 * R_STAGES, s_full = r_empty + 8 * R_STAGES, s_empty = s_full + 16,
                   g_full = s_empty + 16, g_empty = g_full + 16, p_full = g_empty + 16, o_done = p_full + 16;
    const uint32_t sTmemPtr = o_done + 16;
    volatile uint32_t* tmem_ptr_gen = reinterpret_cast<volatile uint32_t*>(gbase + (sTmemPtr - base));
    // the key floor, parked next to the TMEM address: the row warps re-read it per tile instead of holding a register
    volatile int* floor_sm = reinterpret_cast<volatile int*>(gbase + (sTmemPtr - base) + 4);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int bn = blockIdx.y, b = bn / p.N, n = bn % p.N;
    const int i0 = blockIdx.x * BQ;
    const int rows_here = min(BQ, p.Q - i0);
    // row i masks the keys j < min(floor_b, i + M): reset and the ragged-prompt key floor (common.cuh: key_floor)
    const int floor_b = key_floor(p.reset, p.key_start, p.key_base, b, p.M, p.K);

    // key range needed by this query tile (CTA-uniform)
    int jlo = 0, jhi = min(p.K - 1, i0 + rows_here - 1 + p.M);
    if (p.same_length) jlo = max(0, i0 - p.msl + 1);
    jlo = max(jlo, min(floor_b, i0 + p.M));
    const int t_lo = jlo / BJ, t_hi = jhi / BJ;
    const int nt = t_hi - t_lo + 1;      // >= 1
    const int nc = nt + NCHUNK - 1;      // G chunks
    const int P0 = p.Q - 1 - i0 - (BQ - 1) + BJ * t_lo;  // relative position of ring column 0

    if (threadIdx.x == 0) {
        *floor_sm = floor_b;
        for (int s = 0; s < KV_STAGES; ++s) { mbar_init(kv_full + 8 * s, 1); mbar_init(kv_empty + 8 * s, 1); }
        for (int s = 0; s < R_STAGES; ++s) { mbar_init(r_full + 8 * s, 1); mbar_init(r_empty + 8 * s, 1); }
        for (int s = 0; s < 2; ++s) {
            mbar_init(s_full + 8 * s, 1); mbar_init(s_empty + 8 * s, 4);
            mbar_init(g_full + 8 * s, 1); mbar_init(g_empty + 8 * s, 4);
            mbar_init(p_full + 8 * s, 4); mbar_init(o_done + 8 * s, 1);
        }
        fence_barrier_init();
    }
    if (warp == 4) tmem_alloc(sTmemPtr, TM_COLS);

    // ---- stage (q + u), (q + vb) as swizzled K-major A operands (row warps) ----
    if (warp < 4) {
        const int ii = threadIdx.x;  // 0..127
        const bool live = ii < rows_here;
        const bf16* qrow = p.q + ((int64_t)(i0 + ii) * p.B + b) * p.ldq + n * HS;
#pragma unroll
        for (int c = 0; c < HS / 8; ++c) {
            float x[8], a[8], bb[8], uu[8], vv[8];
            if (live) load8(qrow + 8 * c, x);
            load8(p.u + n * HS + 8 * c, uu);
            load8(p.vb + n * HS + 8 * c, vv);
#pragma unroll
            for (int t = 0; t < 8; ++t) {
                a[t] = live ? x[t] + uu[t] : 0.f;
                bb[t] = live ? x[t] + vv[t] : 0.f;
            }
            store8(reinterpret_cast<bf16*>(gbase + OFF_QU + sw128_off(ii, c)), a);
            store8(reinterpret_cast<bf16*>(gbase + OFF_QV + sw128_off(ii, c)), bb);
        }
        fence_proxy_async_smem();  // generic-proxy writes -> visible to the tensor core (async proxy)
    }
    tcgen05_fence_before();
    __syncthreads();
    tcgen05_fence_after();
    const uint32_t tmem_base = *tmem_ptr_gen;

    if (warp == 5) {
        // =========================== K / V tile producer ===========================
        if (lane == 0) {
            for (int tt = 0; tt < nt; ++tt) {
                const int st = tt % KV_STAGES;
                mbar_wait(kv_empty + 8 * st, ((tt / KV_STAGES) & 1) ^ 1);
                mbar_expect_tx(kv_full + 8 * st, 2 * TILE_BYTES);
                const uint32_t dst = sKV + st * (2 * TILE_BYTES);
                tma_load_3d(dst, &tmK, kv_full + 8 * st, n * HS, b, (t_lo + tt) * BJ);
                tma_load_3d(dst + TILE_BYTES, &tmV, kv_full + 8 * st, n * HS, b, (t_lo + tt) * BJ);
            }
        }
    } else if (warp == 6) {
        // =========================== R chunk producer ===========================
        if (lane == 0) {
            for (int cc = 0; cc < nc; ++cc) {
                const int st = cc % R_STAGES;
                mbar_wait(r_empty + 8 * st, ((cc / R_STAGES) & 1) ^ 1);
                mbar_expect_tx(r_full + 8 * st, TILE_BYTES);
                tma_load_2d(sR + st * TILE_BYTES, &tmR, r_full + 8 * st, n * HS, P0 + BJ * cc);
            }
        }
    } else if (warp == 4) {
        // =========================== MMA issuer ===========================
        // The whole warp runs the schedule (converged barrier waits); one elected lane issues the tcgen05 ops.
        // Descriptors are built once and advanced by adding to their start-address field (16-byte units).
        constexpr uint32_t idesc_kk = umma_idesc_bf16(BQ, BJ, 0, 0);  // S, G: A, B K-major, N = 32
        constexpr uint32_t idesc_pv = umma_idesc_bf16(BQ, HS, 0, 1);  // O: A from TMEM, B (= V tile [keys][d]) MN-major
        const uint64_t d_qu = umma_smem_desc(sQu, 16, 1024), d_qv = umma_smem_desc(sQv, 16, 1024);
        const uint64_t d_k0 = umma_smem_desc(sKV, 16, 1024), d_v0 = umma_smem_desc(sKV + TILE_BYTES, 8192, 1024);
        const uint64_t d_r0 = umma_smem_desc(sR, 16, 1024);
        auto mma_s = [&](int tt) {
            if (tt >= nt) return;
            const int st = tt % KV_STAGES;
            mbar_wait(kv_full + 8 * st, (tt / KV_STAGES) & 1);
            mbar_wait(s_empty + 8 * (tt & 1), ((tt >> 1) & 1) ^ 1);
            tcgen05_fence_after();
            if (elect_one()) {
                const uint64_t dk = d_k0 + (uint64_t)((st * 2 * TILE_BYTES) >> 4);
#pragma unroll
                for (int k = 0; k < HS / 16; ++k)
                    umma_bf16(tmem_base + TM_S + BJ * (tt & 1), d_qu + 2 * k, dk + 2 * k, idesc_kk, k != 0);
                umma_commit(s_full + 8 * (tt & 1));
            }
            __syncwarp();
        };
        auto mma_g = [&](int cc) {
            if (cc >= nc) return;
            const int st = cc % R_STAGES;
            mbar_wait(r_full + 8 * st, (cc / R_STAGES) & 1);
            mbar_wait(g_empty + 8 * (cc & 1), ((cc >> 1) & 1) ^ 1);
            tcgen05_fence_after();
            if (elect_one()) {
                const uint64_t dr = d_r0 + (uint64_t)((st * TILE_BYTES) >> 4);
#pragma unroll
                for (int k = 0; k < HS / 16; ++k)
                    umma_bf16(tmem_base + TM_G + BJ * (cc & 1), d_qv + 2 * k, dr + 2 * k, idesc_kk, k != 0);
                umma_commit(g_full + 8 * (cc & 1));
                umma_commit(r_empty + 8 * st);
            }
            __syncwarp();
        };
        auto mma_pv = [&](int tt) {
            const int st = tt % KV_STAGES;
            mbar_wait(p_full + 8 * (tt & 1), (tt >> 1) & 1);
            tcgen05_fence_after();
            if (elect_one()) {
                const uint64_t dv = d_v0 + (uint64_t)((st * 2 * TILE_BYTES) >> 4);
#pragma unroll
                for (int k = 0; k < BJ / 16; ++k)
                    umma_bf16_ts(tmem_base + TM_O, tmem_base + TM_P + 16 * (tt & 1) + 8 * k, dv + (2048 >> 4) * k, idesc_pv,
                                 (tt | k) != 0);
                umma_commit(o_done + 8 * (tt & 1));
                umma_commit(kv_empty + 8 * st);
            }
            __syncwarp();
        };
        for (int cc = 0; cc < NCHUNK; ++cc) mma_g(cc);
        mma_s(0);
        for (int tt = 0; tt < nt; ++tt) {
            mma_g(tt + NCHUNK);
            mma_s(tt + 1);
            mma_pv(tt);
        }
    } else {
        // =========================== row warps: rel-shift / softmax / dropout ===========================
        const int ii = threadIdx.x;
        const int i = i0 + ii;
        const bool live = ii < rows_here;
        const uint32_t lane_off = (uint32_t)(32 * warp) << 16;
        float m_ref = -INFINITY, l = 0.f;
        const uint32_t rowkey = attn_drop_rowkey(step_fold(p.drop_key), (uint32_t)(bn * p.Q + i));
        const float c_log2 = p.scale_log2;
        // thread-private ring row: ring[col * BQ + ii]
        auto pull = [&](int cc) {
            if (cc >= nc) return;
            const int st = cc & 1;
            mbar_wait(g_full + 8 * st, (cc >> 1) & 1);
            tcgen05_fence_after();
            uint32_t g[32];
            tmem_ld32(tmem_base + TM_G + BJ * st + lane_off, g);
            tmem_ld_wait();
            tcgen05_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(g_empty + 8 * st);
            __half* dst = ring + (cc % NCHUNK) * (BJ * BQ) + ii;
#pragma unroll
            for (int c = 0; c < BJ; ++c) dst[c * BQ] = __float2half_rn(__uint_as_float(g[c]));
        };
        for (int cc = 0; cc < NCHUNK - 1; ++cc) pull(cc);
#pragma unroll 1
        for (int tt = 0; tt < nt; ++tt) {
            // 1. the one new G chunk this tile needs
            pull(tt + NCHUNK - 1);
            // 2. content scores
            mbar_wait(s_full + 8 * (tt & 1), (tt >> 1) & 1);
            tcgen05_fence_after();
            uint32_t sr[32];
            tmem_ld32(tmem_base + TM_S + BJ * (tt & 1) + lane_off, sr);
            tmem_ld_wait();
            tcgen05_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(s_empty + 8 * (tt & 1));
            // 3. add the shifted position scores, mask, tile maximum
            const int j0 = (t_lo + tt) * BJ;
            const int start = (BQ - 1 - ii + BJ * tt) % RING_COLS;  // ring column of jj = 0
            const int wrap = RING_COLS - start;                      // first jj that wraps around the ring
            const __half* g0 = ring + start * BQ + ii;               // element jj sits at g0[jj * BQ] before the wrap,
            const __half* g1 = g0 - RING_COLS * BQ;                  // at g1[jj * BQ] after it: one select, no index math
            float x[32];
            float mx = -INFINITY;
            // CTA-uniform: a tile strictly inside every row's [lower, causal] window needs no per-element mask
            const bool interior = rows_here == BQ && j0 + BJ - 1 <= i0 + p.M &&
                                  (!p.same_length || i0 + BQ - p.msl - j0 <= 0) && *floor_sm <= j0;
            if (interior) {
#pragma unroll
                for (int jj = 0; jj < BJ; ++jj) {
                    x[jj] = __uint_as_float(sr[jj]) + __half2float((jj < wrap ? g0 : g1)[jj * BQ]);
                    mx = fmaxf(mx, x[jj]);
                }
            } else {
                int lim_hi = live ? (i + p.M - j0) : -1;  // jj <= lim_hi  (causal + memory)
                int lim_lo = 0;                            // jj >= lim_lo
                if (p.same_length) lim_lo = max(lim_lo, i - p.msl + 1 - j0);
                lim_lo = max(lim_lo, min(*floor_sm, i + p.M) - j0);
                lim_hi = min(lim_hi, p.K - 1 - j0);
#pragma unroll
                for (int jj = 0; jj < BJ; ++jj) {
                    float v = __uint_as_float(sr[jj]) + __half2float((jj < wrap ? g0 : g1)[jj * BQ]);
                    x[jj] = (jj >= lim_lo && jj <= lim_hi) ? v : -INFINITY;
                    mx = fmaxf(mx, x[jj]);
                }
            }
            // 4. lazy rescale of the TMEM-resident output (warp-collective: tcgen05.ld / st are .sync.aligned)
            const float mxs = mx * c_log2;
            const bool grow = mxs > m_ref + RESCALE_THRESHOLD;
            if (__any_sync(0xffffffffu, grow)) {
                float f = 1.f;
                if (grow) {
                    f = (m_ref == -INFINITY) ? 0.f : fast_exp2(m_ref - mxs);
                    m_ref = mxs;
                    l *= f;
                }
                if (tt > 0) {
                    mbar_wait(o_done + 8 * ((tt - 1) & 1), ((tt - 1) >> 1) & 1);  // P V of tile tt-1 has landed
                    tcgen05_fence_after();
#pragma unroll
                    for (int h = 0; h < 2; ++h) {
                        uint32_t o[32];
                        tmem_ld32(tmem_base + TM_O + 32 * h + lane_off, o);
                        tmem_ld_wait();
#pragma unroll
                        for (int d = 0; d < 32; ++d) o[d] = __float_as_uint(__uint_as_float(o[d]) * f);
                        tmem_st32(tmem_base + TM_O + 32 * h + lane_off, o);
                    }
                    tmem_st_wait();
                }
            }
            // 5. probabilities -> (dropout) -> bf16 pairs -> TMEM (A operand of P V)
            const float m_use = (m_ref == -INFINITY) ? 0.f : m_ref;
            float lsum = 0.f;
            uint32_t pk[16];
            const uint32_t rk_tile = rowkey + (uint32_t)(j0 >> 1) * 0x85EBCA77u;
            if (p.drop_thresh) {
                const uint32_t th_hi = p.drop_thresh << 16;
#pragma unroll
                for (int c = 0; c < 16; ++c) {
                    float e0 = fast_exp2(fmaf(x[2 * c], c_log2, -m_use));
                    float e1 = fast_exp2(fmaf(x[2 * c + 1], c_log2, -m_use));
                    lsum += e0 + e1;
                    const uint32_t h = attn_mixlite(rk_tile + (uint32_t)c * 0x85EBCA77u);
                    e0 = ((h << 16) >= th_hi) ? e0 : 0.f;   // low 16 bits decide the even key
                    e1 = (h >= th_hi) ? e1 : 0.f;           // high 16 bits decide the odd key
                    __nv_bfloat162 pr = __floats2bfloat162_rn(e0, e1);
                    pk[c] = *reinterpret_cast<uint32_t*>(&pr);
                }
            } else {
#pragma unroll
                for (int c = 0; c < 16; ++c) {
                    const float e0 = fast_exp2(fmaf(x[2 * c], c_log2, -m_use));
                    const float e1 = fast_exp2(fmaf(x[2 * c + 1], c_log2, -m_use));
                    lsum += e0 + e1;
                    __nv_bfloat162 pr = __floats2bfloat162_rn(e0, e1);
                    pk[c] = *reinterpret_cast<uint32_t*>(&pr);
                }
            }
            l += lsum;
            if (tt >= 2) {  // the P buffer is free once P V of tile tt-2 has completed
                mbar_wait(o_done + 8 * (tt & 1), ((tt >> 1) & 1) ^ 1);
                tcgen05_fence_after();
            }
            tmem_st16(tmem_base + TM_P + 16 * (tt & 1) + lane_off, pk);
            tmem_st_wait();
            tcgen05_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(p_full + 8 * (tt & 1));
        }
        // epilogue: out = O * (1/(1-p)) / l
        mbar_wait(o_done + 8 * ((nt - 1) & 1), ((nt - 1) >> 1) & 1);
        tcgen05_fence_after();
        const float inv = l > 0.f ? p.drop_scale / l : 0.f;
        bf16* orow = p.out + ((int64_t)i * p.B + b) * p.ldo + n * HS;
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            uint32_t o[32];
            tmem_ld32(tmem_base + TM_O + 32 * h + lane_off, o);
            tmem_ld_wait();
            if (live) {
#pragma unroll
                for (int c = 0; c < 4; ++c) {
                    float v8[8];
#pragma unroll
                    for (int t = 0; t < 8; ++t) v8[t] = __uint_as_float(o[8 * c + t]) * inv;
                    store8(orow + 32 * h + 8 * c, v8);
                }
            }
        }
        tcgen05_fence_before();
        if (live) p.lse[(int64_t)bn * p.Q + i] = l > 0.f ? (m_ref + log2f(l)) * 0.6931471805599453f : -INFINITY;
    }
    tcgen05_fence_before();
    __syncthreads();
    if (warp == 4) {
        tcgen05_fence_after();
        tmem_dealloc(tmem_base, TM_COLS);
    }
}
}  // namespace

int tgan_set_step_ctr_relattn_fwd_tc(const void* p) { return tgan_set_step_ctr_local(p); }

int tgan_relattn_fwd_tc(const void* q, int64_t ldq, const void* k, const void* v, int64_t ldkv, const void* r,
                        int64_t ldr, const float* u, const float* vb, const uint8_t* reset, const int32_t* key_start,
                        int64_t key_base, void* out, int64_t ldo, float* lse, int B, int N, int Q, int M, int msl,
                        int same_length, float scale, float drop_p, uint64_t seed, uint64_t site, cudaStream_t st) {
    const int K = M + Q;
    const bool ok = Q >= 32 && (((uintptr_t)q | (uintptr_t)k | (uintptr_t)v | (uintptr_t)r | (uintptr_t)out |
                                 (uintptr_t)u | (uintptr_t)vb) & 15) == 0;
    if (!ok) {
        tgan_set_error("tgan_relattn_fwd: shape not eligible for the tcgen05 kernel (needs Q >= 32, 16-byte alignment)");
        return -1;
    }
    CUtensorMap tmK, tmV, tmR;
    // k / v: [K, B, N*64] with row pitch ldkv: dims (d, b, j), box (64, 1, 32)
    int rc = tc::make_tmap_3d(&tmK, k, (uint64_t)N * HS, (uint64_t)B, (uint64_t)K, (uint64_t)ldkv, (uint64_t)B * ldkv, HS, 1, BJ);
    if (rc) return rc;
    rc = tc::make_tmap_3d(&tmV, v, (uint64_t)N * HS, (uint64_t)B, (uint64_t)K, (uint64_t)ldkv, (uint64_t)B * ldkv, HS, 1, BJ);
    if (rc) return rc;
    rc = tc::make_tmap_2d(&tmR, r, (uint64_t)K, (uint64_t)N * HS, (uint64_t)ldr, BJ, HS);
    if (rc) return rc;
    FwdParams p;
    p.q = (const bf16*)q; p.ldq = ldq; p.out = (bf16*)out; p.ldo = ldo; p.lse = lse; p.u = u; p.vb = vb; p.reset = reset;
    p.key_start = key_start; p.key_base = key_base;
    p.B = B; p.N = N; p.Q = Q; p.M = M; p.K = K; p.msl = msl; p.same_length = same_length;
    p.scale_log2 = scale * 1.4426950408889634f;
    p.drop_scale = drop_p > 0.f ? 1.f / (1.f - drop_p) : 1.f;
    p.drop_thresh = drop_p > 0.f ? dropout_thresh16(drop_p) : 0u;
    p.drop_key = dropout_key(seed, site);
    static bool attr_set = false;
    if (!attr_set) {
        TGAN_CUDA_OK(cudaFuncSetAttribute(relattn_fwd_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, FWD_SMEM));
        attr_set = true;
    }
    dim3 grid(ceil_div(Q, BQ), B * N);
    relattn_fwd_tc_kernel<<<grid, NTHREADS, FWD_SMEM, st>>>(tmK, tmV, tmR, p);
    TGAN_COUNT_LAUNCH();
    TGAN_LAUNCH_OK();
    return 0;
}
