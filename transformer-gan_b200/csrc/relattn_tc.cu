// tcgen05 relative-position attention BACKWARD for sm_100a (bf16 operands, fp32 accumulation in TMEM).
// Reference: autograd of mem_transformer.py:201-244 (+ _rel_shift :133-147, mask :495-547); SURVEY.md section 9.
//
// One CTA per (b, n); requires Q <= 128 (one query tile) so dK / dV tiles are complete per CTA.  16 warps:
//   row warps   (8 of them) thread = (query row = TMEM lane, column half): warp w owns lane quarter w & 3 and the
//               32-column half w >> 2 of every 64-wide tile, so each query row is served by 2 threads.  They do
//               ONLY the per-score work: G ring, P, dS, publish.
//   drain warps (4, one per TMEM lane quarter): move the finished key-side results out of tensor memory -- dK / dV
//               tiles (scaled, bf16, staged for the TMA store) and dR chunks (red.global.add over the batch).  In
//               round 1 the row warps did this between their own phases: 37 % of their tile time (profiles/
//               r1 bwd phase log: flush_keys 1979 + flush_dr 730 of ~7250 clk) sat on the critical path.
//               The dK / dV tiles are staged in shared memory and written by the copy engine (TMA store issued by one
//               drain thread), so the 1.3 MB-strided key rows never go through the SIMT load/store pipe.
//   then one warp each: tcgen05.mma issuer; K / V tile loads (TMA); R chunks for the G product; R chunks for dqR
// Per 64-key tile t (TMEM columns in brackets):
//     S  [0]   = (q+u) K_t^T          G [64]  = (q+v) R_c^T (ring, as in the forward)     dP [128] = dO' V_t^T
//   row threads:  P = exp2(S2 - lse2),  dS = P (keep(dP) - delta),  P~ = keep(P)   -> bf16 tiles in shared memory;
//                 dS is also scattered into a bf16 ring at the INVERSE shift (column p = j + Q-1-i).  The ring is laid
//                 out as un-swizzled 8 x 16-byte core matrices ([i / 8][p][i % 8]), so a finished 64-position chunk IS
//                 a valid tcgen05 operand both as dG (MN-major, M = i) and as dG^T (K-major, M = p): no extraction pass
//     dV_t [384] = P~^T dO'    dK_t [320] = dS^T (q+u)     dqK [192] += dS K_t            (after the tiles are written)
//     dqR [256] += dG_c R_c    dR_c [448] = dG_c^T (q+v)   where dG_c = chunk c of the dS ring (complete after tile c)
// The key-side results of tile t and the dR chunk t are drained one tile later (just before tile t+1 publishes its
// own tiles), so the row warps never sit idle behind the dV / dK / dqK / dqR / dR MMAs.
// dO' = dO / (1 - p_drop) is formed once while staging, so neither P~ nor dP needs a per-element dropout scale;
// the 1/sqrt(d_head) factor of dS is applied when dq / dK / dR / du / dvb leave the CTA.
// dR chunks are reduced over the batch with red.global.add.v4.f32; du / dvb are the column sums of dqK / dqR.
#include <cuda_fp16.h>

#include "tc_common.cuh"

namespace {
using namespace tc;

constexpr int HS = TGAN_HS;  // 64
constexpr int BQ = 128;      // query rows per CTA
constexpr int BJ = 64;       // keys per tile
constexpr int RING_COLS = 192;
constexpr int SPLIT = 2;   // threads per query row: each owns CW columns of every 64-wide tile
constexpr int CW = BJ / SPLIT;
static_assert(CW == 32, "a thread's column slice is one tmem_ld32");
constexpr int ROW_WARPS = 4 * SPLIT;
constexpr int DRAIN0 = ROW_WARPS;          // drain warps DRAIN0 .. DRAIN0 + 3 (DRAIN0 % 4 == 0: warp w reads lane quarter w & 3)
constexpr int MMA_WARP = ROW_WARPS + 4;
constexpr int NTHREADS = 32 * (ROW_WARPS + 8);

constexpr int B_OFF_QU = 0;
constexpr int B_OFF_QV = B_OFF_QU + 16384;
constexpr int B_OFF_DO = B_OFF_QV + 16384;
constexpr int B_OFF_K = B_OFF_DO + 16384;    // 2 stages x 8 KB
constexpr int B_OFF_V = B_OFF_K + 2 * 8192;  // 1 stage
constexpr int B_OFF_RG = B_OFF_V + 8192;     // R chunks for G: 2 stages x 8 KB
constexpr int B_OFF_RD = B_OFF_RG + 2 * 8192; // R chunk for dqR: 1 stage
constexpr int B_OFF_PT = B_OFF_RD + 8192;    // P~ tile
constexpr int B_OFF_DS = B_OFF_PT + 16384;
constexpr int B_OFF_GRING = B_OFF_DS + 16384;                 // fp16 [192][128]
constexpr int B_OFF_DRING = B_OFF_GRING + RING_COLS * BQ * 2; // bf16 [16 row groups][192 positions][8 rows]
constexpr int DR_GROUP = RING_COLS * 16 + 32;                 // byte stride between 8-row groups (+32: bank spread)
constexpr int DRING_BYTES = 16 * DR_GROUP;
constexpr int B_OFF_BAR = B_OFF_DRING + DRING_BYTES;
constexpr int B_NUM_BARS = 28;
constexpr int BWD_SMEM = B_OFF_BAR + B_NUM_BARS * 8 + 16 + 1024;
static_assert(BWD_SMEM <= 232448, "shared memory budget");
constexpr int TB_S = 0, TB_G = 64, TB_DP = 128, TB_DQK = 192, TB_DQR = 256, TB_DK = 320, TB_DV = 384, TB_DR = 448;
constexpr int TM_COLS = 512;

struct BwdParams {
    const bf16* q; int64_t ldq;
    const bf16* out; const bf16* dout; int64_t ldo;
    const float* lse;
    const float* u; const float* vb;
    const uint8_t* reset;
    bf16* dq; bf16* dk; bf16* dv; int64_t lddkv;
    float* dr; int64_t lddr;
    float* du; float* dvb;
    int B, N, Q, M, K, msl, same_length;
    float scale, scale_log2;
    float drop_scale; uint32_t drop_thresh; uint32_t drop_key;
};

__device__ __forceinline__ void red_add_v4(float* addr, float a, float b, float c, float d) {
    asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(addr), "f"(a), "f"(b), "f"(c), "f"(d) : "memory");
}
// the two warps serving one lane quarter (w, w + 4) meet on named barrier 1 + quarter
__device__ __forceinline__ void pair_sync(int quarter) {
    asm volatile("bar.sync %0, %1;" ::"r"(quarter + 1), "n"(32 * SPLIT) : "memory");
}

__global__ void __launch_bounds__(NTHREADS, 1)
relattn_bwd_tc_kernel(const __grid_constant__ CUtensorMap tmK, const __grid_constant__ CUtensorMap tmV,
                      const __grid_constant__ CUtensorMap tmR, const __grid_constant__ CUtensorMap tmDK,
                      const __grid_constant__ CUtensorMap tmDV, BwdParams p) {
    extern __shared__ uint8_t smem_raw[];
    const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
    uint8_t* gbase = smem_raw + (base - smem_u32(smem_raw));
    const uint32_t sQu = base + B_OFF_QU, sQv = base + B_OFF_QV, sDO = base + B_OFF_DO, sK = base + B_OFF_K,
                   sV = base + B_OFF_V, sRG = base + B_OFF_RG, sRD = base + B_OFF_RD, sPT = base + B_OFF_PT,
                   sDS = base + B_OFF_DS;
    __half* gring = reinterpret_cast<__half*>(gbase + B_OFF_GRING);
    const uint32_t sDR = base + B_OFF_DRING;
    const uint32_t bar0 = base + B_OFF_BAR;
    const uint32_t k_full = bar0, k_empty = k_full + 16, v_full = k_empty + 16, v_empty = v_full + 8,
                   rg_full = v_empty + 8, rg_empty = rg_full + 16, rd_full = rg_empty + 16, rd_empty = rd_full + 8,
                   s_full = rd_empty + 8, s_empty = s_full + 8, dp_full = s_empty + 8, dp_empty = dp_full + 8,
                   g_full = dp_empty + 8, g_empty = g_full + 8, p_full = g_empty + 8, kdone = p_full + 8,
                   dr_empty = kdone + 8, rdone = dr_empty + 8, ks_full = rdone + 8, ks_empty = ks_full + 8,
                   kd_empty = ks_empty + 8,  // the drain warps have read dK / dV of a tile out of tensor memory
                   fin = kd_empty + 8;       // single use: every tcgen05 op of the CTA has completed
    const uint32_t sTmemPtr = fin + 8;
    volatile uint32_t* tmem_ptr_gen = reinterpret_cast<volatile uint32_t*>(gbase + (sTmemPtr - base));

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int bn = blockIdx.x, b = bn / p.N, n = bn % p.N;
    const int rows_here = p.Q;  // Q <= 128, single query tile (i0 = 0)
    const bool reset_b = p.reset && p.reset[b];
    int jlo = 0, jhi = min(p.K - 1, rows_here - 1 + p.M);
    if (p.same_length) jlo = max(0, -p.msl + 1);
    if (reset_b) jlo = max(jlo, p.M);
    const int t_lo = jlo / BJ, t_hi = jhi / BJ;
    const int nt = t_hi - t_lo + 1;
    const int nc = nt + 2;
    const int P0 = p.Q - 1 - (BQ - 1) + BJ * t_lo;

    if (threadIdx.x == 0) {
        for (int s = 0; s < 2; ++s) {
            mbar_init(k_full + 8 * s, 1); mbar_init(k_empty + 8 * s, 1);
            mbar_init(rg_full + 8 * s, 1); mbar_init(rg_empty + 8 * s, 1);
        }
        mbar_init(v_full, 1); mbar_init(v_empty, 1);
        mbar_init(rd_full, 1); mbar_init(rd_empty, 1);
        mbar_init(s_full, 1); mbar_init(s_empty, ROW_WARPS);
        mbar_init(dp_full, 1); mbar_init(dp_empty, ROW_WARPS);
        mbar_init(g_full, 1); mbar_init(g_empty, ROW_WARPS);
        mbar_init(p_full, ROW_WARPS); mbar_init(kdone, 1); mbar_init(dr_empty, 4); mbar_init(rdone, 1);
        mbar_init(ks_full, 1); mbar_init(ks_empty, 1); mbar_init(kd_empty, 4); mbar_init(fin, 1);
        fence_barrier_init();
    }
    if (warp == MMA_WARP) tmem_alloc(sTmemPtr, TM_COLS);

    // row-thread identity
    const int quarter = warp & 3, part = (warp >> 2) & (SPLIT - 1);
    const int ii = 32 * quarter + lane;
    float delta = 0.f, lse2 = 0.f;
    // row ii's SPLIT partial sums of delta meet inside the row's own 128 bytes of the (still unused) P~ tile
    float* delta_x = reinterpret_cast<float*>(gbase + B_OFF_PT + (ii >> 3) * 1024 + (ii & 7) * 128);
    if (warp < ROW_WARPS) {
        const bool live = ii < rows_here;
        const int64_t row = (int64_t)ii * p.B + b;
        const bf16* qrow = p.q + row * p.ldq + n * HS;
        const bf16* orow = p.out + row * p.ldo + n * HS;
        const bf16* grow = p.dout + row * p.ldo + n * HS;
#pragma unroll
        for (int cc = 0; cc < HS / 8 / SPLIT; ++cc) {  // this thread stages (and sums delta over) its CW columns of the row
            const int c = part * (HS / 8 / SPLIT) + cc;
            float o[8], g[8];
            if (live) { load8(orow + 8 * c, o); load8(grow + 8 * c, g); }
#pragma unroll
            for (int t = 0; t < 8; ++t) delta += live ? g[t] * o[t] : 0.f;
            {
                float x[8], a[8], bb[8], uu[8], vv[8];
                if (live) load8(qrow + 8 * c, x);
                load8(p.u + n * HS + 8 * c, uu);
                load8(p.vb + n * HS + 8 * c, vv);
#pragma unroll
                for (int t = 0; t < 8; ++t) {
                    a[t] = live ? x[t] + uu[t] : 0.f;
                    bb[t] = live ? x[t] + vv[t] : 0.f;
                    g[t] = live ? g[t] * p.drop_scale : 0.f;
                }
                store8(reinterpret_cast<bf16*>(gbase + B_OFF_QU + sw128_off(ii, c)), a);
                store8(reinterpret_cast<bf16*>(gbase + B_OFF_QV + sw128_off(ii, c)), bb);
                store8(reinterpret_cast<bf16*>(gbase + B_OFF_DO + sw128_off(ii, c)), g);
            }
        }
        delta_x[part] = delta;
        lse2 = live ? p.lse[(int64_t)bn * p.Q + ii] * 1.4426950408889634f : 0.f;
        // zero the dS ring
        for (int o = threadIdx.x * 16; o < DRING_BYTES; o += 32 * ROW_WARPS * 16)
            *reinterpret_cast<uint4*>(gbase + B_OFF_DRING + o) = make_uint4(0, 0, 0, 0);
        // keys this (b, n) never attends to get zero gradients
        for (int j = threadIdx.x; j < p.K; j += 32 * ROW_WARPS) {
            if (j >= t_lo * BJ && j < (t_hi + 1) * BJ) continue;
            uint4 z = make_uint4(0, 0, 0, 0);
            uint4* dkr = reinterpret_cast<uint4*>(p.dk + ((int64_t)j * p.B + b) * p.lddkv + n * HS);
            uint4* dvr = reinterpret_cast<uint4*>(p.dv + ((int64_t)j * p.B + b) * p.lddkv + n * HS);
#pragma unroll
            for (int c = 0; c < 8; ++c) { dkr[c] = z; dvr[c] = z; }
        }
        fence_proxy_async_smem();
    }
    tcgen05_fence_before();
    __syncthreads();
    tcgen05_fence_after();
    const uint32_t tmem_base = *tmem_ptr_gen;
    if (warp < ROW_WARPS) {
        delta = 0.f;
#pragma unroll
        for (int t = 0; t < SPLIT; ++t) delta += delta_x[t];
    }

    if (warp == MMA_WARP + 1) {
        // =========================== K / V producer ===========================
        if (lane == 0) {
            for (int tt = 0; tt < nt; ++tt) {
                const int st = tt & 1;
                mbar_wait(k_empty + 8 * st, ((tt >> 1) & 1) ^ 1);
                mbar_expect_tx(k_full + 8 * st, 8192);
                tma_load_3d(sK + st * 8192, &tmK, k_full + 8 * st, n * HS, b, (t_lo + tt) * BJ);
                mbar_wait(v_empty, (tt & 1) ^ 1);
                mbar_expect_tx(v_full, 8192);
                tma_load_3d(sV, &tmV, v_full, n * HS, b, (t_lo + tt) * BJ);
            }
        }
    } else if (warp == MMA_WARP + 2) {
        // =========================== R chunks feeding G = (q+v) R^T ===========================
        if (lane == 0) {
            for (int cc = 0; cc < nc; ++cc) {
                const int st = cc & 1;
                mbar_wait(rg_empty + 8 * st, ((cc >> 1) & 1) ^ 1);
                mbar_expect_tx(rg_full + 8 * st, 8192);
                tma_load_2d(sRG + st * 8192, &tmR, rg_full + 8 * st, n * HS, P0 + BJ * cc);
            }
        }
    } else if (warp == MMA_WARP + 3) {
        // =========================== R chunks feeding dqR += dG R ===========================
        if (lane == 0) {
            for (int cc = 0; cc < nc; ++cc) {
                mbar_wait(rd_empty, (cc & 1) ^ 1);
                mbar_expect_tx(rd_full, 8192);
                tma_load_2d(sRD, &tmR, rd_full, n * HS, P0 + BJ * cc);
            }
        }
    } else if (warp == MMA_WARP) {
        // =========================== MMA issuer ===========================
        // The whole warp runs the schedule (converged barrier waits); one elected lane issues the tcgen05 ops.
        // Descriptors are built once and advanced by adding to their start-address field (16-byte units).
        constexpr uint32_t id_kk = umma_idesc_bf16(128, 64, 0, 0);    // S, G, dP: A, B K-major
        constexpr uint32_t id_kn = umma_idesc_bf16(128, 64, 0, 1);    // dqK: A K-major, B MN-major
        constexpr uint32_t id_nn = umma_idesc_bf16(64, 64, 1, 1);     // dV, dK: A, B MN-major (M = 64)
        constexpr uint32_t id_nn128 = umma_idesc_bf16(128, 64, 1, 1); // dqR: A (ring chunk), B MN-major
        constexpr uint32_t id_kn64 = umma_idesc_bf16(64, 64, 0, 1);   // dR: A (ring chunk) K-major, B MN-major
        const uint64_t k_qu = umma_smem_desc(sQu, 16, 1024), k_qv = umma_smem_desc(sQv, 16, 1024),
                       k_do = umma_smem_desc(sDO, 16, 1024), k_k0 = umma_smem_desc(sK, 16, 1024),
                       k_v = umma_smem_desc(sV, 16, 1024), k_rg0 = umma_smem_desc(sRG, 16, 1024),
                       k_ds = umma_smem_desc(sDS, 16, 1024);
        const uint64_t n_pt = umma_smem_desc(sPT, 8192, 1024), n_ds = umma_smem_desc(sDS, 8192, 1024),
                       n_do = umma_smem_desc(sDO, 8192, 1024), n_qu = umma_smem_desc(sQu, 8192, 1024),
                       n_qv = umma_smem_desc(sQv, 8192, 1024), n_k0 = umma_smem_desc(sK, 8192, 1024),
                       n_rd = umma_smem_desc(sRD, 8192, 1024);
        const uint64_t ring_mn0 = umma_smem_desc_noswz(sDR, 128, DR_GROUP), ring_k0 = umma_smem_desc_noswz(sDR, DR_GROUP, 128);
        auto mma_s = [&](int tt) {
            if (tt >= nt) return;
            mbar_wait(k_full + 8 * (tt & 1), (tt >> 1) & 1);
            mbar_wait(s_empty, (tt & 1) ^ 1);
            tcgen05_fence_after();
            if (elect_one()) {
                const uint64_t dk = k_k0 + (uint64_t)(((tt & 1) * 8192) >> 4);
#pragma unroll
                for (int k = 0; k < 4; ++k) umma_bf16(tmem_base + TB_S, k_qu + 2 * k, dk + 2 * k, id_kk, k != 0);
                umma_commit(s_full);
            }
            __syncwarp();
        };
        auto mma_dp = [&](int tt) {
            if (tt >= nt) return;
            mbar_wait(v_full, tt & 1);
            mbar_wait(dp_empty, (tt & 1) ^ 1);
            tcgen05_fence_after();
            if (elect_one()) {
#pragma unroll
                for (int k = 0; k < 4; ++k) umma_bf16(tmem_base + TB_DP, k_do + 2 * k, k_v + 2 * k, id_kk, k != 0);
                umma_commit(dp_full);
                umma_commit(v_empty);
            }
            __syncwarp();
        };
        auto mma_g = [&](int cc) {
            if (cc >= nc) return;
            mbar_wait(rg_full + 8 * (cc & 1), (cc >> 1) & 1);
            mbar_wait(g_empty, (cc & 1) ^ 1);
            tcgen05_fence_after();
            if (elect_one()) {
                const uint64_t dr = k_rg0 + (uint64_t)(((cc & 1) * 8192) >> 4);
#pragma unroll
                for (int k = 0; k < 4; ++k) umma_bf16(tmem_base + TB_G, k_qv + 2 * k, dr + 2 * k, id_kk, k != 0);
                umma_commit(g_full);
                umma_commit(rg_empty + 8 * (cc & 1));
            }
            __syncwarp();
        };
        auto mma_key = [&](int tt) {
            mbar_wait(p_full, tt & 1);
            if (tt > 0) mbar_wait(kd_empty, (tt - 1) & 1);  // dK / dV of tile tt-1 have left tensor memory
            tcgen05_fence_after();
            if (elect_one()) {
                const uint64_t dkn = n_k0 + (uint64_t)(((tt & 1) * 8192) >> 4);
#pragma unroll
                for (int k = 0; k < 8; ++k)  // dV = P~^T dO'   (contraction over the 128 query rows)
                    umma_bf16(tmem_base + TB_DV, n_pt + 128 * k, n_do + 128 * k, id_nn, k != 0);
#pragma unroll
                for (int k = 0; k < 8; ++k)  // dK = dS^T (q + u)
                    umma_bf16(tmem_base + TB_DK, n_ds + 128 * k, n_qu + 128 * k, id_nn, k != 0);
#pragma unroll
                for (int k = 0; k < 4; ++k)  // dqK += dS K_t   (contraction over the 64 keys)
                    umma_bf16(tmem_base + TB_DQK, k_ds + 2 * k, dkn + 128 * k, id_kn, (tt | k) != 0);
                umma_commit(kdone);
                umma_commit(k_empty + 8 * (tt & 1));
            }
            __syncwarp();
        };
        auto mma_rel = [&](int cc) {
            mbar_wait(rd_full, cc & 1);
            if (cc > 0) mbar_wait(dr_empty, (cc - 1) & 1);  // the row warps have drained dR of chunk cc-1
            tcgen05_fence_after();
            if (elect_one()) {
                const uint32_t cboff = ((cc % 3) * (BJ * 16)) >> 4;  // chunk cc = ring positions 64*(cc%3) .. +63
#pragma unroll
                for (int k = 0; k < 4; ++k)  // dqR += dG_c R_c   (A = dG: M = i, MN-major, un-swizzled ring chunk)
                    umma_bf16(tmem_base + TB_DQR, ring_mn0 + cboff + 16 * k, n_rd + 128 * k, id_nn128, (cc | k) != 0);
#pragma unroll
                for (int k = 0; k < 8; ++k)  // dR_c = dG_c^T (q + v)   (A = dG^T: M = p, K-major, same chunk)
                    umma_bf16(tmem_base + TB_DR, ring_k0 + cboff + ((2 * DR_GROUP) >> 4) * k, n_qv + 128 * k, id_kn64, k != 0);
                umma_commit(rdone);
                umma_commit(rd_empty);
            }
            __syncwarp();
        };
        mma_s(0); mma_dp(0); mma_g(0); mma_g(1); mma_g(2);
        for (int tt = 0; tt < nt; ++tt) {
            mma_g(tt + 3);       // needs only the previous chunk pulled
            mma_s(tt + 1);       // issued BEFORE the long key / rel MMAs of tile tt so the next tile never waits
            mma_dp(tt + 1);
            mma_key(tt);
            mma_rel(tt);
        }
        for (int cc = nt; cc < nc; ++cc) mma_rel(cc);
        if (elect_one()) umma_commit(fin);
        __syncwarp();
    } else if (warp >= DRAIN0) {
        // =========================== drain warps: key-side results out of tensor memory ===========================
        // dK / dV of tile tk and dR of chunk cc sit in TMEM in the M = 64 layout: row r = 16 * quarter + lane, lanes 0..15.
        const int dq_ = warp & 3;
        const uint32_t lane_off = (uint32_t)(32 * dq_) << 16;
        const int r = 16 * dq_ + lane;
        auto flush_dr = [&](int cc) {
            mbar_wait(rdone, cc & 1);
            tcgen05_fence_after();
            uint32_t v[64];
            tmem_ld32(tmem_base + TB_DR + lane_off, v);
            tmem_ld32(tmem_base + TB_DR + 32 + lane_off, v + 32);
            tmem_ld_wait();
            tcgen05_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(dr_empty);
            const int pr = P0 + BJ * cc + r;
            if (lane < 16 && pr >= 0 && pr < p.K) {
                float* dst = p.dr + (int64_t)pr * p.lddr + n * HS;
#pragma unroll
                for (int c = 0; c < 16; ++c)
                    red_add_v4(dst + 4 * c, __uint_as_float(v[4 * c]) * p.scale, __uint_as_float(v[4 * c + 1]) * p.scale,
                               __uint_as_float(v[4 * c + 2]) * p.scale, __uint_as_float(v[4 * c + 3]) * p.scale);
            }
        };
        // -> bf16 tiles staged in the P~ buffer (free between the key MMAs of tile tk and the publication of tile tk+1),
        // in the swizzled layout the TMA store expects; the store warp writes them out
        auto stage_keys = [&](int tk) {
            mbar_wait(kdone, tk & 1);
            tcgen05_fence_after();
#pragma unroll
            for (int m = 0; m < 2; ++m) {  // m = 0: dK (scaled), m = 1: dV
                uint32_t a[64];
                tmem_ld32(tmem_base + (m ? TB_DV : TB_DK) + lane_off, a);
                tmem_ld32(tmem_base + (m ? TB_DV : TB_DK) + 32 + lane_off, a + 32);
                tmem_ld_wait();
                const float mul = m ? 1.f : p.scale;
                if (lane < 16) {
#pragma unroll
                    for (int c = 0; c < 8; ++c) {
                        float f[8];
#pragma unroll
                        for (int t = 0; t < 8; ++t) f[t] = __uint_as_float(a[8 * c + t]) * mul;
                        store8(reinterpret_cast<bf16*>(gbase + B_OFF_PT + 8192 * m + sw128_off(r, c)), f);
                    }
                }
            }
            tcgen05_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(kd_empty);  // the next tile's key MMAs may overwrite dK / dV
            fence_proxy_async_smem();
            asm volatile("bar.sync 5, 128;" ::: "memory");  // all four drain warps have staged their 16 key rows
            if (warp == DRAIN0 && lane == 0) {
                tma_store_3d(&tmDK, sPT, n * HS, b, (t_lo + tk) * BJ);
                tma_store_3d(&tmDV, sPT + 8192, n * HS, b, (t_lo + tk) * BJ);
                tma_store_commit();
                tma_store_wait_read();
                mbar_arrive(ks_empty);  // the P~ buffer may be overwritten (tile tk+1's publication)
            }
            __syncwarp();
        };
        for (int tt = 0; tt < nt; ++tt) {
            stage_keys(tt);
            flush_dr(tt);
        }
        for (int cc = nt; cc < nc; ++cc) flush_dr(cc);
        if (warp == DRAIN0 && lane == 0) tma_store_wait_all();
    } else {
        // =========================== row warps ===========================
        const bool live = ii < rows_here;
        const uint32_t lane_off = (uint32_t)(32 * quarter) << 16;
        const int hc = CW * part;  // first column of this thread's slice
        const uint32_t rowkey = attn_drop_rowkey(step_fold(p.drop_key), (uint32_t)(bn * p.Q + ii));
        const uint32_t th_hi = p.drop_thresh << 16;
        int consumed = 0;
        uint8_t* drow = gbase + B_OFF_DRING + (ii >> 3) * DR_GROUP + (ii & 7) * 2;  // ring entry (p, ii) at drow + 16 p
#pragma unroll 1
        for (int tt = 0; tt < nt; ++tt) {
            // 1. new G chunks (tile tt reads chunks tt .. tt+2): this thread converts its CW-column slice.  The ring third
            //    being overwritten was last read in tile tt-1, which both threads of the row finished before pair sync B.
            while (consumed <= tt + 2 && consumed < nc) {
                mbar_wait(g_full, consumed & 1);
                tcgen05_fence_after();
                uint32_t g[CW];
                tmem_ld32(tmem_base + TB_G + hc + lane_off, g);
                tmem_ld_wait();
                tcgen05_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(g_empty);
                __half* dst = gring + ((consumed % 3) * BJ + hc) * BQ + ii;
#pragma unroll
                for (int c = 0; c < CW; ++c) dst[c * BQ] = __float2half_rn(__uint_as_float(g[c]));
                ++consumed;
            }
            pair_sync(quarter);  // A: both halves of the new chunk are in the ring
            const int j0 = (t_lo + tt) * BJ;
            const int start = (BQ - 1 - ii + BJ * tt + hc) % RING_COLS;  // ring column of this thread's jj = 0
            const int wrap = RING_COLS - start;                         // first jj that wraps around
            const __half* g0 = gring + start * BQ + ii;
            const __half* g1 = g0 - RING_COLS * BQ;
            // 2. P = exp2((S + G) * scale * log2e - lse2)
            float pr[CW];
            {
                mbar_wait(s_full, tt & 1);
                tcgen05_fence_after();
                uint32_t sr[CW];
                tmem_ld32(tmem_base + TB_S + hc + lane_off, sr);
                tmem_ld_wait();
                tcgen05_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(s_empty);
                const bool interior = rows_here == BQ && j0 + BJ - 1 <= p.M && (!p.same_length || BQ - p.msl - j0 <= 0) &&
                                      (!reset_b || p.M <= j0);
                if (interior) {
#pragma unroll
                    for (int jj = 0; jj < CW; ++jj) {
                        const float gv = __half2float((jj < wrap ? g0 : g1)[jj * BQ]);
                        pr[jj] = fast_exp2(fmaf(__uint_as_float(sr[jj]) + gv, p.scale_log2, -lse2));
                    }
                } else {
                    int lim_hi = live ? (ii + p.M - j0 - hc) : -1;
                    int lim_lo = 0;
                    if (p.same_length) lim_lo = max(lim_lo, ii - p.msl + 1 - j0 - hc);
                    if (reset_b) lim_lo = max(lim_lo, p.M - j0 - hc);
                    lim_hi = min(lim_hi, p.K - 1 - j0 - hc);
#pragma unroll
                    for (int jj = 0; jj < CW; ++jj) {
                        const float gv = __half2float((jj < wrap ? g0 : g1)[jj * BQ]);
                        const float e = fast_exp2(fmaf(__uint_as_float(sr[jj]) + gv, p.scale_log2, -lse2));
                        pr[jj] = (jj >= lim_lo && jj <= lim_hi) ? e : 0.f;
                    }
                }
            }
            pair_sync(quarter);  // B: both threads of the row are done reading the G ring for this tile
            // 3. dP
            mbar_wait(dp_full, tt & 1);
            tcgen05_fence_after();
            uint32_t dpr[CW];
            tmem_ld32(tmem_base + TB_DP + hc + lane_off, dpr);
            tmem_ld_wait();
            tcgen05_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(dp_empty);
            // 4. P~ = keep(P), dS = P (keep(dP) - delta), packed to bf16 pairs in registers
            uint32_t ptw[CW / 2], dsw[CW / 2];
            {
                const uint32_t rk_tile = rowkey + (uint32_t)((j0 + hc) >> 1) * 0x85EBCA77u;
#pragma unroll
                for (int c = 0; c < CW / 2; ++c) {
                    float p0 = pr[2 * c], p1 = pr[2 * c + 1];
                    float dp0 = __uint_as_float(dpr[2 * c]), dp1 = __uint_as_float(dpr[2 * c + 1]);
                    float pt0 = p0, pt1 = p1;
                    if (p.drop_thresh) {
                        const uint32_t h = attn_mixlite(rk_tile + (uint32_t)c * 0x85EBCA77u);
                        const bool k0 = (h << 16) >= th_hi, k1 = h >= th_hi;
                        pt0 = k0 ? p0 : 0.f; pt1 = k1 ? p1 : 0.f;
                        dp0 = k0 ? dp0 : 0.f; dp1 = k1 ? dp1 : 0.f;
                    }
                    __nv_bfloat162 a = __floats2bfloat162_rn(pt0, pt1);
                    __nv_bfloat162 d = __floats2bfloat162_rn(p0 * (dp0 - delta), p1 * (dp1 - delta));
                    ptw[c] = *reinterpret_cast<uint32_t*>(&a);
                    dsw[c] = *reinterpret_cast<uint32_t*>(&d);
                }
            }
            // 5. the ring third this tile's scatter is about to reuse must have been consumed (dqR / dR MMAs of chunk
            //    tt-1), and the P~ buffer must be free again (the drain warps staged tile tt-1's dK / dV in it and the
            //    TMA store has finished reading them)
            if (tt > 0) {
                mbar_wait(rdone, (tt - 1) & 1);
                mbar_wait(ks_empty, (tt - 1) & 1);
            }
            if (tt + 2 >= nt) {
                // chunk tt+2 is one of the two tail chunks whose upper positions are never written: clear this thread's
                // half of the ring third before anyone scatters into it
                uint8_t* z = drow + (((tt + 2) % 3) * BJ + hc) * 16;
#pragma unroll
                for (int c = 0; c < CW; ++c) *reinterpret_cast<uint16_t*>(z + 16 * c) = 0;
                pair_sync(quarter);
            }
            // 6. publish: P~ and dS tiles (swizzled K-major) + inverse-shift scatter of dS into the ring
            {
                uint8_t* d0 = drow + start * 16;
                uint8_t* d1 = d0 - RING_COLS * 16;
#pragma unroll
                for (int c = 0; c < CW / 8; ++c) {
                    *reinterpret_cast<uint4*>(gbase + B_OFF_PT + sw128_off(ii, (CW / 8) * part + c)) =
                        make_uint4(ptw[4 * c], ptw[4 * c + 1], ptw[4 * c + 2], ptw[4 * c + 3]);
                    *reinterpret_cast<uint4*>(gbase + B_OFF_DS + sw128_off(ii, (CW / 8) * part + c)) =
                        make_uint4(dsw[4 * c], dsw[4 * c + 1], dsw[4 * c + 2], dsw[4 * c + 3]);
                }
#pragma unroll
                for (int c = 0; c < CW / 2; ++c) {
                    *reinterpret_cast<uint16_t*>((2 * c < wrap ? d0 : d1) + 32 * c) = (uint16_t)(dsw[c] & 0xffffu);
                    *reinterpret_cast<uint16_t*>((2 * c + 1 < wrap ? d0 : d1) + 32 * c + 16) = (uint16_t)(dsw[c] >> 16);
                }
            }
            fence_proxy_async_smem();
            __syncwarp();
            if (lane == 0) mbar_arrive(p_full);
        }
        // dq = (dqK + dqR) / sqrt(d); du / dvb = column sums over the query rows.  `fin` is committed after the last
        // MMA (a parity wait on `rdone` would be ambiguous here: the row warps are up to three phases behind it).
        mbar_wait(fin, 0);
        tcgen05_fence_after();
        {
            uint32_t a[CW], c2[CW];
            tmem_ld32(tmem_base + TB_DQK + hc + lane_off, a);
            tmem_ld32(tmem_base + TB_DQR + hc + lane_off, c2);
            tmem_ld_wait();
            tcgen05_fence_before();
            if (live) {
                bf16* dst = p.dq + ((int64_t)ii * p.B + b) * p.ldq + n * HS + hc;
#pragma unroll
                for (int c = 0; c < CW / 8; ++c) {
                    float f[8];
#pragma unroll
                    for (int t = 0; t < 8; ++t) f[t] = (__uint_as_float(a[8 * c + t]) + __uint_as_float(c2[8 * c + t])) * p.scale;
                    store8(dst + 8 * c, f);
                }
            }
            float su = 0.f, sv = 0.f;
#pragma unroll
            for (int d = 0; d < CW; ++d) {
                const float tk = warp_sum(live ? __uint_as_float(a[d]) : 0.f);
                const float tr = warp_sum(live ? __uint_as_float(c2[d]) : 0.f);
                if (d == lane) { su = tk; sv = tr; }
            }
            if (lane < CW) {
                atomicAdd(&p.du[n * HS + hc + lane], su * p.scale);
                atomicAdd(&p.dvb[n * HS + hc + lane], sv * p.scale);
            }
        }
    }
    tcgen05_fence_before();
    __syncthreads();
    if (warp == MMA_WARP) {
        tcgen05_fence_after();
        tmem_dealloc(tmem_base, TM_COLS);
    }
}
}  // namespace

int tgan_set_step_ctr_relattn_bwd_tc(const void* p) { return tgan_set_step_ctr_local(p); }

int tgan_relattn_bwd_tc(const void* q, int64_t ldq, const void* k, const void* v, int64_t ldkv, const void* r,
                        int64_t ldr, const float* u, const float* vb, const uint8_t* reset, const void* out,
                        const void* dout, int64_t ldo, const float* lse, float* delta, void* dq, void* dk, void* dv,
                        int64_t lddkv, float* dr, int64_t lddr, float* du, float* dvb, int B, int N, int Q, int M,
                        int msl, int same_length, float scale, float drop_p, uint64_t seed, uint64_t site,
                        cudaStream_t st) {
    (void)delta;
    const int K = M + Q;
    const uintptr_t al = (uintptr_t)q | (uintptr_t)k | (uintptr_t)v | (uintptr_t)r | (uintptr_t)out | (uintptr_t)dout |
                         (uintptr_t)dq | (uintptr_t)dk | (uintptr_t)dv | (uintptr_t)dr | (uintptr_t)u | (uintptr_t)vb;
    if (!(Q >= 32 && Q <= BQ && (al & 15) == 0 && lddr % 4 == 0)) {
        tgan_set_error("tgan_relattn_bwd: shape not eligible for the tcgen05 kernel (needs 32 <= Q <= 128, 16-byte alignment)");
        return -1;
    }
    CUtensorMap tmK, tmV, tmR;
    int rc = tc::make_tmap_3d(&tmK, k, (uint64_t)N * HS, (uint64_t)B, (uint64_t)K, (uint64_t)ldkv, (uint64_t)B * ldkv, HS, 1, BJ);
    if (rc) return rc;
    rc = tc::make_tmap_3d(&tmV, v, (uint64_t)N * HS, (uint64_t)B, (uint64_t)K, (uint64_t)ldkv, (uint64_t)B * ldkv, HS, 1, BJ);
    if (rc) return rc;
    rc = tc::make_tmap_2d(&tmR, r, (uint64_t)K, (uint64_t)N * HS, (uint64_t)ldr, BJ, HS);
    if (rc) return rc;
    CUtensorMap tmDK, tmDV;
    rc = tc::make_tmap_3d(&tmDK, dk, (uint64_t)N * HS, (uint64_t)B, (uint64_t)K, (uint64_t)lddkv, (uint64_t)B * lddkv, HS, 1, BJ);
    if (rc) return rc;
    rc = tc::make_tmap_3d(&tmDV, dv, (uint64_t)N * HS, (uint64_t)B, (uint64_t)K, (uint64_t)lddkv, (uint64_t)B * lddkv, HS, 1, BJ);
    if (rc) return rc;
    BwdParams p;
    p.q = (const bf16*)q; p.ldq = ldq; p.out = (const bf16*)out; p.dout = (const bf16*)dout; p.ldo = ldo; p.lse = lse;
    p.u = u; p.vb = vb; p.reset = reset; p.dq = (bf16*)dq; p.dk = (bf16*)dk; p.dv = (bf16*)dv; p.lddkv = lddkv;
    p.dr = dr; p.lddr = lddr; p.du = du; p.dvb = dvb;
    p.B = B; p.N = N; p.Q = Q; p.M = M; p.K = K; p.msl = msl; p.same_length = same_length;
    p.scale = scale; p.scale_log2 = scale * 1.4426950408889634f;
    p.drop_scale = drop_p > 0.f ? 1.f / (1.f - drop_p) : 1.f;
    p.drop_thresh = drop_p > 0.f ? dropout_thresh16(drop_p) : 0u;
    p.drop_key = dropout_key(seed, site);
    static bool attr_set = false;
    if (!attr_set) {
        TGAN_CUDA_OK(cudaFuncSetAttribute(relattn_bwd_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, BWD_SMEM));
        attr_set = true;
    }
    TGAN_CUDA_OK(cudaMemset2DAsync(dr, lddr * sizeof(float), 0, (size_t)N * HS * sizeof(float), K, st));
    relattn_bwd_tc_kernel<<<B * N, NTHREADS, BWD_SMEM, st>>>(tmK, tmV, tmR, tmDK, tmDV, p);
    TGAN_COUNT_LAUNCH();
    TGAN_LAUNCH_OK();
    return 0;
}
