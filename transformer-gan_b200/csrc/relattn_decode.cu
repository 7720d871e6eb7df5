// Relative-position attention for single-token calls (Q = 1): every Gumbel sampling step of the GAN phase
// (transformer_gan.py:299-334 -> mem_transformer.py:602-651) and every generated token (generate.py -> :578-600).
// Reference arithmetic: mem_transformer.py:201-244 with qlen = 1; the rel-shift (:133-147) degenerates to
// BD[j] = (q + r_r_bias) . R[j], the mask (:495-547) to "all keys" (minus the memory columns of a reset row).
//
// The work per (sequence b, head n) is one query row against K <= mem_len + 1 key rows of 64 dims: ~K * 400 bytes
// streamed, ~K * 400 FMAs.  It is HBM-bound on the projected-K/V cache, so the kernels are organised around the byte
// stream, not the math:
//   * one WARP per (b, n); lane = (key group kg = lane / 8, dim chunk dc = lane % 8).  A key row (64 dims, 128 bytes in
//     bf16) is one 16-byte load per lane of an 8-lane group -> every global access is a full, coalesced 128-byte line
//     and a warp covers 4 key rows per step; the 4 key groups run independent online softmaxes that are merged once.
//   * q (+ biases) lives in 16 registers per lane; scores are reduced with three shuffles inside the 8-lane group.
//   * forward: one pass over K, R, V.  Backward (fused, replaces the three generic passes rows / keys / rel that each
//     recomputed the scores): one pass over K, R, V producing dq, dk, dv and dS; dR (a reduction over the BATCH) is a
//     second tiny kernel over the dS scratch instead of B*N*K*64 global atomics.
//   * split backward (tgan_relattn_bwd_step, used by the captured sampling chain): the pass over K, R, V produces only
//     what the dgrad chain needs (dq, dk / dv of the current position) plus warp-contiguous scratch rows (dS, P~, the
//     per-sequence bias-gradient parts); dk / dv of the detached memory rows (pure outer products of the scratch), dR
//     and the bias sums are separate kernels that the host puts on a side stream.
// Dropout masks come from the same stateless hash as every other attention kernel (common.cuh: attn_drop_keep).
#include "common.cuh"

namespace {
constexpr int HS = TGAN_HS;  // 64
constexpr int DW_MAX = 16;   // warps per CTA = heads of ONE sequence when N <= 16 (else 4 consecutive (b, n) pairs): per key row
                             // the CTA then touches N * 128 contiguous bytes of K and of V instead of isolated 128-byte lines

struct DecArgs {
    int B, N, M, K;          // Q == 1
    int jlo0;                // first key a same_length window keeps (0 otherwise)
    float scale, scale_log2, drop_scale;
    uint32_t thresh, key;
    int split;               // backward: 1 = query side only (dk / dv of the memory rows are left to relattn_dec_keys)
    const int32_t* key_start;  // forward: per-sequence key floor (common.cuh: key_floor), NULL = off
    int64_t key_base;
};

// 8 consecutive elements kept in their storage format (bf16: one 16-byte register quad) until they are consumed: the
// loads of the next key row are issued before the current row's arithmetic and cost 12 registers, not 24.
template <typename T> struct Raw8;
template <> struct Raw8<bf16> {
    uint4 v;
    __device__ __forceinline__ void ld(const bf16* p) { v = *reinterpret_cast<const uint4*>(p); }
    __device__ __forceinline__ void get(float* o) const {
        const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&v);
#pragma unroll
        for (int i = 0; i < 4; ++i) { const float2 f = __bfloat1622float2(h[i]); o[2 * i] = f.x; o[2 * i + 1] = f.y; }
    }
};
template <> struct Raw8<float> {
    float4 a, b;
    __device__ __forceinline__ void ld(const float* p) {
        a = *reinterpret_cast<const float4*>(p); b = *reinterpret_cast<const float4*>(p + 4);
    }
    __device__ __forceinline__ void get(float* o) const {
        o[0] = a.x; o[1] = a.y; o[2] = a.z; o[3] = a.w; o[4] = b.x; o[5] = b.y; o[6] = b.z; o[7] = b.w;
    }
};

// Per-lane FIFO of key rows in shared memory, filled with cp.async: a lane copies ITS 8 elements of the k / r / v rows
// of a key and later reads back exactly those bytes, so no other thread is involved -- cp.async.wait_group is the only
// synchronisation.  PF stages deep: a warp keeps PF key quartets in flight without spending registers on them.  A warp
// walks ~K/4 iterations; with the one-deep register prefetch each one cost a full DRAM round trip (~1 us) and the
// kernel ran at 2.4 TB/s in two unbalanced waves; the FIFO hides the latency behind PF iterations.
constexpr int PF = 4;
template <typename T>
__device__ __forceinline__ void cp_row8(uint32_t dst, const T* src) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(src) : "memory");
    if constexpr (sizeof(T) == 4)
        asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst + 16), "l"(src + 4) : "memory");
}
__device__ __forceinline__ void cp_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N> __device__ __forceinline__ void cp_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

// Sum over the 8 lanes of one key group.  Called with the FULL warp converged: the key loops below run the same trip
// count on every lane (lanes whose key index is past the end are predicated off around the shuffles, not out of the
// loop).  A per-group member mask also works but costs ~4x: a lane-dependent mask sends every shuffle through the
// compiler's divergent-mask slow path (REDUX.OR + BRA.DIV loop over the distinct masks).
__device__ __forceinline__ float group8_sum(float v) {
    v += __shfl_xor_sync(0xffffffffu, v, 1);
    v += __shfl_xor_sync(0xffffffffu, v, 2);
    v += __shfl_xor_sync(0xffffffffu, v, 4);
    return v;
}

template <typename T>
__global__ void __launch_bounds__(DW_MAX * 32, 2)
relattn_dec_fwd(const T* __restrict__ q, int64_t ldq, const T* __restrict__ k, const T* __restrict__ v, int64_t ldkv,
                const T* __restrict__ r, int64_t ldr, const float* __restrict__ u, const float* __restrict__ vb,
                const uint8_t* __restrict__ reset, T* __restrict__ out, int64_t ldo, float* __restrict__ lse, DecArgs a) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int DW = blockDim.x >> 5;
    const int bn = blockIdx.x * DW + warp;
    if (bn >= a.B * a.N) return;
    const int b = bn / a.N, n = bn % a.N;
    const int kg = lane >> 3, dc = lane & 7;
    const int col = n * HS + 8 * dc;
    float qu[8], qv[8];
    {
        float x[8], uu[8], vv[8];
        load8(q + (int64_t)b * ldq + col, x);
        load8(u + col, uu);
        load8(vb + col, vv);
#pragma unroll
        for (int t = 0; t < 8; ++t) { qu[t] = x[t] + uu[t]; qv[t] = x[t] + vv[t]; }
    }
    // the key loop starts at the floor: masked rows (reset memory, the pad rows of a shorter prompt) are never streamed
    const int jlo = max(a.jlo0, min(key_floor(reset, a.key_start, a.key_base, b, a.M, a.K), a.M)), jhi = a.K - 1;
    const uint32_t rowkey = attn_drop_rowkey(step_fold(a.key), (uint32_t)bn);
    float m = -INFINITY, l = 0.f, acc[8];
#pragma unroll
    for (int t = 0; t < 8; ++t) acc[t] = 0.f;
    const T* kbase = k + (int64_t)b * ldkv + col;
    const T* vbase = v + (int64_t)b * ldkv + col;
    const int64_t kstride = (int64_t)a.B * ldkv;
    // FIFO slot (stage st, tensor x) of this thread: fifo + ((st * 3 + x) * blockDim.x + threadIdx.x) * CH
    extern __shared__ __align__(16) uint8_t fifo_raw[];
    constexpr int CH = 8 * sizeof(T);
    uint8_t* fifo = fifo_raw + threadIdx.x * CH;
    const uint32_t fifo_s = (uint32_t)__cvta_generic_to_shared(fifo);
    const uint32_t slot = blockDim.x * CH;
    // running pointers (one 64-bit add per row and step instead of an index * stride multiply chain -- the first
    // version of this loop spent 45 % of its instructions on address arithmetic)
    const int64_t kstep = 4 * kstride, rstep = 4 * ldr;
    int j = jlo + kg;
    const T* kp = kbase + j * kstride;          // prefetch cursors: row of key jp
    const T* rp = r + (int64_t)j * ldr + col;
    const T* vp = vbase + j * kstride;
    int jp = j;
    uint32_t wr = fifo_s;                       // FIFO write / read cursors (stage = 3 * slot bytes)
    const uint32_t fifo_end = fifo_s + PF * 3 * slot;
    auto issue = [&]() {
        if (jp <= jhi) {
            cp_row8(wr, kp);
            cp_row8(wr + slot, rp);
            cp_row8(wr + 2 * slot, vp);
        }
        cp_commit();  // one group per stage, empty past the end: wait_group counts stay uniform
        kp += kstep; rp += rstep; vp += kstep; jp += 4;
        wr += 3 * slot;
        if (wr == fifo_end) wr = fifo_s;
    };
#pragma unroll
    for (int st = 0; st < PF - 1; ++st) issue();
    const uint8_t* rd = fifo;
    const uint8_t* rd_end = fifo + PF * 3 * slot;
#pragma unroll 1
    for (int j0 = jlo; j0 <= jhi; j0 += 4, j += 4) {  // same trip count on all 32 lanes; j = j0 + kg
        issue();
        cp_wait<PF - 1>();  // the group of the stage at `rd` has landed
        const bool valid = j <= jhi;
        float k8[8], r8[8];
        load8(reinterpret_cast<const T*>(rd), k8);
        load8(reinterpret_cast<const T*>(rd + slot), r8);
        float s = 0.f;
#pragma unroll
        for (int t = 0; t < 8; ++t) s = fmaf(qu[t], k8[t], fmaf(qv[t], r8[t], s));
        s = group8_sum(s) * a.scale_log2;  // (stale FIFO bytes on lanes past the end: discarded below)
        if (valid) {
            const float mn = fmaxf(m, s);
            const float corr = fast_exp2(m - mn);  // m = -inf on the first key: exp2(-inf) = 0
            const float pe = fast_exp2(s - mn);
            l = fmaf(l, corr, pe);
            const float pw = (!a.thresh || attn_drop_keep(rowkey, j, a.thresh)) ? pe : 0.f;
            float v8[8];
            load8(reinterpret_cast<const T*>(rd + 2 * slot), v8);
#pragma unroll
            for (int t = 0; t < 8; ++t) acc[t] = fmaf(pw, v8[t], acc[t] * corr);
            m = mn;
        }
        rd += 3 * slot;
        if (rd == rd_end) rd = fifo;
    }
    cp_wait<0>();
    __syncwarp();  // the groups leave the loop at different trip counts: reconverge before full-warp shuffles
    // merge the 4 key groups (lanes with equal dc): max, then rescaled sums
    float m_all = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, 8));
    m_all = fmaxf(m_all, __shfl_xor_sync(0xffffffffu, m_all, 16));
    const float f = (m == -INFINITY) ? 0.f : fast_exp2(m - m_all);
    l *= f;
    l += __shfl_xor_sync(0xffffffffu, l, 8);
    l += __shfl_xor_sync(0xffffffffu, l, 16);
#pragma unroll
    for (int t = 0; t < 8; ++t) {
        float x = acc[t] * f;
        x += __shfl_xor_sync(0xffffffffu, x, 8);
        x += __shfl_xor_sync(0xffffffffu, x, 16);
        acc[t] = x;
    }
    if (kg == 0) {
        const float inv = l > 0.f ? a.drop_scale / l : 0.f;
#pragma unroll
        for (int t = 0; t < 8; ++t) acc[t] *= inv;
        store8(out + (int64_t)b * ldo + col, acc);
        if (dc == 0) lse[bn] = l > 0.f ? (m_all + log2f(l)) * 0.6931471805599453f : -INFINITY;
    }
}

// Fused backward for Q = 1.  dsbuf: fp32 [B, N, K] scratch (dS already multiplied by scale; one contiguous row per
// warp, written 16 bytes per key quartet -- the [N, K, B] layout of an earlier version meant one isolated 4-byte
// write per key).  Split mode appends P~ [B, N, K] and the per-sequence dq parts [2][B, N * 64].
template <typename T, bool SPLIT>
__global__ void __launch_bounds__(128, 5)
relattn_dec_bwd(const T* __restrict__ q, int64_t ldq, const T* __restrict__ k, const T* __restrict__ v, int64_t ldkv,
                const T* __restrict__ r, int64_t ldr, const float* __restrict__ u, const float* __restrict__ vb,
                const uint8_t* __restrict__ reset, const T* __restrict__ out, const T* __restrict__ dout, int64_t ldo,
                const float* __restrict__ lse, T* __restrict__ dq, T* __restrict__ dk, T* __restrict__ dv, int64_t lddkv,
                float* __restrict__ dsbuf, float* __restrict__ du, float* __restrict__ dvb, DecArgs a) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int DW = blockDim.x >> 5;
    const int bn = blockIdx.x * DW + warp;
    const bool active = bn < a.B * a.N;
    const int b = active ? bn / a.N : 0, n = active ? bn % a.N : 0;
    const int kg = lane >> 3, dc = lane & 7;
    const int col = n * HS + 8 * dc;
    float dqk[8], dqr[8];
#pragma unroll
    for (int t = 0; t < 8; ++t) { dqk[t] = 0.f; dqr[t] = 0.f; }
    if (active) {
        float qu[8], qv[8], g8[8];
        float delta;
        {
            float x[8], uu[8], vv[8], o8[8];
            load8(q + (int64_t)b * ldq + col, x);
            load8(u + col, uu);
            load8(vb + col, vv);
            load8(out + (int64_t)b * ldo + col, o8);
            load8(dout + (int64_t)b * ldo + col, g8);
            float d = 0.f;
#pragma unroll
            for (int t = 0; t < 8; ++t) { qu[t] = x[t] + uu[t]; qv[t] = x[t] + vv[t]; d = fmaf(g8[t], o8[t], d); }
            delta = group8_sum(d);
        }
        const float L2 = lse[bn] * 1.4426950408889634f;
        const int jlo = (reset && reset[b]) ? max(a.M, a.jlo0) : a.jlo0, jhi = a.K - 1;
        const uint32_t rowkey = attn_drop_rowkey(step_fold(a.key), (uint32_t)bn);
        const T* kbase = k + (int64_t)b * ldkv + col;
        const T* vbase = v + (int64_t)b * ldkv + col;
        T* dkbase = dk + (int64_t)b * lddkv + col;
        T* dvbase = dv + (int64_t)b * lddkv + col;
        const int64_t kstride = (int64_t)a.B * ldkv, dstride = (int64_t)a.B * lddkv;
        float* dsrow = dsbuf + (int64_t)bn * a.K;            // entry j at dsrow[j]: a warp writes its own contiguous row
        const int64_t pw_off = (int64_t)a.N * a.K * a.B;    // split mode: the dropped weights P~ follow the dS block
        // keys a reset row does not attend to: zero gradients
        for (int j = kg; j < jlo; j += 4) {
            if constexpr (!SPLIT) {
                float z[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
                store8(dkbase + j * dstride, z);
                store8(dvbase + j * dstride, z);
            }
            if (dc == 0) {
                dsrow[j] = 0.f;
                if constexpr (SPLIT) dsrow[j + pw_off] = 0.f;
            }
        }
        extern __shared__ __align__(16) uint8_t fifo_raw[];
        constexpr int CH = 8 * sizeof(T);
        uint8_t* fifo = fifo_raw + threadIdx.x * CH;
        const uint32_t fifo_s = (uint32_t)__cvta_generic_to_shared(fifo);
        const uint32_t slot = blockDim.x * CH;
        const int64_t kstep = 4 * kstride, rstep = 4 * ldr, dstep = 4 * dstride, sstep = 4;
        int j = jlo + kg;
        const T* kp = kbase + j * kstride;
        const T* rp = r + (int64_t)j * ldr + col;
        const T* vp = vbase + j * kstride;
        T* dkp = dkbase + j * dstride;
        T* dvp = dvbase + j * dstride;
        float* dsp = dsrow + j;
        int jp = j;
        uint32_t wr = fifo_s;
        const uint32_t fifo_end = fifo_s + PF * 3 * slot;
        auto issue = [&]() {
            if (jp <= jhi) {
                cp_row8(wr, kp);
                cp_row8(wr + slot, rp);
                cp_row8(wr + 2 * slot, vp);
            }
            cp_commit();
            kp += kstep; rp += rstep; vp += kstep; jp += 4;
            wr += 3 * slot;
            if (wr == fifo_end) wr = fifo_s;
        };
#pragma unroll
        for (int st = 0; st < PF - 1; ++st) issue();
        const uint8_t* rd = fifo;
        const uint8_t* rd_end = fifo + PF * 3 * slot;
#pragma unroll 1
        for (int j0 = jlo; j0 <= jhi; j0 += 4, j += 4) {  // same trip count on all 32 lanes; j = j0 + kg
            issue();
            cp_wait<PF - 1>();
            const bool valid = j <= jhi;
            float k8[8], r8[8], v8[8];
            load8(reinterpret_cast<const T*>(rd), k8);
            load8(reinterpret_cast<const T*>(rd + slot), r8);
            load8(reinterpret_cast<const T*>(rd + 2 * slot), v8);
            rd += 3 * slot;
            if (rd == rd_end) rd = fifo;
            float s = 0.f, dp = 0.f;
#pragma unroll
            for (int t = 0; t < 8; ++t) {
                s = fmaf(qu[t], k8[t], fmaf(qv[t], r8[t], s));
                dp = fmaf(g8[t], v8[t], dp);
            }
            s = group8_sum(s);
            dp = group8_sum(dp);
            if (valid) {  // (after the shuffles: every lane took part in them)
                const float pr = fast_exp2(fmaf(s, a.scale_log2, -L2));
                const bool keep = !a.thresh || attn_drop_keep(rowkey, j, a.thresh);
                const float pw = keep ? pr * a.drop_scale : 0.f;
                const float ds = pr * ((keep ? dp * a.drop_scale : 0.f) - delta) * a.scale;
#pragma unroll
                for (int t = 0; t < 8; ++t) {
                    dqk[t] = fmaf(ds, k8[t], dqk[t]);
                    dqr[t] = fmaf(ds, r8[t], dqr[t]);
                }
                // split mode: only the current row (the one whose dk / dv the dgrad chain needs) is written here;
                // the memory rows are outer products of the saved (dS, P~) with (q + u, dO): relattn_dec_keys
                if (!SPLIT || j == jhi) {
                    float dk8[8], dv8[8];
#pragma unroll
                    for (int t = 0; t < 8; ++t) { dk8[t] = ds * qu[t]; dv8[t] = pw * g8[t]; }
                    store8(dkp, dk8);
                    store8(dvp, dv8);
                }
                if constexpr (SPLIT) {  // two lanes of the key group write the two scratch values side by side
                    if (dc < 2) dsp[dc ? pw_off : 0] = dc ? pw : ds;
                } else {
                    if (dc == 0) *dsp = ds;
                }
            }
            dkp += dstep; dvp += dstep; dsp += sstep;
        }
        cp_wait<0>();
        __syncwarp();  // reconverge the key groups before the full-warp shuffles
#pragma unroll
        for (int t = 0; t < 8; ++t) {
            float x = dqk[t], y = dqr[t];
            x += __shfl_xor_sync(0xffffffffu, x, 8);
            x += __shfl_xor_sync(0xffffffffu, x, 16);
            y += __shfl_xor_sync(0xffffffffu, y, 8);
            y += __shfl_xor_sync(0xffffffffu, y, 16);
            dqk[t] = x; dqr[t] = y;
        }
        if (kg == 0) {
            float s8[8];
#pragma unroll
            for (int t = 0; t < 8; ++t) s8[t] = dqk[t] + dqr[t];
            store8(dq + (int64_t)b * ldq + col, s8);
        }
    }
    // du = column sums of the content part of dq, dvb of the position part (r_w_bias / r_r_bias are shared by all rows):
    // 128 float atomics per warp onto N * 128 addresses.  (A first version merged the warps of a CTA in shared memory
    // first; its head-matching loops with integer modulo cost more instructions than the whole key loop of short rows.)
    // Split mode: the 128 x B*N atomics land 512-deep on N * 128 addresses -- on the critical path of the chain.  The
    // per-sequence rows go to the scratch instead ([2][B, N * 64] after the dS / P~ blocks) and relattn_dec_bias sums
    // them over the batch on the side stream.
    if (active && kg == 0) {
        if constexpr (SPLIT) {
            float* rows = dsbuf + 2 * (int64_t)a.N * a.K * a.B + (int64_t)b * a.N * HS + col;
            store8(rows, dqk);
            store8(rows + (int64_t)a.B * a.N * HS, dqr);
        } else {
#pragma unroll
            for (int t = 0; t < 8; ++t) {
                atomicAdd(&du[col + t], dqk[t]);
                atomicAdd(&dvb[col + t], dqr[t]);
            }
        }
    }
}

// du[c] += sum_b rows[0][b, c],  dvb[c] += sum_b rows[1][b, c]   (split mode, memory-side phase)
__global__ void __launch_bounds__(256)
relattn_dec_bias(const float* __restrict__ rows, float* __restrict__ du, float* __restrict__ dvb, int B, int NH) {
    __shared__ float part[8][33];
    const int c = blockIdx.x * 32 + threadIdx.x;
    const float* src = rows + (int64_t)blockIdx.y * B * NH;
    float s = 0.f;
    if (c < NH)
        for (int b = threadIdx.y; b < B; b += 8) s += src[(int64_t)b * NH + c];
    part[threadIdx.y][threadIdx.x] = s;
    __syncthreads();
    if (threadIdx.y == 0 && c < NH) {
        float t = 0.f;
#pragma unroll
        for (int i = 0; i < 8; ++i) t += part[i][threadIdx.x];
        atomicAdd(blockIdx.y ? &dvb[c] : &du[c], t);
    }
}

// dR[j, n, :] += sum_b dS[b, n, j] * (q[b, n, :] + r_r_bias[n, :])      (dS carries the 1/sqrt(d_head) factor)
// One CTA per (16-key tile, head n, batch slice): thread = (key jj, 4 dims); per sequence the CTA reads 16 consecutive
// dS values (one 64-byte piece of the warp-contiguous [B, N, K] scratch rows) and the head's 128-byte q row.  The
// batch is cut into DR_SLICES slices for parallelism (the whole reduction is 44 MFMA: latency, not throughput); the
// slices meet in the zeroed dr through atomics (DR_SLICES-way contention).
constexpr int DR_THREADS = 256, DR_KEYS = 16, DR_SLICES = 8;
template <typename T>
__global__ void __launch_bounds__(DR_THREADS)
relattn_dec_dr(const T* __restrict__ q, int64_t ldq, const float* __restrict__ vb, const float* __restrict__ dsbuf,
               float* __restrict__ dr, int64_t lddr, DecArgs a) {
    const int n = blockIdx.y;
    const int jj = threadIdx.x >> 4, dq4 = (threadIdx.x & 15) * 4;
    const int j = blockIdx.x * DR_KEYS + jj;
    const int per = (a.B + DR_SLICES - 1) / DR_SLICES;
    const int b0 = blockIdx.z * per, b1 = min(a.B, b0 + per);
    if (j >= a.K) return;
    const float* ds = dsbuf + (int64_t)n * a.K + j;  // dS[b, n, j] at ds[b * N * K]
    const int64_t bstride = (int64_t)a.N * a.K;
    const T* qp = q + n * HS + dq4;
    float acc[4] = {0.f, 0.f, 0.f, 0.f}, sum = 0.f;
#pragma unroll 8
    for (int b = b0; b < b1; ++b) {
        const float w = ds[b * bstride];
        const T* qr = qp + (int64_t)b * ldq;
#pragma unroll
        for (int t = 0; t < 4; ++t) acc[t] = fmaf(w, to_f(qr[t]), acc[t]);
        sum += w;
    }
    float* dst = dr + (int64_t)j * lddr + n * HS + dq4;
#pragma unroll
    for (int t = 0; t < 4; ++t) atomicAdd(dst + t, fmaf(sum, vb[n * HS + dq4 + t], acc[t]));
}

// Memory-row half of the split backward: dk[j, b, n, :] = dS[n, j, b] (q + r_w_bias)[b, n, :],
// dv[j, b, n, :] = P~[n, j, b] dO[b, n, :] for the rows j < M.  These rows feed only the K/V weight gradient (the memory
// is detached, mem_transformer.py:461-475), so the kernel runs OFF the sampling chain's critical path, on a side
// stream.  Pure write stream: one thread per 8 dims, a CTA per (key row, 32 sequences).
template <typename T>
__global__ void __launch_bounds__(320)
relattn_dec_keys(const T* __restrict__ q, int64_t ldq, const float* __restrict__ u, const T* __restrict__ dout, int64_t ldo,
                 const float* __restrict__ dsbuf, T* __restrict__ dk, T* __restrict__ dv, int64_t lddkv, int NC, DecArgs a) {
    const int j = blockIdx.x;
    const int64_t pw_off = (int64_t)a.N * a.K * a.B;
    for (int e = threadIdx.x; e < 32 * NC; e += blockDim.x) {
        const int b = blockIdx.y * 32 + e / NC, c = e % NC;
        if (b >= a.B) break;
        const int n = c >> 3, col = 8 * c;
        const float* sp = dsbuf + ((int64_t)b * a.N + n) * a.K + j;
        const float ds = sp[0], pw = sp[pw_off];
        float x[8], uu[8], g8[8], dk8[8], dv8[8];
        load8(q + (int64_t)b * ldq + col, x);
        load8(u + col, uu);
        load8(dout + (int64_t)b * ldo + col, g8);
#pragma unroll
        for (int t = 0; t < 8; ++t) { dk8[t] = ds * (x[t] + uu[t]); dv8[t] = pw * g8[t]; }
        const int64_t row = ((int64_t)j * a.B + b) * lddkv + col;
        store8(dk + row, dk8);
        store8(dv + row, dv8);
    }
}

DecArgs make_dec(int B, int N, int M, int msl, int same_length, float scale, float drop_p, uint64_t seed, uint64_t site) {
    DecArgs a;
    a.split = 0;
    a.B = B; a.N = N; a.M = M; a.K = M + 1;
    // mem_transformer.py:496-503 at qlen = 1: keys j <= -msl are cut
    a.jlo0 = same_length ? (1 - msl > 0 ? 1 - msl : 0) : 0;
    a.scale = scale; a.scale_log2 = scale * 1.4426950408889634f;
    a.drop_scale = drop_p > 0.f ? 1.f / (1.f - drop_p) : 1.f;
    a.thresh = drop_p > 0.f ? dropout_thresh16(drop_p) : 0u;
    a.key = dropout_key(seed, site);
    a.key_start = nullptr;
    a.key_base = 0;
    return a;
}
}  // namespace

int tgan_set_step_ctr_relattn_decode(const void* p) { return tgan_set_step_ctr_local(p); }

// Eligibility: Q == 1, rows aligned for 16-byte (bf16) / 32-byte (fp32) vector access.
int tgan_relattn_fwd_decode1(int dtype, const void* q, int64_t ldq, const void* k, const void* v, int64_t ldkv,
                             const void* r, int64_t ldr, const float* u, const float* vb, const uint8_t* reset,
                             const int32_t* key_start, int64_t key_base, void* out, int64_t ldo, float* lse, int B, int N,
                             int M, int msl, int same_length, float scale, float drop_p, uint64_t seed, uint64_t site,
                             cudaStream_t st) {
    DecArgs a = make_dec(B, N, M, msl, same_length, scale, drop_p, seed, site);
    a.key_start = key_start;
    a.key_base = key_base;
    const int DW = N <= DW_MAX ? N : 4;
    const int grid = ceil_div((int64_t)B * N, DW);
    const size_t sm_f32 = (size_t)PF * 3 * DW * 32 * 32, sm_bf16 = (size_t)PF * 3 * DW * 32 * 16;
    static bool attr = false;
    if (!attr) {
        TGAN_CUDA_OK(cudaFuncSetAttribute(relattn_dec_fwd<float>, cudaFuncAttributeMaxDynamicSharedMemorySize, PF * 3 * DW_MAX * 32 * 32));
        TGAN_CUDA_OK(cudaFuncSetAttribute(relattn_dec_fwd<bf16>, cudaFuncAttributeMaxDynamicSharedMemorySize, PF * 3 * DW_MAX * 32 * 16));
        attr = true;
    }
    if (dtype == TGAN_F32)
        relattn_dec_fwd<float><<<grid, DW * 32, sm_f32, st>>>((const float*)q, ldq, (const float*)k, (const float*)v, ldkv,
                                                          (const float*)r, ldr, u, vb, reset, (float*)out, ldo, lse, a);
    else
        relattn_dec_fwd<bf16><<<grid, DW * 32, sm_bf16, st>>>((const bf16*)q, ldq, (const bf16*)k, (const bf16*)v, ldkv,
                                                         (const bf16*)r, ldr, u, vb, reset, (bf16*)out, ldo, lse, a);
    TGAN_COUNT_LAUNCH();
    TGAN_LAUNCH_OK();
    return 0;
}

// phase 0: the whole backward on `st`.  phase 1: query side only (dq, du / dvb, dk / dv of the current row, the dS / P~
// scratch); phase 2: memory side (dk / dv of the rows j < M from the scratch, dR) -- see tgan_relattn_bwd_step.
int tgan_relattn_bwd_decode1(int dtype, const void* q, int64_t ldq, const void* k, const void* v, int64_t ldkv,
                             const void* r, int64_t ldr, const float* u, const float* vb, const uint8_t* reset,
                             const void* out, const void* dout, int64_t ldo, const float* lse, float* scratch, void* dq,
                             void* dk, void* dv, int64_t lddkv, float* dr, int64_t lddr, float* du, float* dvb, int B,
                             int N, int M, int msl, int same_length, float scale, float drop_p, uint64_t seed,
                             uint64_t site, cudaStream_t st, int phase) {
    DecArgs a = make_dec(B, N, M, msl, same_length, scale, drop_p, seed, site);
    a.split = phase != 0;
    if (phase == 2) {
        if (M > 0) {
            const int NC = N * (HS / 8);
            dim3 gk(M, ceil_div(B, 32));
            if (dtype == TGAN_F32)
                relattn_dec_keys<float><<<gk, 320, 0, st>>>((const float*)q, ldq, u, (const float*)dout, ldo, scratch,
                                                            (float*)dk, (float*)dv, lddkv, NC, a);
            else
                relattn_dec_keys<bf16><<<gk, 320, 0, st>>>((const bf16*)q, ldq, u, (const bf16*)dout, ldo, scratch,
                                                           (bf16*)dk, (bf16*)dv, lddkv, NC, a);
            TGAN_COUNT_LAUNCH();
            TGAN_LAUNCH_OK();
        }
        TGAN_CUDA_OK(cudaMemset2DAsync(dr, lddr * sizeof(float), 0, (size_t)N * HS * sizeof(float), a.K, st));
        dim3 g2(ceil_div(a.K, DR_KEYS), N, DR_SLICES);
        if (dtype == TGAN_F32)
            relattn_dec_dr<float><<<g2, DR_THREADS, 0, st>>>((const float*)q, ldq, vb, scratch, dr, lddr, a);
        else
            relattn_dec_dr<bf16><<<g2, DR_THREADS, 0, st>>>((const bf16*)q, ldq, vb, scratch, dr, lddr, a);
        TGAN_COUNT_LAUNCH();
        TGAN_LAUNCH_OK();
        relattn_dec_bias<<<dim3(ceil_div(N * HS, 32), 2), dim3(32, 8), 0, st>>>(scratch + 2 * (int64_t)N * a.K * B, du, dvb, B,
                                                                             N * HS);
        TGAN_COUNT_LAUNCH();
        TGAN_LAUNCH_OK();
        return 0;
    }
    const int DW = 4;  // <= 96 registers x 128 threads: 5 CTAs (20 warps) per SM; 10-warp CTAs at 128 registers fit only once
    const int grid = ceil_div((int64_t)B * N, DW);
    const size_t sm_f32 = (size_t)PF * 3 * DW * 32 * 32, sm_bf16 = (size_t)PF * 3 * DW * 32 * 16;
    static bool attr = false;
    if (!attr) {  // fp32: 48 KB of FIFO + the static du / dvb staging exceeds the default 48 KB window
        TGAN_CUDA_OK(cudaFuncSetAttribute(relattn_dec_bwd<float, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, PF * 3 * 128 * 32));
        TGAN_CUDA_OK(cudaFuncSetAttribute(relattn_dec_bwd<float, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, PF * 3 * 128 * 32));
        attr = true;
    }
#define TGAN_DEC_BWD(T, S, SM)                                                                                         \
    relattn_dec_bwd<T, S><<<grid, DW * 32, SM, st>>>((const T*)q, ldq, (const T*)k, (const T*)v, ldkv, (const T*)r, ldr, u, \
                                                     vb, reset, (const T*)out, (const T*)dout, ldo, lse, (T*)dq, (T*)dk,  \
                                                     (T*)dv, lddkv, scratch, du, dvb, a)
    if (dtype == TGAN_F32) {
        if (phase) TGAN_DEC_BWD(float, true, sm_f32); else TGAN_DEC_BWD(float, false, sm_f32);
    } else {
        if (phase) TGAN_DEC_BWD(bf16, true, sm_bf16); else TGAN_DEC_BWD(bf16, false, sm_bf16);
    }
#undef TGAN_DEC_BWD
    TGAN_COUNT_LAUNCH();
    TGAN_LAUNCH_OK();
    if (phase == 1) return 0;
    TGAN_CUDA_OK(cudaMemset2DAsync(dr, lddr * sizeof(float), 0, (size_t)N * HS * sizeof(float), a.K, st));
    dim3 g2(ceil_div(a.K, DR_KEYS), N, DR_SLICES);
    if (dtype == TGAN_F32)
        relattn_dec_dr<float><<<g2, DR_THREADS, 0, st>>>((const float*)q, ldq, vb, scratch, dr, lddr, a);
    else
        relattn_dec_dr<bf16><<<g2, DR_THREADS, 0, st>>>((const bf16*)q, ldq, vb, scratch, dr, lddr, a);
    TGAN_COUNT_LAUNCH();
    TGAN_LAUNCH_OK();
    return 0;
}

extern "C" int tgan_relattn_bwd_step(int phase, int dtype, const void* q, int64_t ldq, const void* k, const void* v,
                                     int64_t ldkv, const void* r, int64_t ldr, const float* u, const float* vb,
                                     const uint8_t* reset, const void* out, const void* dout, int64_t ldo,
                                     const float* lse, float* scratch, void* dq, void* dk, void* dv, int64_t lddkv,
                                     float* dr, int64_t lddr, float* du, float* dvb, int B, int N, int M, int msl,
                                     int same_length, float scale, float drop_p, uint64_t seed, uint64_t site,
                                     void* stream) {
    TGAN_CHECK_ARG(phase == 1 || phase == 2, "tgan_relattn_bwd_step: phase must be 1 (query side) or 2 (memory side)");
    TGAN_CHECK_ARG(B > 0 && N > 0 && M >= 0, "tgan_relattn_bwd_step: bad dims");
    const uintptr_t al = (uintptr_t)q | (uintptr_t)k | (uintptr_t)v | (uintptr_t)r | (uintptr_t)out | (uintptr_t)dout |
                         (uintptr_t)dq | (uintptr_t)dk | (uintptr_t)dv | (uintptr_t)u | (uintptr_t)vb;
    TGAN_CHECK_ARG((al & 31) == 0 && ldq % 8 == 0 && ldkv % 8 == 0 && ldr % 8 == 0 && ldo % 8 == 0 && lddkv % 8 == 0 &&
                   lddr % 4 == 0, "tgan_relattn_bwd_step: operands must be 32-byte aligned, ld multiples of 8");
    return tgan_relattn_bwd_decode1(dtype, q, ldq, k, v, ldkv, r, ldr, u, vb, reset, out, dout, ldo, lse, scratch, dq, dk,
                                    dv, lddkv, dr, lddr, du, dvb, B, N, M, msl, same_length, scale, drop_p, seed, site,
                                    (cudaStream_t)stream, phase);
}
