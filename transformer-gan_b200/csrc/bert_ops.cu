// Row / attention kernels of the BERT discriminator (transformer_gan.py:391-445: BertForSequenceClassification on
// `inputs_embeds`, and calc_gradient_penalty :203-230).  The reference calls the third-party HuggingFace modules
// (transformers ==2.5.1, modeling_bert.py: BertEmbeddings / BertSelfAttention / BertSelfOutput / BertIntermediate /
// BertOutput); these kernels restate that published arithmetic:
//   embeddings : LayerNorm(inputs_embeds + position_embeddings[t] + token_type_embeddings[0]) -> dropout
//   attention  : softmax(Q K^T / sqrt(d_head)) -> dropout -> . V       per (sequence, head), T <= 64 tokens
//   GELU       : x * 0.5 * (1 + erf(x / sqrt 2))                        (hidden_act "gelu")
// in three flavours each -- value, input-gradient (dgrad) and forward-mode tangent (JVP).  The WGAN-GP penalty needs
// d/dtheta ||grad_x D(x)||: with every encoder weight frozen (the shipped freeze_layers ['0'..'4'] + pretrained
// embeddings) theta sits behind the encoder, so that derivative is J_enc applied to a direction = one JVP pass; no
// double-backward graph is ever built.  The dense layers run on tgan_gemm (tcgen05); everything here is HBM- or
// latency-bound glue plus the 64 x 64 attention tiles (3 % of the encoder's FLOPs).
#include "common.cuh"

namespace {
constexpr float INV_SQRT2 = 0.70710678118654752440f;
constexpr float INV_SQRT_2PI = 0.39894228040143267794f;

__device__ __forceinline__ float gelu_f(float x) { return 0.5f * x * (1.f + erff(x * INV_SQRT2)); }
__device__ __forceinline__ float gelu_grad_f(float x) {
    return 0.5f * (1.f + erff(x * INV_SQRT2)) + x * INV_SQRT_2PI * __expf(-0.5f * x * x);
}

// mode 0: out = gelu(u);  mode 1: out = t * gelu'(u)   (dgrad and JVP are the same map)
template <typename T>
__global__ void gelu_kernel(const T* __restrict__ u, int64_t ldu, const T* __restrict__ t, int64_t ldt, T* __restrict__ out,
                            int64_t ldo, int rows, int cols8, int mode) {
    const int64_t total = (int64_t)rows * cols8;
    for (int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (int64_t)gridDim.x * blockDim.x) {
        const int row = (int)(idx / cols8), c = (int)(idx % cols8) * 8;
        float x[8], o[8];
        load8(u + (int64_t)row * ldu + c, x);
        if (mode == 0) {
#pragma unroll
            for (int i = 0; i < 8; ++i) o[i] = gelu_f(x[i]);
        } else {
            float g[8];
            load8(t + (int64_t)row * ldt + c, g);
#pragma unroll
            for (int i = 0; i < 8; ++i) o[i] = g[i] * gelu_grad_f(x[i]);
        }
        store8(out + (int64_t)row * ldo + c, o);
    }
}

// z[row, :] = x[row, :] (+ table[row % period, :]);  x given directly (x != NULL) or gathered: x[row] = E[ids[row]]
template <typename T>
__global__ void embed_rows_kernel(const T* __restrict__ x, int64_t ldx, const int64_t* __restrict__ ids,
                                  const T* __restrict__ E, int64_t lde, const float* __restrict__ table, int period,
                                  float* __restrict__ z, int64_t ldz, int rows, int cols8) {
    const int64_t total = (int64_t)rows * cols8;
    for (int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (int64_t)gridDim.x * blockDim.x) {
        const int row = (int)(idx / cols8), c = (int)(idx % cols8) * 8;
        float v[8], tb[8];
        if (x) load8(x + (int64_t)row * ldx + c, v);
        else load8(E + ids[row] * lde + c, v);
        if (table) {
            load8(table + (int64_t)(row % period) * (cols8 * 8) + c, tb);
#pragma unroll
            for (int i = 0; i < 8; ++i) v[i] += tb[i];
        }
        store8(z + (int64_t)row * ldz + c, v);
    }
}

// LayerNorm tangent: ydot = gamma * rstd * (zd - mean(zd) - xhat * mean(zd * xhat)),  xhat = (z - mean) * rstd.
// One warp per row; D <= 1024, D % 4 == 0.
constexpr int WPB = 8;
template <typename T>
__global__ void ln_jvp_kernel(const float* __restrict__ zd, int64_t ldzd, const float* __restrict__ z, int64_t ldz,
                              const float* __restrict__ gamma, const float* __restrict__ mean,
                              const float* __restrict__ rstd, T* __restrict__ yd, int64_t ldy, int rows, int D) {
    const int row = blockIdx.x * WPB + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (row >= rows) return;
    const float mu = mean[row], rs = rstd[row];
    float t[8][4], xh[8][4];
    float s1 = 0.f, s2 = 0.f;
#pragma unroll
    for (int u = 0; u < 8; ++u) {
        const int c = lane * 4 + 128 * u;
        if (c < D) {
            const float4 a = *reinterpret_cast<const float4*>(zd + (int64_t)row * ldzd + c);
            const float4 b = *reinterpret_cast<const float4*>(z + (int64_t)row * ldz + c);
            t[u][0] = a.x; t[u][1] = a.y; t[u][2] = a.z; t[u][3] = a.w;
            xh[u][0] = (b.x - mu) * rs; xh[u][1] = (b.y - mu) * rs; xh[u][2] = (b.z - mu) * rs; xh[u][3] = (b.w - mu) * rs;
#pragma unroll
            for (int i = 0; i < 4; ++i) { s1 += t[u][i]; s2 += t[u][i] * xh[u][i]; }
        }
    }
    s1 = warp_sum(s1) / D; s2 = warp_sum(s2) / D;
#pragma unroll
    for (int u = 0; u < 8; ++u) {
        const int c = lane * 4 + 128 * u;
        if (c < D) {
            const float4 g = *reinterpret_cast<const float4*>(gamma + c);
            const float gg[4] = {g.x, g.y, g.z, g.w};
            T* o = yd + (int64_t)row * ldy + c;
#pragma unroll
            for (int i = 0; i < 4; ++i) o[i] = from_f<T>(gg[i] * rs * (t[u][i] - s1 - xh[u][i] * s2));
        }
    }
}

// ------------------------------------------------------------------------------------------------------------
// attention tiles: one CTA (256 threads) per (sequence b, head h); T <= 64 tokens, d_head <= 64 (multiple of 8).
// Operands live in shared memory as fp32 with an odd leading dimension; each thread owns a 4 x 4 block of every
// T x T or T x d_head product.  qkv rows: [B*T, 3*H] = [Q | K | V], head h at columns h*dh of each third.
// ------------------------------------------------------------------------------------------------------------
constexpr int AT = 64, ALD = 65, ATHREADS = 256;

struct BertAttnArgs {
    int B, heads, T, dh, H;   // H = heads * dh
    float scale, drop_scale;
    uint32_t thresh, key;
};

template <typename T>
__device__ __forceinline__ void load_tile(float* s, const T* g, int64_t ldg, int rows, int cols) {
    // rows x cols (cols % 8 == 0) -> s[r * ALD + c]; rows beyond `rows` are zero filled up to AT
    const int c8 = cols / 8;
    for (int idx = threadIdx.x; idx < AT * c8; idx += ATHREADS) {
        const int r = idx / c8, c = (idx % c8) * 8;
        float v[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
        if (r < rows) load8(g + (int64_t)r * ldg + c, v);
#pragma unroll
        for (int i = 0; i < 8; ++i) s[r * ALD + c + i] = v[i];
    }
}
// C[i][j] (+)= sum_k A[i][k] * B[j][k]      (i, j < 64; k < K)      "NT"
__device__ __forceinline__ void mm_nt(const float* A, const float* B, int K, float acc[4][4]) {
    const int bi = (threadIdx.x >> 4) * 4, bj = (threadIdx.x & 15) * 4;
    for (int k = 0; k < K; ++k) {
        float a[4], b[4];
#pragma unroll
        for (int x = 0; x < 4; ++x) { a[x] = A[(bi + x) * ALD + k]; b[x] = B[(bj + x) * ALD + k]; }
#pragma unroll
        for (int x = 0; x < 4; ++x)
#pragma unroll
            for (int y = 0; y < 4; ++y) acc[x][y] = fmaf(a[x], b[y], acc[x][y]);
    }
}
// C[i][j] (+)= sum_k A[i][k] * B[k][j]      "NN"
__device__ __forceinline__ void mm_nn(const float* A, const float* B, int K, float acc[4][4]) {
    const int bi = (threadIdx.x >> 4) * 4, bj = (threadIdx.x & 15) * 4;
    for (int k = 0; k < K; ++k) {
        float a[4], b[4];
#pragma unroll
        for (int x = 0; x < 4; ++x) { a[x] = A[(bi + x) * ALD + k]; b[x] = B[k * ALD + bj + x]; }
#pragma unroll
        for (int x = 0; x < 4; ++x)
#pragma unroll
            for (int y = 0; y < 4; ++y) acc[x][y] = fmaf(a[x], b[y], acc[x][y]);
    }
}
// C[i][j] (+)= sum_k A[k][i] * B[k][j]      "TN"
__device__ __forceinline__ void mm_tn(const float* A, const float* B, int K, float acc[4][4]) {
    const int bi = (threadIdx.x >> 4) * 4, bj = (threadIdx.x & 15) * 4;
    for (int k = 0; k < K; ++k) {
        float a[4], b[4];
#pragma unroll
        for (int x = 0; x < 4; ++x) { a[x] = A[k * ALD + bi + x]; b[x] = B[k * ALD + bj + x]; }
#pragma unroll
        for (int x = 0; x < 4; ++x)
#pragma unroll
            for (int y = 0; y < 4; ++y) acc[x][y] = fmaf(a[x], b[y], acc[x][y]);
    }
}
__device__ __forceinline__ void zero_acc(float acc[4][4]) {
#pragma unroll
    for (int x = 0; x < 4; ++x)
#pragma unroll
        for (int y = 0; y < 4; ++y) acc[x][y] = 0.f;
}
__device__ __forceinline__ void store_acc(float* S, const float acc[4][4], float mul) {
    const int bi = (threadIdx.x >> 4) * 4, bj = (threadIdx.x & 15) * 4;
#pragma unroll
    for (int x = 0; x < 4; ++x)
#pragma unroll
        for (int y = 0; y < 4; ++y) S[(bi + x) * ALD + bj + y] = acc[x][y] * mul;
}
// rows x cols block of the thread-owned accumulators -> global [rows, ld] (cols % 4 == 0)
template <typename T>
__device__ __forceinline__ void store_acc_global(T* g, int64_t ldg, const float acc[4][4], int rows, int cols, float mul) {
    const int bi = (threadIdx.x >> 4) * 4, bj = (threadIdx.x & 15) * 4;
    if (bj >= cols) return;
#pragma unroll
    for (int x = 0; x < 4; ++x) {
        if (bi + x >= rows) continue;
#pragma unroll
        for (int y = 0; y < 4; ++y) g[(int64_t)(bi + x) * ldg + bj + y] = from_f<T>(acc[x][y] * mul);
    }
}
__device__ __forceinline__ bool bert_keep(const BertAttnArgs& a, uint32_t key, int bh, int i, int j) {
    if (!a.thresh) return true;
    return dropout_keep_k(key, ((uint64_t)bh * a.T + i) * a.T + j, a.thresh);
}

// forward: ctx = drop(softmax(Q K^T * scale)) V ;  lse [B*heads*T] saved for the recompute in dgrad / JVP
template <typename T>
__global__ void __launch_bounds__(ATHREADS)
bert_attn_fwd_kernel(const T* __restrict__ qkv, int64_t ldq, T* __restrict__ ctx, int64_t ldc, float* __restrict__ lse,
                     BertAttnArgs a) {
    extern __shared__ float sm[];
    float *sQ = sm, *sK = sm + AT * ALD, *sV = sm + 2 * AT * ALD, *sS = sm + 3 * AT * ALD;
    const int bh = blockIdx.x, b = bh / a.heads, h = bh % a.heads;
    const T* base = qkv + (int64_t)b * a.T * ldq + h * a.dh;
    load_tile(sQ, base, ldq, a.T, a.dh);
    load_tile(sK, base + a.H, ldq, a.T, a.dh);
    load_tile(sV, base + 2 * a.H, ldq, a.T, a.dh);
    __syncthreads();
    float acc[4][4];
    zero_acc(acc);
    mm_nt(sQ, sK, a.dh, acc);
    store_acc(sS, acc, a.scale);
    __syncthreads();
    const uint32_t key = step_fold(a.key);
    {   // 4 threads per query row (adjacent lanes), 16 columns each: softmax + dropout in place.  (One thread per row
        // left 192 of the 256 threads idle through the longest dependent chain of the kernel.)
        const int i = threadIdx.x >> 2, part = threadIdx.x & 3, j0 = part * 16, j1 = min(j0 + 16, a.T);
        float* row = sS + i * ALD;
        const bool live = i < a.T;
        float m = -INFINITY;
        if (live)
            for (int j = j0; j < j1; ++j) m = fmaxf(m, row[j]);
        m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, 1));
        m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, 2));
        float l = 0.f;
        if (live)
            for (int j = j0; j < j1; ++j) { const float e = __expf(row[j] - m); row[j] = e; l += e; }
        l += __shfl_xor_sync(0xffffffffu, l, 1);
        l += __shfl_xor_sync(0xffffffffu, l, 2);
        if (live) {
            const float inv = 1.f / l;
            for (int j = j0; j < j1; ++j) row[j] = bert_keep(a, key, bh, i, j) ? row[j] * inv * a.drop_scale : 0.f;
            if (part == 0) lse[(int64_t)bh * a.T + i] = m + __logf(l);
        }
        for (int j = max(j0, live ? a.T : 0); j < j0 + 16; ++j) row[j] = 0.f;
    }
    __syncthreads();
    zero_acc(acc);
    mm_nn(sS, sV, a.T, acc);
    store_acc_global(ctx + (int64_t)b * a.T * ldc + h * a.dh, ldc, acc, a.T, a.dh, 1.f);
}

// Shared by dgrad and JVP: S tile -> P (un-dropped probabilities) from the saved lse
__device__ __forceinline__ void probs_from_lse(float* sS, const float* lse_row, int T) {
    for (int idx = threadIdx.x; idx < AT * AT; idx += ATHREADS) {
        const int i = idx / AT, j = idx % AT;
        sS[i * ALD + j] = (i < T && j < T) ? __expf(sS[i * ALD + j] - lse_row[i]) : 0.f;
    }
}

// dgrad: dqkv from dctx.   dV = P~^T dO ;  dP~ = dO V^T ;  dS = P (drop'(dP~) - delta) ;  dQ = dS K s ;  dK = dS^T Q s
template <typename T>
__global__ void __launch_bounds__(ATHREADS)
bert_attn_bwd_kernel(const T* __restrict__ qkv, int64_t ldq, const T* __restrict__ dctx, int64_t ldc,
                     const float* __restrict__ lse, T* __restrict__ dqkv, int64_t lddq, BertAttnArgs a) {
    extern __shared__ float sm[];
    float *sQ = sm, *sK = sm + AT * ALD, *sV = sm + 2 * AT * ALD, *sS = sm + 3 * AT * ALD, *sG = sm + 4 * AT * ALD,
          *sD = sm + 5 * AT * ALD;
    __shared__ float s_lse[AT], s_delta[AT];
    const int bh = blockIdx.x, b = bh / a.heads, h = bh % a.heads;
    const T* base = qkv + (int64_t)b * a.T * ldq + h * a.dh;
    load_tile(sQ, base, ldq, a.T, a.dh);
    load_tile(sK, base + a.H, ldq, a.T, a.dh);
    load_tile(sV, base + 2 * a.H, ldq, a.T, a.dh);
    load_tile(sG, dctx + (int64_t)b * a.T * ldc + h * a.dh, ldc, a.T, a.dh);
    if (threadIdx.x < AT) s_lse[threadIdx.x] = threadIdx.x < a.T ? lse[(int64_t)bh * a.T + threadIdx.x] : 0.f;
    __syncthreads();
    float acc[4][4];
    zero_acc(acc);
    mm_nt(sQ, sK, a.dh, acc);
    store_acc(sS, acc, a.scale);
    zero_acc(acc);
    mm_nt(sG, sV, a.dh, acc);   // dP~[i][j] = dO_i . V_j
    store_acc(sD, acc, 1.f);
    __syncthreads();
    probs_from_lse(sS, s_lse, a.T);
    __syncthreads();
    const uint32_t key = step_fold(a.key);
    {   // 4 threads per row: delta = sum_j P~ dP~ ; then sD := dS, sS := P~
        const int i = threadIdx.x >> 2, part = threadIdx.x & 3, j0 = part * 16, j1 = min(j0 + 16, a.T);
        float* p = sS + i * ALD;
        float* d = sD + i * ALD;
        const bool live = i < a.T;
        float delta = 0.f;
        if (live)
            for (int j = j0; j < j1; ++j) {
                const bool keep = bert_keep(a, key, bh, i, j);
                const float dpk = keep ? d[j] * a.drop_scale : 0.f;   // gradient w.r.t. the un-dropped probability
                delta += p[j] * dpk;
                d[j] = dpk;
            }
        delta += __shfl_xor_sync(0xffffffffu, delta, 1);
        delta += __shfl_xor_sync(0xffffffffu, delta, 2);
        if (live)
            for (int j = j0; j < j1; ++j) {
                const float pj = p[j];
                const bool keep = bert_keep(a, key, bh, i, j);
                d[j] = pj * (d[j] - delta);
                p[j] = keep ? pj * a.drop_scale : 0.f;
            }
    }
    __syncthreads();
    T* obase = dqkv + (int64_t)b * a.T * lddq + h * a.dh;
    zero_acc(acc);
    mm_nn(sD, sK, a.T, acc);                                   // dQ = dS K
    store_acc_global(obase, lddq, acc, a.T, a.dh, a.scale);
    zero_acc(acc);
    mm_tn(sD, sQ, a.T, acc);                                   // dK = dS^T Q
    store_acc_global(obase + a.H, lddq, acc, a.T, a.dh, a.scale);
    zero_acc(acc);
    mm_tn(sS, sG, a.T, acc);                                   // dV = P~^T dO
    store_acc_global(obase + 2 * a.H, lddq, acc, a.T, a.dh, 1.f);
}

// JVP: ctx_dot from qkv_dot.  Sd = (Qd K^T + Q Kd^T) s ;  Pd = P (Sd - rowsum(P Sd)) ;  ctx_d = drop(Pd) V + drop(P) Vd
template <typename T>
__global__ void __launch_bounds__(ATHREADS)
bert_attn_jvp_kernel(const T* __restrict__ qkv, int64_t ldq, const T* __restrict__ qkvd, int64_t ldqd,
                     const float* __restrict__ lse, T* __restrict__ ctxd, int64_t ldc, BertAttnArgs a) {
    extern __shared__ float sm[];
    float *sQ = sm, *sK = sm + AT * ALD, *sV = sm + 2 * AT * ALD, *sS = sm + 3 * AT * ALD, *sQd = sm + 4 * AT * ALD,
          *sKd = sm + 5 * AT * ALD, *sVd = sm + 6 * AT * ALD, *sSd = sm + 7 * AT * ALD;
    __shared__ float s_lse[AT];
    const int bh = blockIdx.x, b = bh / a.heads, h = bh % a.heads;
    const T* base = qkv + (int64_t)b * a.T * ldq + h * a.dh;
    const T* based = qkvd + (int64_t)b * a.T * ldqd + h * a.dh;
    load_tile(sQ, base, ldq, a.T, a.dh);
    load_tile(sK, base + a.H, ldq, a.T, a.dh);
    load_tile(sV, base + 2 * a.H, ldq, a.T, a.dh);
    load_tile(sQd, based, ldqd, a.T, a.dh);
    load_tile(sKd, based + a.H, ldqd, a.T, a.dh);
    load_tile(sVd, based + 2 * a.H, ldqd, a.T, a.dh);
    if (threadIdx.x < AT) s_lse[threadIdx.x] = threadIdx.x < a.T ? lse[(int64_t)bh * a.T + threadIdx.x] : 0.f;
    __syncthreads();
    float acc[4][4];
    zero_acc(acc);
    mm_nt(sQ, sK, a.dh, acc);
    store_acc(sS, acc, a.scale);
    zero_acc(acc);
    mm_nt(sQd, sK, a.dh, acc);
    mm_nt(sQ, sKd, a.dh, acc);
    store_acc(sSd, acc, a.scale);
    __syncthreads();
    probs_from_lse(sS, s_lse, a.T);
    __syncthreads();
    const uint32_t key = step_fold(a.key);
    {   // 4 threads per row: sSd := drop(Pd), sS := drop(P)
        const int i = threadIdx.x >> 2, part = threadIdx.x & 3, j0 = part * 16, j1 = min(j0 + 16, a.T);
        float* p = sS + i * ALD;
        float* d = sSd + i * ALD;
        const bool live = i < a.T;
        float dot = 0.f;
        if (live)
            for (int j = j0; j < j1; ++j) dot += p[j] * d[j];
        dot += __shfl_xor_sync(0xffffffffu, dot, 1);
        dot += __shfl_xor_sync(0xffffffffu, dot, 2);
        if (live)
            for (int j = j0; j < j1; ++j) {
                const float m = bert_keep(a, key, bh, i, j) ? a.drop_scale : 0.f;
                const float pj = p[j];
                d[j] = pj * (d[j] - dot) * m;
                p[j] = pj * m;
            }
        for (int j = max(j0, live ? a.T : 0); j < j0 + 16; ++j) d[j] = 0.f;
    }
    __syncthreads();
    zero_acc(acc);
    mm_nn(sSd, sV, a.T, acc);
    mm_nn(sS, sVd, a.T, acc);
    store_acc_global(ctxd + (int64_t)b * a.T * ldc + h * a.dh, ldc, acc, a.T, a.dh, 1.f);
}

BertAttnArgs make_bargs(int B, int heads, int T, int dh, float drop_p, uint64_t seed, uint64_t site) {
    BertAttnArgs a;
    a.B = B; a.heads = heads; a.T = T; a.dh = dh; a.H = heads * dh;
    a.scale = 1.f / sqrtf((float)dh);
    a.drop_scale = drop_p > 0.f ? 1.f / (1.f - drop_p) : 1.f;
    a.thresh = drop_p > 0.f ? dropout_thresh16(drop_p) : 0u;
    a.key = dropout_key(seed, site);
    return a;
}
// not a stream operation: safe under graph capture.  (No "set once" cache keyed on the kernel's TYPE: the dgrad and JVP
// kernels have identical signatures.)
template <typename K>
int set_smem(K kernel, int bytes) {
    return (int)cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
}
int grid_for(int64_t n, int threads) {
    int64_t g = (n + threads - 1) / threads;
    return (int)(g < 148 * 16 ? (g < 1 ? 1 : g) : 148 * 16);
}
}  // namespace

#define ST ((cudaStream_t)stream)
#define DISPATCH_T(dtype, call)                        \
    do {                                               \
        if ((dtype) == TGAN_F32) { using T = float; call; } \
        else { using T = bf16; call; }                 \
    } while (0)

int tgan_set_step_ctr_bert(const void* p) { return tgan_set_step_ctr_local(p); }

extern "C" int tgan_gelu(int dtype, int mode, const void* u, int64_t ldu, const void* t, int64_t ldt, void* out,
                         int64_t ldo, int rows, int cols, void* stream) {
    if (rows <= 0 || cols <= 0) return 0;
    TGAN_CHECK_ARG(cols % 8 == 0 && ldu % 8 == 0 && ldo % 8 == 0 && (mode == 0 || (t && ldt % 8 == 0)),
                   "tgan_gelu: cols / ld must be multiples of 8; mode 1 needs t");
    const int64_t n = (int64_t)rows * (cols / 8);
    DISPATCH_T(dtype, (gelu_kernel<T><<<grid_for(n, 256), 256, 0, ST>>>((const T*)u, ldu, (const T*)t, ldt, (T*)out, ldo,
                                                                         rows, cols / 8, mode)));
    TGAN_COUNT_LAUNCH();
    TGAN_LAUNCH_OK();
    return 0;
}

extern "C" int tgan_bert_embed_rows(int dtype, const void* x, int64_t ldx, const int64_t* ids, const void* E, int64_t lde,
                                    const float* table, int period, float* z, int64_t ldz, int rows, int cols,
                                    void* stream) {
    if (rows <= 0) return 0;
    TGAN_CHECK_ARG(cols % 8 == 0 && ldz % 8 == 0 && ((x && ldx % 8 == 0) || (ids && E && lde % 8 == 0)) && period > 0,
                   "tgan_bert_embed_rows: cols / ld multiples of 8; x or (ids, E) required");
    const int64_t n = (int64_t)rows * (cols / 8);
    DISPATCH_T(dtype, (embed_rows_kernel<T><<<grid_for(n, 256), 256, 0, ST>>>((const T*)x, ldx, ids, (const T*)E, lde, table,
                                                                               period, z, ldz, rows, cols / 8)));
    TGAN_COUNT_LAUNCH();
    TGAN_LAUNCH_OK();
    return 0;
}

extern "C" int tgan_ln_jvp(int dtype, const float* zd, int64_t ldzd, const float* z, int64_t ldz, const float* gamma,
                           const float* mean, const float* rstd, void* yd, int64_t ldy, int rows, int D, void* stream) {
    if (rows <= 0) return 0;
    TGAN_CHECK_ARG(D % 4 == 0 && D <= 1024 && ldzd % 4 == 0 && ldz % 4 == 0 &&
                       (((uintptr_t)zd | (uintptr_t)z | (uintptr_t)gamma) & 15) == 0,
                   "tgan_ln_jvp: D <= 1024, multiples of 4, 16-byte aligned rows");
    DISPATCH_T(dtype, (ln_jvp_kernel<T><<<ceil_div(rows, WPB), WPB * 32, 0, ST>>>(zd, ldzd, z, ldz, gamma, mean, rstd,
                                                                                   (T*)yd, ldy, rows, D)));
    TGAN_COUNT_LAUNCH();
    TGAN_LAUNCH_OK();
    return 0;
}

// bf16 tiles with d_head a multiple of 16 and 16-byte aligned rows run on the tensor cores (bert_attn_mma.cu)
static bool mma_ok(int dtype, int dh, int64_t ld0, int64_t ld1, int64_t ld2, const void* p0, const void* p1, const void* p2) {
    return dtype == TGAN_BF16 && dh % 16 == 0 && ld0 % 8 == 0 && ld1 % 8 == 0 && ld2 % 8 == 0 &&
           ((((uintptr_t)p0 | (uintptr_t)p1 | (uintptr_t)p2) & 15) == 0);
}

static int check_attn(int T, int dh, int64_t ldq, const char* who) {
    if (!(T >= 1 && T <= AT && dh >= 8 && dh <= AT && dh % 8 == 0 && ldq % 8 == 0)) {
        tgan_set_error("%s: needs 1 <= T <= 64 tokens, d_head a multiple of 8 <= 64, ld multiples of 8", who);
        return 1;
    }
    return 0;
}

extern "C" int tgan_bert_attn_fwd(int dtype, const void* qkv, int64_t ldq, void* ctx, int64_t ldc, float* lse, int B,
                                  int heads, int T, int dh, float drop_p, uint64_t seed, uint64_t site, void* stream) {
    if (check_attn(T, dh, ldq, "tgan_bert_attn_fwd")) return 1;
    if (mma_ok(dtype, dh, ldq, ldc, 8, qkv, ctx, nullptr))
        return tgan_bert_attn_fwd_mma(qkv, ldq, ctx, ldc, lse, B, heads, T, dh, drop_p, seed, site, ST);
    BertAttnArgs a = make_bargs(B, heads, T, dh, drop_p, seed, site);
    const int smem = 4 * AT * ALD * sizeof(float);
    if (dtype == TGAN_F32) TGAN_CUDA_OK((cudaError_t)set_smem(bert_attn_fwd_kernel<float>, smem));
    else TGAN_CUDA_OK((cudaError_t)set_smem(bert_attn_fwd_kernel<bf16>, smem));
    DISPATCH_T(dtype, (bert_attn_fwd_kernel<T><<<B * heads, ATHREADS, smem, ST>>>((const T*)qkv, ldq, (T*)ctx, ldc, lse, a)));
    TGAN_COUNT_LAUNCH();
    TGAN_LAUNCH_OK();
    return 0;
}

extern "C" int tgan_bert_attn_bwd(int dtype, const void* qkv, int64_t ldq, const void* dctx, int64_t ldc, const float* lse,
                                  void* dqkv, int64_t lddq, int B, int heads, int T, int dh, float drop_p, uint64_t seed,
                                  uint64_t site, void* stream) {
    if (check_attn(T, dh, ldq, "tgan_bert_attn_bwd")) return 1;
    if (mma_ok(dtype, dh, ldq, ldc, lddq, qkv, dctx, dqkv))
        return tgan_bert_attn_bwd_mma(qkv, ldq, dctx, ldc, lse, dqkv, lddq, B, heads, T, dh, drop_p, seed, site, ST);
    BertAttnArgs a = make_bargs(B, heads, T, dh, drop_p, seed, site);
    const int smem = 6 * AT * ALD * sizeof(float);
    if (dtype == TGAN_F32) TGAN_CUDA_OK((cudaError_t)set_smem(bert_attn_bwd_kernel<float>, smem));
    else TGAN_CUDA_OK((cudaError_t)set_smem(bert_attn_bwd_kernel<bf16>, smem));
    DISPATCH_T(dtype, (bert_attn_bwd_kernel<T><<<B * heads, ATHREADS, smem, ST>>>((const T*)qkv, ldq, (const T*)dctx, ldc, lse,
                                                                                   (T*)dqkv, lddq, a)));
    TGAN_COUNT_LAUNCH();
    TGAN_LAUNCH_OK();
    return 0;
}

extern "C" int tgan_bert_attn_jvp(int dtype, const void* qkv, int64_t ldq, const void* qkvd, int64_t ldqd, const float* lse,
                                  void* ctxd, int64_t ldc, int B, int heads, int T, int dh, float drop_p, uint64_t seed,
                                  uint64_t site, void* stream) {
    if (check_attn(T, dh, ldq, "tgan_bert_attn_jvp")) return 1;
    if (mma_ok(dtype, dh, ldq, ldqd, ldc, qkv, qkvd, ctxd))
        return tgan_bert_attn_jvp_mma(qkv, ldq, qkvd, ldqd, lse, ctxd, ldc, B, heads, T, dh, drop_p, seed, site, ST);
    BertAttnArgs a = make_bargs(B, heads, T, dh, drop_p, seed, site);
    const int smem = 8 * AT * ALD * sizeof(float);
    if (dtype == TGAN_F32) TGAN_CUDA_OK((cudaError_t)set_smem(bert_attn_jvp_kernel<float>, smem));
    else TGAN_CUDA_OK((cudaError_t)set_smem(bert_attn_jvp_kernel<bf16>, smem));
    DISPATCH_T(dtype, (bert_attn_jvp_kernel<T><<<B * heads, ATHREADS, smem, ST>>>((const T*)qkv, ldq, (const T*)qkvd, ldqd, lse,
                                                                                   (T*)ctxd, ldc, a)));
    TGAN_COUNT_LAUNCH();
    TGAN_LAUNCH_OK();
    return 0;
}
