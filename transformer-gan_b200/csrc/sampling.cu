// Batched on-device generation post-processing: generate.py:228-304 for a whole batch of sequences in ONE launch, no
// per-token host synchronisation (the reference does this on the host for a single sequence, one `.item()` per token).
// Per row of fp32 logits [V]:
//   exclude_bos (drop token 0, :232-233), empty-bar suppression (drop `empty_token` when the row's flag is set,
//   :235-247), temperature (:250-259; 0 = argmax), softmax, then "topk" (keep the k most probable, renormalise,
//   :270-275), "nucleus" (keep the sorted prefix whose EXCLUSIVE cumulative probability is < p, renormalise, :277-296)
//   or "random" (plain), then one categorical draw.  torch.multinomial's RNG stream cannot be reproduced, so the draw is
//   the inverse CDF of a uniform u in [0, 1): either injected per row (parity tests) or from Philox4x32-10.
// One warp per row; the row lives in shared memory; ranks are an all-pairs count (V = 310: 3 k compares per lane).
#include "common.cuh"

namespace {
constexpr int SW = 4;        // rows (warps) per CTA
constexpr int SMAXV = 1024;

struct SampleArgs {
    int rows, V, exclude_bos, empty_token, mode, topk;  // mode 0 random, 1 topk, 2 nucleus
    float temperature, top_p;
    uint64_t seed, site;
};

// One row of the post-processing above, by one warp: logits x [V] -> the sampled token; p [V] (shared) ends up as the
// filtered, renormalised distribution.  u_in: the injected uniform of this row, or NULL for Philox keyed by
// (seed, site, rng_row).  Every argument but x / p / lane is the same for the whole warp.
__device__ __forceinline__ int sample_row(const float* __restrict__ x, float* p, int lane, int V, bool sup,
                                          int exclude_bos, int empty_token, int mode, int topk, float top_p,
                                          float temperature, const float* u_in, uint64_t seed, uint64_t site,
                                          uint64_t rng_row) {
    // 1. masked, temperature-scaled logits; running max / argmax
    float mx = -INFINITY;
    int amax = V;
    for (int i = lane; i < V; i += 32) {
        const bool excluded = (exclude_bos && i == 0) || (sup && i == empty_token);
        float v = excluded ? -INFINITY : x[i];
        if (temperature > 0.f) v /= temperature;
        p[i] = v;
        if (v > mx) { mx = v; amax = i; }   // strict >: the lowest index wins ties inside a lane (ascending i)
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const float om = __shfl_xor_sync(0xffffffffu, mx, o);
        const int oi = __shfl_xor_sync(0xffffffffu, amax, o);
        if (om > mx || (om == mx && oi < amax)) { mx = om; amax = oi; }
    }
    __syncwarp();
    if (temperature == 0.f) {  // argmax (:250-253); the later filters keep the single non-zero entry
        for (int i = lane; i < V; i += 32) p[i] = i == amax ? 1.f : 0.f;
        return amax;
    }
    // 2. softmax
    float z = 0.f;
    for (int i = lane; i < V; i += 32) { const float e = __expf(p[i] - mx); p[i] = e; z += e; }
    z = warp_sum(z);
    const float inv = 1.f / z;
    for (int i = lane; i < V; i += 32) p[i] *= inv;
    __syncwarp();
    // 3. filter: rank_i = #{j : p_j > p_i or (p_j == p_i and j < i)},  before_i = sum of those p_j
    if ((mode == 1 && topk > 0 && topk < V) || (mode == 2 && top_p > 0.f)) {
        float keep_sum = 0.f;
        uint32_t keepbits = 0;  // this lane's elements i = lane + 32 t, t < 32
        for (int t = 0, i = lane; i < V; ++t, i += 32) {
            const float pi = p[i];
            int rank = 0;
            float before = 0.f;
            for (int j = 0; j < V; ++j) {
                const float pj = p[j];
                const bool ahead = pj > pi || (pj == pi && j < i);
                rank += ahead;
                before += ahead ? pj : 0.f;
            }
            const bool keep = mode == 1 ? rank < topk : (rank == 0 || before < top_p);
            if (keep) { keepbits |= 1u << t; keep_sum += pi; }
        }
        keep_sum = warp_sum(keep_sum);
        __syncwarp();
        const float rn = 1.f / keep_sum;
        for (int t = 0, i = lane; i < V; ++t, i += 32) p[i] = ((keepbits >> t) & 1) ? p[i] * rn : 0.f;
        __syncwarp();
    }
    // 4. inverse-CDF draw: token = first i with cumsum_i > u * total
    float u;
    if (u_in) u = *u_in;
    else {
        const Philox4 r = philox4x32_10(seed, step_fold_site(site), rng_row);
        u = (float)(r.x >> 8) * (1.f / 16777216.f);
    }
    const int C = (V + 31) / 32;           // contiguous chunk per lane
    const int lo = lane * C, hi = min(V, lo + C);
    float local = 0.f;
    for (int i = lo; i < hi; ++i) local += p[i];
    float incl = local;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const float t = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += t;
    }
    const float total = __shfl_sync(0xffffffffu, incl, 31);
    const float target = u * total;
    float c = incl - local;
    int found = V;
    for (int i = lo; i < hi; ++i) {
        c += p[i];
        if (found == V && c > target && p[i] > 0.f) found = i;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) found = min(found, __shfl_xor_sync(0xffffffffu, found, o));
    if (found == V) {  // rounding at the very top of the CDF: last entry with non-zero probability
        int last = -1;
        for (int i = lane; i < V; i += 32) if (p[i] > 0.f) last = max(last, i);
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) last = max(last, __shfl_xor_sync(0xffffffffu, last, o));
        found = last;
    }
    return found;
}

__global__ void __launch_bounds__(SW * 32)
sample_kernel(const float* __restrict__ logits, int64_t ldl, const float* __restrict__ u_in,
              const uint8_t* __restrict__ suppress, int64_t* __restrict__ ids, float* __restrict__ probs_out,
              int64_t ldp, SampleArgs a) {
    __shared__ float s_p[SW][SMAXV];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int row = blockIdx.x * SW + warp;
    if (row >= a.rows) return;
    float* p = s_p[warp];
    const bool sup = suppress && suppress[row];
    const int token = sample_row(logits + (int64_t)row * ldl, p, lane, a.V, sup, a.exclude_bos, a.empty_token, a.mode,
                                 a.topk, a.top_p, a.temperature, u_in ? u_in + row : nullptr, a.seed, a.site,
                                 (uint64_t)row);
    if (lane == 0) ids[row] = token;
    if (probs_out) {
        __syncwarp();
        for (int i = lane; i < a.V; i += 32) probs_out[(int64_t)row * ldp + i] = p[i];
    }
}

// One step of generation from a request queue (tgan_b200.h, tgan_sample_step): column b serves request req[b]
// (-1 = idle) with that request's settings, sampled by the same row body as sample_kernel.
struct StepArgs {
    const float* logits; int64_t ldl;
    const int32_t *req, *start, *out_off, *forced_next, *req_i, *run0;
    const float *req_f, *u;
    int32_t* run; int64_t *cur, *out; float* probs_out; int64_t ldp;
    int B, V, step;
    uint64_t seed, site;
};

__global__ void __launch_bounds__(SW * 32) sample_step_kernel(StepArgs a) {
    __shared__ float s_p[SW][SMAXV];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int b = blockIdx.x * SW + warp;
    if (b >= a.B) return;
    const int r = a.req[b];
    int64_t next = a.forced_next ? a.forced_next[b] : -1;
    if (r >= 0) {
        const int32_t* si = a.req_i + 5 * (int64_t)r;  // mode, topk, exclude_bos, empty_token, k
        const int empty_token = si[3], k = si[4];
        // empty-bar run over the column's input tokens; a request starting at this step starts a new run, from the run
        // over the conditioning tokens its context pass consumed
        int run = a.start[b] == a.step ? (a.run0 ? a.run0[r] : 0) : a.run[b];
        run = a.cur[b] == empty_token ? run + 1 : 0;
        const int off = a.out_off[b];
        const int token = sample_row(a.logits + (int64_t)b * a.ldl, s_p[warp], lane, a.V, k > 0 && run >= k, si[2],
                                     empty_token, si[0], si[1], a.req_f[2 * (int64_t)r + 1], a.req_f[2 * (int64_t)r],
                                     (a.u && off >= 0) ? a.u + off : nullptr, a.seed, a.site, (uint64_t)b);
        if (lane == 0) {
            a.run[b] = run;
            if (off >= 0) a.out[off] = token;
        }
        if (next < 0) next = token;
        if (a.probs_out) {
            __syncwarp();
            for (int i = lane; i < a.V; i += 32) a.probs_out[(int64_t)b * a.ldp + i] = s_p[warp][i];
        }
    }
    if (lane == 0 && next >= 0) a.cur[b] = next;  // every lane has read cur[b] above
}
}  // namespace

int tgan_set_step_ctr_sampling(const void* p) { return tgan_set_step_ctr_local(p); }

extern "C" int tgan_sample_tokens(const float* logits, int64_t ldl, const float* u, const uint8_t* suppress_empty,
                                  int64_t* ids, float* probs_out, int64_t ldp, int rows, int V, int exclude_bos,
                                  int empty_token, int mode, int topk, float top_p, float temperature, uint64_t seed,
                                  uint64_t site, void* stream) {
    if (rows <= 0) return 0;
    TGAN_CHECK_ARG(V >= 1 && V <= SMAXV && mode >= 0 && mode <= 2 && temperature >= 0.f,
                   "tgan_sample_tokens: 1 <= V <= 1024, mode in {0 random, 1 topk, 2 nucleus}, temperature >= 0");
    SampleArgs a;
    a.rows = rows; a.V = V; a.exclude_bos = exclude_bos; a.empty_token = empty_token; a.mode = mode; a.topk = topk;
    a.temperature = temperature; a.top_p = top_p; a.seed = seed; a.site = site;
    sample_kernel<<<ceil_div(rows, SW), SW * 32, 0, (cudaStream_t)stream>>>(logits, ldl, u, suppress_empty, ids, probs_out,
                                                                            ldp, a);
    TGAN_COUNT_LAUNCH();
    TGAN_LAUNCH_OK();
    return 0;
}

extern "C" int tgan_sample_step(const float* logits, int64_t ldl, const int32_t* req, const int32_t* start,
                                const int32_t* out_off, const int32_t* forced_next, const int32_t* req_i,
                                const float* req_f, const float* u, const int32_t* run0, int32_t* run, int64_t* cur,
                                int64_t* out, float* probs_out, int64_t ldp, int B, int V, int step, uint64_t seed,
                                uint64_t site, void* stream) {
    if (B <= 0) return 0;
    TGAN_CHECK_ARG(V >= 1 && V <= SMAXV, "tgan_sample_step: 1 <= V <= 1024");
    StepArgs a;
    a.logits = logits; a.ldl = ldl;
    a.req = req; a.start = start; a.out_off = out_off; a.forced_next = forced_next; a.req_i = req_i;
    a.req_f = req_f; a.u = u; a.run0 = run0;
    a.run = run; a.cur = cur; a.out = out; a.probs_out = probs_out; a.ldp = ldp;
    a.B = B; a.V = V; a.step = step; a.seed = seed; a.site = site;
    sample_step_kernel<<<ceil_div(B, SW), SW * 32, 0, (cudaStream_t)stream>>>(a);
    TGAN_COUNT_LAUNCH();
    TGAN_LAUNCH_OK();
    return 0;
}
