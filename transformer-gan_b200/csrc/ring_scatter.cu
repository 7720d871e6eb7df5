// Prefilled prompt rows into the windows of a request queue's ring (MemTransformerLM.generate_requests with
// context_pass=True).  A group of prompts is prefilled by one context pass into a ring of its own; at the step where a
// request starts, its rows are copied into its column of the queue's ring, right below the step's write position, in
// every layer-input slab and every projected-K/V layer: the memory a context pass over that prompt alone leaves behind.
// Descriptor i = (source column, first source position, destination column, rows).  Pure 16-byte copies, HBM-bound:
// rows * (n_slab * DP + n_kv * KW) * es bytes read and written per descriptor.
// Grid: (descriptor, plane = slab or K/V layer, chunk of RB rows); a CTA strides over the rows of its plane.
#include "common.cuh"

namespace {
constexpr int ST = 128;  // threads per CTA
constexpr int RB = 8;    // rows per CTA and chunk

struct ScatterArgs {
    const int32_t* desc;
    const uint4 *src_x, *src_kv;
    uint4 *dst_x, *dst_kv;
    int64_t src_xs, dst_xs, src_kvs, dst_kvs;  // slab / layer strides, in 16-byte vectors
    int xw, kvw;                               // row widths, in 16-byte vectors
    int n_slab, src_cols, dst_cols, dst_end;
};

__global__ void __launch_bounds__(ST) ring_scatter_kernel(ScatterArgs a) {
    const int4 d = reinterpret_cast<const int4*>(a.desc)[blockIdx.x];  // x src col, y src pos, z dst col, w rows
    const bool kv = (int)blockIdx.y >= a.n_slab;
    const int p = kv ? blockIdx.y - a.n_slab : blockIdx.y;
    const int w = kv ? a.kvw : a.xw;
    const uint4* __restrict__ src = kv ? a.src_kv + p * a.src_kvs : a.src_x + p * a.src_xs;
    uint4* __restrict__ dst = kv ? a.dst_kv + p * a.dst_kvs : a.dst_x + p * a.dst_xs;
    const int dst_pos = a.dst_end - d.w;
    for (int r0 = blockIdx.z * RB; r0 < d.w; r0 += gridDim.z * RB) {
        const int n = min(RB, d.w - r0) * w;
        for (int i = threadIdx.x; i < n; i += ST) {
            const int r = r0 + i / w, e = i - (i / w) * w;
            dst[((int64_t)(dst_pos + r) * a.dst_cols + d.z) * w + e] = src[((int64_t)(d.y + r) * a.src_cols + d.x) * w + e];
        }
    }
}
}  // namespace

extern "C" int tgan_ring_scatter(int dtype, const int32_t* desc, int n, int max_rows, int dst_end, const void* src_x,
                                 int64_t src_x_stride, void* dst_x, int64_t dst_x_stride, int n_slab, int DP,
                                 const void* src_kv, int64_t src_kv_stride, void* dst_kv, int64_t dst_kv_stride,
                                 int n_kv, int KW, int src_cols, int dst_cols, void* stream) {
    if (n <= 0 || max_rows <= 0 || n_slab + n_kv <= 0) return 0;
    TGAN_CHECK_ARG(dtype == TGAN_F32 || dtype == TGAN_BF16, "tgan_ring_scatter: bad dtype");
    const int es = dtype == TGAN_F32 ? 4 : 2, ve = 16 / es;  // elements per 16-byte vector
    TGAN_CHECK_ARG(n_slab >= 0 && n_kv >= 0 && n_slab + n_kv <= 65535 && src_cols >= 1 && dst_cols >= 1 &&
                       dst_end >= 0 && desc != nullptr && ((uintptr_t)desc & 15) == 0,
                   "tgan_ring_scatter: bad sizes or descriptor table (int32 [n][4], 16-byte aligned)");
    TGAN_CHECK_ARG(n_slab == 0 || (DP > 0 && DP % 64 == 0 && src_x && dst_x && ((uintptr_t)src_x & 15) == 0 &&
                                   ((uintptr_t)dst_x & 15) == 0 && src_x_stride % ve == 0 && dst_x_stride % ve == 0),
                   "tgan_ring_scatter: slab rows must be 16-byte aligned, DP a multiple of 64");
    TGAN_CHECK_ARG(n_kv == 0 || (KW > 0 && KW % 64 == 0 && src_kv && dst_kv && ((uintptr_t)src_kv & 15) == 0 &&
                                 ((uintptr_t)dst_kv & 15) == 0 && src_kv_stride % ve == 0 && dst_kv_stride % ve == 0),
                   "tgan_ring_scatter: K/V rows must be 16-byte aligned, KW a multiple of 64");
    ScatterArgs a;
    a.desc = desc;
    a.src_x = (const uint4*)src_x; a.dst_x = (uint4*)dst_x;
    a.src_kv = (const uint4*)src_kv; a.dst_kv = (uint4*)dst_kv;
    a.src_xs = src_x_stride / ve; a.dst_xs = dst_x_stride / ve;
    a.src_kvs = src_kv_stride / ve; a.dst_kvs = dst_kv_stride / ve;
    a.xw = DP / ve; a.kvw = KW / ve;
    a.n_slab = n_slab; a.src_cols = src_cols; a.dst_cols = dst_cols; a.dst_end = dst_end;
    const dim3 grid(n, n_slab + n_kv, min(ceil_div(max_rows, RB), 65535));
    ring_scatter_kernel<<<grid, ST, 0, (cudaStream_t)stream>>>(a);
    TGAN_COUNT_LAUNCH();
    TGAN_LAUNCH_OK();
    return 0;
}
