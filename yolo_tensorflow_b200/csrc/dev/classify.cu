// classify.cu — the classifier tail of darknet's ImageNet models (Darknet-19, Darknet-53): [avgpool] (forward_avgpool_layer),
// [softmax] (forward_softmax_layer -> softmax_cpu -> softmax of blas.c) and the top-k ranking predict_classifier applies to
// the probabilities (top_k of utils.c).  All three are launched with programmatic stream serialization like the tcgen05
// convolutions: a kernel may become resident while its predecessor drains and waits (pdl_wait) before its first read.
#include "kernels.h"
#include "softmax.cuh"
#include "tc_ptx.cuh"

static const int kThreads = 256;

template <typename... Params, typename... Args>
static void launch_pdl_kernel(void (*kernel)(Params...), dim3 grid, size_t smem, cudaStream_t s, Args... args)
{
    static const bool no_pdl = getenv("B200_NO_PDL") != nullptr;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid;
    cfg.blockDim = dim3(kThreads);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = s;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = no_pdl ? 0 : 1;
    B200_CHECK(cudaLaunchKernelEx(&cfg, kernel, ((Params)args)...));
    B200_LAUNCHED();
}

// ---------------------------------------------------------------------------------------------------
// [avgpool]: out[b][c] = (sum over the h*w pixels of in[b][y][x][c]) / (h*w), fp32 sum.  A CTA takes one image and a slice of
// 32 channel vectors (16 bytes each: 8 bf16 or 4 fp32 channels); its 8 warps split the pixels and add their partial sums in
// shared memory.  The sum order differs from the reference's pixel-by-pixel loop: within fp32 rounding.
// ---------------------------------------------------------------------------------------------------
template <typename T, typename U, bool VEC>
__global__ void __launch_bounds__(kThreads) avgpool_kernel(const T *__restrict__ in, U *__restrict__ out, int hw, int c, int ld, int ldo)
{
    constexpr int V = VEC ? Elem<T>::VEC : 1;
    __shared__ float part[kThreads / 32][32 * V];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, b = blockIdx.y;
    const int c0 = (blockIdx.x * 32 + lane) * V;
    pdl_launch_dependents();
    pdl_wait();
    float acc[V];
#pragma unroll
    for (int k = 0; k < V; ++k) acc[k] = 0.f;
    if (c0 < c) {
        const T *src = in + (size_t)b * hw * ld + c0;
        for (int p = warp; p < hw; p += kThreads / 32) {
            float v[V];
            if (VEC) load_vec<T>(src + (size_t)p * ld, v);
            else v[0] = Elem<T>::load(src + (size_t)p * ld);
#pragma unroll
            for (int k = 0; k < V; ++k) acc[k] += v[k];
        }
    }
#pragma unroll
    for (int k = 0; k < V; ++k) part[warp][lane * V + k] = acc[k];
    __syncthreads();
    if (warp == 0 && c0 < c) {
        float r[V];
#pragma unroll
        for (int k = 0; k < V; ++k) {
            float t = 0.f;
            for (int w = 0; w < kThreads / 32; ++w) t += part[w][lane * V + k];
            r[k] = t / (float)hw;                                                   // avgpool_layer.c: output /= l.h*l.w
        }
        U *dst = out + (size_t)b * ldo + c0;
        if constexpr (VEC && sizeof(U) == sizeof(T)) store_vec<U>(dst, r);
        else
            for (int k = 0; k < V; ++k) Elem<U>::store(dst + k, r[k]);
    }
}

template <typename T, typename U>
static void avgpool_typed(TView in, TView out, cudaStream_t s)
{
    const int hw = in.h * in.w;
    const bool vec = in.c % Elem<T>::VEC == 0 && in.ld % Elem<T>::VEC == 0 && ((uintptr_t)in.p & 15) == 0 &&
                     (sizeof(U) != sizeof(T) || (out.ld % Elem<T>::VEC == 0 && ((uintptr_t)out.p & 15) == 0));
    const int per_cta = 32 * (vec ? Elem<T>::VEC : 1);
    const dim3 grid(div_up(in.c, per_cta), in.n);
    if (vec) launch_pdl_kernel(avgpool_kernel<T, U, true>, grid, 0, s, (const T *)in.p, (U *)out.p, hw, in.c, in.ld, out.ld);
    else launch_pdl_kernel(avgpool_kernel<T, U, false>, grid, 0, s, (const T *)in.p, (U *)out.p, hw, in.c, in.ld, out.ld);
}

void launch_avgpool(TView in, TView out, cudaStream_t s)
{
    if (in.dtype == DT_BF16 && out.dtype == DT_BF16) avgpool_typed<bf16, bf16>(in, out, s);
    else if (in.dtype == DT_BF16) avgpool_typed<bf16, float>(in, out, s);
    else if (out.dtype == DT_BF16) avgpool_typed<float, bf16>(in, out, s);
    else avgpool_typed<float, float>(in, out, s);
}

// ---------------------------------------------------------------------------------------------------
// [softmax]: one CTA per (image, group) runs softmax() of blas.c (group_softmax, shared with the [region] head) over the
// group's `n` values; input element j of image b at in[b*ld + g*n + j], output fp32 [b][groups*n].
// ---------------------------------------------------------------------------------------------------
__device__ __forceinline__ float block_all(float v, bool is_max)
{
    __shared__ float red[kThreads / 32];
    __shared__ float result;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    v = is_max ? warp_all_max(v) : warp_all_sum(v);
    if (lane == 0) red[warp] = v;
    __syncthreads();
    if (warp == 0) {
        float t = lane < kThreads / 32 ? red[lane] : (is_max ? -FLT_MAX : 0.f);
        t = is_max ? warp_all_max(t) : warp_all_sum(t);
        if (lane == 0) result = t;
    }
    __syncthreads();
    const float r = result;
    __syncthreads();                                       // red / result are reused by the next call
    return r;
}

template <typename T>
__global__ void __launch_bounds__(kThreads) softmax_kernel(const T *__restrict__ in, float *__restrict__ out, int n, int groups, int ld, float temp)
{
    const int b = blockIdx.x / groups, g = blockIdx.x % groups;
    const T *src = in + (size_t)b * ld + (size_t)g * n;
    float *dst = out + ((size_t)b * groups + g) * n;
    pdl_launch_dependents();
    pdl_wait();
    group_softmax(n, temp, (int)threadIdx.x, kThreads, [&](int j) { return Elem<T>::load(src + j); },
                  [&](int j) -> float & { return dst[j]; }, [](float v) { return block_all(v, true); },
                  [](float v) { return block_all(v, false); });
}

void launch_softmax(TView in, float *out, int batch, int groups, float temp, cudaStream_t s)
{
    const int n = in.c / groups;
    if (in.dtype == DT_F32) launch_pdl_kernel(softmax_kernel<float>, dim3(batch * groups), 0, s, (const float *)in.p, out, n, groups, in.ld, temp);
    else launch_pdl_kernel(softmax_kernel<bf16>, dim3(batch * groups), 0, s, (const bf16 *)in.p, out, n, groups, in.ld, temp);
}

// ---------------------------------------------------------------------------------------------------
// top_k of utils.c on every row: index[j] = -1; for i: curr = i; for j < k: if (index[j] < 0 || a[curr] > a[index[j]])
// swap(curr, index[j]).  The result is that loop's, equal values included (a displaced entry moves on only past strictly
// smaller ones, so ties do not always keep index order).  One CTA per row:
//   1. the k-th largest value t (as an order-preserving key, -0 folded into +0) by bisection over the 32 key bits, each step
//      one block-wide count;
//   2. the loop itself, run by one thread over the candidates a[i] >= t only, in index order.  Entries below t never move an
//      entry >= t: an insertion only shifts entries smaller than the inserted value, and the slot an entry >= t lands in is
//      the first one holding a smaller value or nothing — the same whether that slot held an entry below t or was empty.
//      So the loop over the candidates leaves the same list as the loop over the whole row.
// With distinct values there are exactly k candidates; a row of n equal values makes all n of them candidates.
// ---------------------------------------------------------------------------------------------------
__device__ __forceinline__ unsigned order_key(float x)
{
    unsigned u = __float_as_uint(x + 0.f);                 // -0 + 0 = +0: equal under `>`, equal keys
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}

__global__ void __launch_bounds__(kThreads) topk_kernel(const float *__restrict__ a, int n, int ld, int k, int *__restrict__ classes,
                                                        float *__restrict__ probs)
{
    __shared__ int count;
    __shared__ int index[64];
    const float *row = a + (size_t)blockIdx.x * ld;
    pdl_launch_dependents();
    pdl_wait();
    unsigned t = 0;
    for (int bit = 31; bit >= 0; --bit) {
        const unsigned probe = t | (1u << bit);
        int mine = 0;
        for (int i = threadIdx.x; i < n; i += kThreads) mine += order_key(row[i]) >= probe;
        if (threadIdx.x == 0) count = 0;
        __syncthreads();
        if (mine) atomicAdd(&count, mine);
        __syncthreads();
        if (count >= k) t = probe;
        __syncthreads();
    }
    if (threadIdx.x < 32) {                                // warp 0 walks the row in index order, lane 0 inserts
        const int lane = threadIdx.x;
        if (lane == 0) for (int j = 0; j < k; ++j) index[j] = -1;
        __syncwarp();
        for (int base = 0; base < n; base += 32) {
            const int i = base + lane;
            unsigned hits = __ballot_sync(0xffffffffu, i < n && order_key(row[i]) >= t);
            if (lane == 0)
                while (hits) {
                    int curr = base + __ffs(hits) - 1;
                    hits &= hits - 1;
                    for (int j = 0; j < k; ++j)
                        if (index[j] < 0 || row[curr] > row[index[j]]) { const int swap = curr; curr = index[j]; index[j] = swap; }
                }
            __syncwarp();
        }
        for (int j = lane; j < k; j += 32) {
            const int c = index[j];
            classes[(size_t)blockIdx.x * k + j] = c;
            if (probs) probs[(size_t)blockIdx.x * k + j] = c >= 0 ? row[c] : 0.f;
        }
    }
}

void launch_topk(const float *a, int rows, int n, int ld, int k, int *classes, float *probs, cudaStream_t s)
{
    launch_pdl_kernel(topk_kernel, dim3(rows), 0, s, a, n, ld, k, classes, probs);
}
