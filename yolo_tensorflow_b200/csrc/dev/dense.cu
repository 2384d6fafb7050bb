// dense.cu — YOLOv1's two weight-bandwidth-bound layers.
//
//  * local (unshared 3x3 convolution, local_layer.c:91-120): every output location owns a [filters][size*size*c]
//    weight block; out[b][o][loc] = bias[o][loc] + sum_k W[loc][o][k] * col[k][loc], then the activation.
//  * connected (connected_layer.c:151-167): out[b][o] = sum_i in[b][i]*W[o][i], then scale/shift, activation.
//
// Both stream their weights exactly once per group of BT images: one warp owns one weight row, lanes stride the
// row with 16-byte loads (fully coalesced), and BT accumulators per lane reuse every weight vector across the
// batch group; a shuffle tree finishes the dot products.  Algorithmic bytes = the weight matrix once per batch
// (231 MB bf16 for the YOLOv1 local layer, 43 MB for the connected layer) + activations.
#include "kernels.h"

#define DENSE_BT 8

template <typename T> __device__ __forceinline__ void fma_vec(const float *w, const T *x, float &acc)
{
    float v[Elem<T>::VEC];
    load_vec<T>(x, v);
#pragma unroll
    for (int i = 0; i < Elem<T>::VEC; ++i) acc = fmaf(w[i], v[i], acc);
}

__device__ __forceinline__ float warp_sum(float v)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// ---- local ---------------------------------------------------------------------------------------------
// weights repacked to [loc][o][(ky,kx,c)] (same dtype as activations); bias transposed to [loc][o] fp32 at upload
template <typename T, bool EXACT>
__global__ void __launch_bounds__(256)
local_kernel(const T *__restrict__ in, int N, int H, int W, int C, int ldi, T *__restrict__ out, int OH, int OW, int ldo,
             int F, const T *__restrict__ wt, const float *__restrict__ bias, int size, int stride, int pad, int act)
{
    constexpr int V = Elem<T>::VEC;
    const int lane = threadIdx.x & 31;
    const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int locations = OH * OW;
    if (warp >= locations * F) return;
    const int loc = warp / F, o = warp % F;
    const int oy = loc / OW, ox = loc % OW;
    const int K = size * size * C;
    const T *wrow = wt + ((size_t)loc * F + o) * K;
    for (int b0 = 0; b0 < N; b0 += DENSE_BT) {
        float acc[DENSE_BT];
#pragma unroll
        for (int i = 0; i < DENSE_BT; ++i) acc[i] = 0.f;
        for (int ky = 0; ky < size; ++ky) {
            int y = oy * stride + ky - pad;
            if (y < 0 || y >= H) continue;
            for (int kx = 0; kx < size; ++kx) {
                int x = ox * stride + kx - pad;
                if (x < 0 || x >= W) continue;
                const T *wtap = wrow + (size_t)(ky * size + kx) * C;
                for (int c = lane * V; c < C; c += 32 * V) {
                    float wv[V];
                    load_vec<T>(wtap + c, wv);
#pragma unroll
                    for (int i = 0; i < DENSE_BT; ++i)
                        if (b0 + i < N) fma_vec<T>(wv, in + (((size_t)(b0 + i) * H + y) * W + x) * ldi + c, acc[i]);
                }
            }
        }
#pragma unroll
        for (int i = 0; i < DENSE_BT; ++i) {
            float v = warp_sum(acc[i]);
            if (lane == 0 && b0 + i < N)
                Elem<T>::store(out + ((size_t)(b0 + i) * locations + loc) * ldo + o, apply_act<EXACT>(v + bias[(size_t)loc * F + o], act));
        }
    }
}

void launch_local(TView in, TView out, const void *w, const float *bias, int size, int stride, int pad, int act, cudaStream_t s)
{
    long long warps = (long long)out.h * out.w * out.c;
    int grid = div_up(warps * 32, 256);
    if (in.c % Elem<bf16>::VEC != 0 || in.ld % Elem<bf16>::VEC != 0) { fprintf(stderr, "b200-darknet: local layer needs C %% 8 == 0\n"); abort(); }
    if (in.dtype == DT_F32)
        local_kernel<float, true><<<grid, 256, 0, s>>>((const float *)in.p, in.n, in.h, in.w, in.c, in.ld, (float *)out.p, out.h, out.w, out.ld,
                                                         out.c, (const float *)w, bias, size, stride, pad, act);
    else
        local_kernel<bf16, false><<<grid, 256, 0, s>>>((const bf16 *)in.p, in.n, in.h, in.w, in.c, in.ld, (bf16 *)out.p, out.h, out.w, out.ld,
                                                         out.c, (const bf16 *)w, bias, size, stride, pad, act);
    B200_LAUNCHED();
}

// ---- connected -------------------------------------------------------------------------------------------
// TI = input, TW = weights.  They differ after another [connected] (or [softmax]) in bf16 mode: those layers write fp32 rows.
template <typename TI, typename TW, bool EXACT>
__global__ void __launch_bounds__(256)
connected_kernel(const TI *__restrict__ in, int N, int K, int O, const TW *__restrict__ wt, const float *__restrict__ scale,
                 const float *__restrict__ shift, int act, float *__restrict__ out)
{
    constexpr int V = Elem<TW>::VEC, VI = Elem<TI>::VEC;
    static_assert(V % VI == 0, "one weight vector spans whole input vectors");
    const int lane = threadIdx.x & 31;
    const int o = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (o >= O) return;
    const TW *wrow = wt + (size_t)o * K;
    const int Kv = K - K % V;
    for (int b0 = 0; b0 < N; b0 += DENSE_BT) {
        float acc[DENSE_BT];
#pragma unroll
        for (int i = 0; i < DENSE_BT; ++i) acc[i] = 0.f;
        for (int k = lane * V; k < Kv; k += 32 * V) {
            float wv[V];
            load_vec<TW>(wrow + k, wv);
#pragma unroll
            for (int i = 0; i < DENSE_BT; ++i)
                if (b0 + i < N)
#pragma unroll
                    for (int j = 0; j < V; j += VI) fma_vec<TI>(wv + j, in + (size_t)(b0 + i) * K + k + j, acc[i]);
        }
        for (int k = Kv + lane; k < K; k += 32) {               // scalar tail when K is not a multiple of the vector width
            float wv = Elem<TW>::load(wrow + k);
#pragma unroll
            for (int i = 0; i < DENSE_BT; ++i)
                if (b0 + i < N) acc[i] = fmaf(wv, Elem<TI>::load(in + (size_t)(b0 + i) * K + k), acc[i]);
        }
#pragma unroll
        for (int i = 0; i < DENSE_BT; ++i) {
            float v = warp_sum(acc[i]);
            if (lane == 0 && b0 + i < N) out[(size_t)(b0 + i) * O + o] = apply_act<EXACT>(fmaf(v, scale[o], shift[o]), act);
        }
    }
}

void launch_connected(const void *in, int in_dtype, int batch, int inputs, int outputs, const void *w, int w_dtype,
                      const float *scale, const float *shift, int act, float *out, cudaStream_t s)
{
    int grid = div_up((long long)outputs * 32, 256);
    bool aligned = ((uintptr_t)in % 16 == 0) && ((uintptr_t)w % 16 == 0) && (inputs % Elem<bf16>::VEC == 0);
    if (!aligned) { fprintf(stderr, "b200-darknet: connected layer needs 16-byte aligned rows (inputs %% 8 == 0)\n"); abort(); }
    if (in_dtype == DT_F32 && w_dtype == DT_F32)
        connected_kernel<float, float, true><<<grid, 256, 0, s>>>((const float *)in, batch, inputs, outputs, (const float *)w, scale, shift, act, out);
    else if (in_dtype == DT_BF16 && w_dtype == DT_BF16)
        connected_kernel<bf16, bf16, false><<<grid, 256, 0, s>>>((const bf16 *)in, batch, inputs, outputs, (const bf16 *)w, scale, shift, act, out);
    else if (in_dtype == DT_F32 && w_dtype == DT_BF16)
        connected_kernel<float, bf16, false><<<grid, 256, 0, s>>>((const float *)in, batch, inputs, outputs, (const bf16 *)w, scale, shift, act, out);
    else { fprintf(stderr, "b200-darknet: connected layer: unsupported input / weight dtype pair\n"); abort(); }
    B200_LAUNCHED();
}

// [rows][ld] fp32 -> dense [rows][cols]: the tcgen05 connected layer computes into 64-filter-padded rows
__global__ void unpad_rows_f32_kernel(const float *__restrict__ src, int ld, float *__restrict__ dst, int cols, long long total)
{
    for (long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x; t < total; t += (long long)gridDim.x * blockDim.x)
        dst[t] = src[(t / cols) * ld + t % cols];
}

void launch_unpad_rows_f32(const float *src, int ld, float *dst, int cols, int rows, cudaStream_t s)
{
    long long total = (long long)rows * cols;
    int grid = (int)((total + 255) / 256); if (grid > 148 * 8) grid = 148 * 8;
    unpad_rows_f32_kernel<<<grid, 256, 0, s>>>(src, ld, dst, cols, total);
    B200_LAUNCHED();
}
