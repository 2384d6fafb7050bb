// softmax.cuh — softmax() of blas.c with darknet's arithmetic, shared by the [region] head (heads.cu, one warp per box) and
// the classifier's [softmax] layer (classify.cu, one CTA per image and group).
#pragma once
#include "common.cuh"
#include <cfloat>

// The n values of one group, spread over `lanes` threads (this one is `lane`): largest, e = exp(x/temp - largest/temp)
// evaluated in double and stored as float, fp32 sum, divide.  in(j) reads value j, out(j) is where probability j goes (it
// holds e until the divide); all_max / all_sum combine one value per thread across the `lanes` threads and return the
// result to every one of them.  The sum is taken in the order of those reductions instead of index order: within fp32
// rounding of the reference.  With temp = 1 the divisions are exact, x/1 == x.
template <typename In, typename Out, typename AllMax, typename AllSum>
__device__ __forceinline__ void group_softmax(int n, float temp, int lane, int lanes, In in, Out out, AllMax all_max, AllSum all_sum)
{
    float largest = -FLT_MAX;
    for (int j = lane; j < n; j += lanes) largest = fmaxf(largest, in(j));
    largest = all_max(largest);
    float sum = 0.f;
    for (int j = lane; j < n; j += lanes) {
        const float e = (float)exp((double)(in(j) / temp - largest / temp));
        sum += e;
        out(j) = e;
    }
    sum = all_sum(sum);
    for (int j = lane; j < n; j += lanes) out(j) /= sum;
}

__device__ __forceinline__ float warp_all_max(float v)
{
    for (int o = 16; o; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}
__device__ __forceinline__ float warp_all_sum(float v)
{
    for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
