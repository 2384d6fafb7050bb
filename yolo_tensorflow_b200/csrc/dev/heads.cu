// heads.cu — forward_yolo_layer / forward_region_layer / forward_detection_layer (inference part) on device.
//
// Input: the linear head convolution's NHWC logits.  Output: the layer's `l.output` in DARKNET layout
// (fp32, per image [anchor][entry][h*w], entry_index() of yolo_layer.c:125-130 / region_layer.c:151-156),
// with the reference's activations applied: LOGISTIC in double precision on x,y and obj(+classes)
// (yolo_layer.c:137-146, region_layer.c:163-172, activations.h:32), raw w,h, and the strided class softmax
// of the region layer (region_layer.c:182-185 -> blas.c:305-332).  The NHWC->NCHW transpose is fused into
// the same pass, so logits are read once and activations written once: 2 x outputs x 4 bytes of HBM traffic.
#include "kernels.h"
#include "softmax.cuh"
#include <cfloat>

static const int kThreads = 256;

__device__ __forceinline__ float logistic_ref(float x) { return (float)(1. / (1. + exp(-(double)x))); }

// 32x32 shared-memory transpose tiles: per (image, anchor) the [HW][entries] NHWC slab becomes the
// [entries][HW] darknet slab, so both the logits read (entry fastest) and the activation write (cell fastest)
// are coalesced; the logistic is applied on the way through.
template <typename T>
__global__ void yolo_forward_kernel(const T *__restrict__ in, float *__restrict__ out, int HW, int ld, int anchors, int entries)
{
    __shared__ float tile[32][33];
    const int n = blockIdx.z / anchors, a = blockIdx.z % anchors;
    const int p0 = blockIdx.x * 32, e0 = blockIdx.y * 32;
    const T *src = in + (size_t)n * HW * ld + a * entries;
    float *dst = out + ((size_t)n * anchors + a) * entries * HW;
    for (int i = threadIdx.y; i < 32; i += blockDim.y) {
        int p = p0 + i, e = e0 + threadIdx.x;
        tile[i][threadIdx.x] = (p < HW && e < entries) ? Elem<T>::load(src + (size_t)p * ld + e) : 0.f;
    }
    __syncthreads();
    for (int i = threadIdx.y; i < 32; i += blockDim.y) {
        int e = e0 + i, p = p0 + threadIdx.x;
        if (e < entries && p < HW) {
            float v = tile[threadIdx.x][i];
            if (e != 2 && e != 3) v = logistic_ref(v);
            dst[(size_t)e * HW + p] = v;
        }
    }
}

void launch_yolo_forward(TView in, float *out, int anchors, int classes, cudaStream_t s)
{
    int HW = in.h * in.w, entries = classes + 5;
    dim3 grid(div_up(HW, 32), div_up(entries, 32), in.n * anchors), block(32, 8);
    if (in.dtype == DT_F32) yolo_forward_kernel<float><<<grid, block, 0, s>>>((const float *)in.p, out, HW, in.ld, anchors, entries);
    else yolo_forward_kernel<bf16><<<grid, block, 0, s>>>((const bf16 *)in.p, out, HW, in.ld, anchors, entries);
    B200_LAUNCHED();
}

// detection (YOLOv1): plain copy of the connected layer's fp32 output, optional per-cell class softmax
__global__ void detection_forward_kernel(const float *__restrict__ in, float *__restrict__ out, int batch, int outputs,
                                         int side, int classes, int softmax)
{
    const long long total = (long long)batch * outputs;
    if (!softmax) {      // pass 0: copy
        for (long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x; t < total; t += (long long)gridDim.x * blockDim.x) out[t] = in[t];
        return;
    }
    // pass 1 (separate launch): per-cell class softmax, one thread per (image, cell)
    const long long cells = (long long)batch * side * side;
    for (long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x; t < cells; t += (long long)gridDim.x * blockDim.x) {
        int b = (int)(t / (side * side)), i = (int)(t % (side * side));
        const float *src = in + (size_t)b * outputs + i * classes;
        float *dst = out + (size_t)b * outputs + i * classes;
        float largest = -FLT_MAX;
        for (int j = 0; j < classes; ++j) if (src[j] > largest) largest = src[j];
        float sum = 0;
        for (int j = 0; j < classes; ++j) { float e = (float)exp((double)(src[j] - largest)); sum += e; dst[j] = e; }
        for (int j = 0; j < classes; ++j) dst[j] /= sum;
    }
}

void launch_detection_forward(const float *in, float *out, int batch, int outputs, int side, int classes, int softmax, cudaStream_t s)
{
    long long total = (long long)batch * outputs;
    int grid = (int)((total + kThreads - 1) / kThreads);
    if (grid > 148 * 8) grid = 148 * 8;
    if (softmax) {
        // two dependent passes over the same buffer: run the softmax pass as its own launch to stay race-free
        detection_forward_kernel<<<grid, kThreads, 0, s>>>(in, out, batch, outputs, side, classes, 0);
        B200_LAUNCHED();
        detection_forward_kernel<<<grid, kThreads, 0, s>>>(in, out, batch, outputs, side, classes, 1);
        B200_LAUNCHED();
    } else {
        detection_forward_kernel<<<grid, kThreads, 0, s>>>(in, out, batch, outputs, side, classes, 0);
        B200_LAUNCHED();
    }
}

// batch == 2 flip-averaging of `detector valid2` (avg_flipped_yolo, yolo_layer.c:290-314; the same loop inlined in
// get_region_detections, region_layer.c:368-390), IN PLACE like the reference: item 1 (the mirrored image) is flipped back
// horizontally, item 0 becomes the mean of the two.  The reference indexes the planes as [z][n] while l.output is laid out
// [n][z]; both enumerate every plane once, so the flip is layout-independent, but the sign change it applies "for z == 0"
// lands on the FIRST l.n planes of the buffer (not on each anchor's x entry) and skips the middle column of an odd width —
// reproduced as is.  Two launches: the average reads what the flip wrote.
__global__ void flip_item_kernel(float *__restrict__ flip, int w, int h, int planes, int neg_planes)
{
    const int half = w / 2;
    const long long total = (long long)planes * h * half;
    for (long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x; t < total; t += (long long)gridDim.x * blockDim.x) {
        const int i = (int)(t % half), j = (int)((t / half) % h), p = (int)(t / ((long long)half * h));
        float *row = flip + ((size_t)p * h + j) * w;
        float a = row[i], b = row[w - i - 1];
        if (p < neg_planes) { a = -a; b = -b; }
        row[i] = b; row[w - i - 1] = a;
    }
}

__global__ void average_items_kernel(float *__restrict__ out, const float *__restrict__ flip, int outputs)
{
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < outputs; i += gridDim.x * blockDim.x)
        out[i] = (float)((double)__fadd_rn(out[i], flip[i]) / 2.);
}

void launch_avg_flipped(float *head_out, int w, int h, int anchors, int entries, int outputs, cudaStream_t s)
{
    const int planes = anchors * entries;
    const long long swaps = (long long)planes * h * (w / 2);
    if (swaps > 0) {
        flip_item_kernel<<<(int)((swaps + kThreads - 1) / kThreads), kThreads, 0, s>>>(head_out + outputs, w, h, planes, anchors);
        B200_LAUNCHED();
    }
    average_items_kernel<<<div_up(outputs, kThreads), kThreads, 0, s>>>(head_out, head_out + outputs, outputs);
    B200_LAUNCHED();
}

// ---------------------------------------------------------------------------------------------------
// YOLO9000: [region] with a WordTree (SURVEY §8f-4).  forward_region_layer's softmax_tree branch as the reference's GPU build
// runs it (region_layer.c:455-457 -> softmax_tree, blas_kernels.cu): per box, one softmax over every sibling group of the
// tree at temperature 1, class entries strided by h*w.  (The reference's CPU build cannot run this branch: it divides by
// l.temperature, which parse_region never sets — region_layer.c:179 — so every class probability comes out NaN there.)
// One warp per box: the box's logits are contiguous in the NHWC input.
// ---------------------------------------------------------------------------------------------------
// The same kernel serves the plain region head (gsize == nullptr): one group over all classes when softmax = 1
// (region_layer.c:182-185 -> blas.c:305-321), a logistic on every class otherwise (:171).
template <typename T>
__global__ void region_forward_kernel(const T *__restrict__ in, float *__restrict__ out, int N, int HW, int ld, int anchors,
                                           int classes, int coords, const int *__restrict__ gsize, const int *__restrict__ goff, int groups,
                                           int softmax)
{
    const int entries = coords + 1 + classes;
    const int lane = threadIdx.x & 31, warps = blockDim.x >> 5;
    const long long total = (long long)N * anchors * HW;
    for (long long t = (long long)blockIdx.x * warps + (threadIdx.x >> 5); t < total; t += (long long)gridDim.x * warps) {
        const int loc = (int)(t % HW), a = (int)((t / HW) % anchors), n = (int)(t / ((long long)HW * anchors));
        const T *src = in + ((size_t)n * HW + loc) * ld + a * entries;
        float *dst = out + ((size_t)n * anchors + a) * entries * HW + loc;
        if (lane == 0) {
            dst[0] = logistic_ref(Elem<T>::load(src + 0));
            dst[HW] = logistic_ref(Elem<T>::load(src + 1));
            for (int e = 2; e < coords; ++e) dst[(size_t)e * HW] = Elem<T>::load(src + e);
            dst[(size_t)coords * HW] = logistic_ref(Elem<T>::load(src + coords));
        }
        if (!softmax) {
            for (int j = lane; j < classes; j += 32) dst[(size_t)(coords + 1 + j) * HW] = logistic_ref(Elem<T>::load(src + coords + 1 + j));
            continue;
        }
        for (int g = 0; g < groups; ++g) {
            const int off = coords + 1 + (gsize ? goff[g] : 0), sz = gsize ? gsize[g] : classes;
            group_softmax(sz, 1.f, lane, 32, [&](int j) { return Elem<T>::load(src + off + j); },
                          [&](int j) -> float & { return dst[(size_t)(off + j) * HW]; }, warp_all_max, warp_all_sum);
        }
    }
}


// Tiled variant for heads whose entries fit shared memory (YOLOv2: 85 per box): a CTA takes 32 consecutive cells of one (image,
// anchor); each warp reads its boxes' logits coalesced (lanes over entries), the activations go into a [entries][32 cells] tile,
// and the tile leaves with lanes over CELLS, i.e. as full 128-byte lines of the darknet layout.  (ncu, round 2: thread-per-box
// reads were uncoalesced, 69 us for 37 MB; warp-per-box with direct stores wrote one sector per lane, 148 us.)
template <typename T>
__global__ void __launch_bounds__(256)
region_forward_tiled_kernel(const T *__restrict__ in, float *__restrict__ out, int N, int HW, int ld, int anchors, int classes, int coords,
                            const int *__restrict__ gsize, const int *__restrict__ goff, int groups, int softmax, int tiles_per_plane)
{
    extern __shared__ float tile[];                              // [entries][33]
    const int entries = coords + 1 + classes;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const long long total = (long long)N * anchors * tiles_per_plane;
    for (long long t = blockIdx.x; t < total; t += gridDim.x) {
        const int tl = (int)(t % tiles_per_plane), a = (int)((t / tiles_per_plane) % anchors), n = (int)(t / ((long long)tiles_per_plane * anchors));
        const int loc0 = tl * 32, cells = (HW - loc0) < 32 ? (HW - loc0) : 32;
        for (int b = warp; b < cells; b += 8) {
            const T *src = in + ((size_t)n * HW + loc0 + b) * ld + a * entries;
            for (int e = lane; e <= coords; e += 32) {
                const float v = Elem<T>::load(src + e);
                tile[e * 33 + b] = (e < 2 || e == coords) ? logistic_ref(v) : v;
            }
            if (!softmax) {
                for (int j = lane; j < classes; j += 32) tile[(coords + 1 + j) * 33 + b] = logistic_ref(Elem<T>::load(src + coords + 1 + j));
                continue;
            }
            for (int g = 0; g < groups; ++g) {
                const int off = coords + 1 + (gsize ? goff[g] : 0), sz = gsize ? gsize[g] : classes;
                group_softmax(sz, 1.f, lane, 32, [&](int j) { return Elem<T>::load(src + off + j); },
                              [&](int j) -> float & { return tile[(off + j) * 33 + b]; }, warp_all_max, warp_all_sum);
            }
        }
        __syncthreads();
        float *dst = out + ((size_t)n * anchors + a) * entries * HW + loc0;
        for (int e = warp; e < entries; e += 8)
            if (lane < cells) dst[(size_t)e * HW + lane] = tile[e * 33 + lane];
        __syncthreads();
    }
}

template <typename T>
static bool region_forward_tiled(TView in, float *out, int anchors, int classes, int coords, const int *gsize, const int *goff, int groups,
                                 int softmax, cudaStream_t s)
{
    const int entries = coords + 1 + classes;
    const size_t smem = (size_t)entries * 33 * sizeof(float);
    if (smem > 48 * 1024) return false;                          // YOLO9000-sized heads keep the direct-store kernel
    const int HW = in.h * in.w, tiles = (HW + 31) / 32;
    long long total = (long long)in.n * anchors * tiles;
    int grid = (int)(total < 148 * 8 ? total : 148 * 8);
    region_forward_tiled_kernel<T><<<grid, 256, smem, s>>>((const T *)in.p, out, in.n, HW, in.ld, anchors, classes, coords, gsize, goff, groups, softmax, tiles);
    B200_LAUNCHED();
    return true;
}

void launch_region_tree_forward(TView in, float *out, int anchors, int classes, int coords, const int *gsize, const int *goff, int groups, cudaStream_t s)
{
    if (in.dtype == DT_F32 ? region_forward_tiled<float>(in, out, anchors, classes, coords, gsize, goff, groups, 1, s)
                           : region_forward_tiled<bf16>(in, out, anchors, classes, coords, gsize, goff, groups, 1, s)) return;
    const int HW = in.h * in.w;
    const long long boxes = (long long)in.n * anchors * HW;
    int grid = (int)((boxes + 7) / 8);
    if (grid > 148 * 16) grid = 148 * 16;
    if (in.dtype == DT_F32) region_forward_kernel<float><<<grid, kThreads, 0, s>>>((const float *)in.p, out, in.n, HW, in.ld, anchors, classes, coords, gsize, goff, groups, 1);
    else region_forward_kernel<bf16><<<grid, kThreads, 0, s>>>((const bf16 *)in.p, out, in.n, HW, in.ld, anchors, classes, coords, gsize, goff, groups, 1);
    B200_LAUNCHED();
}

// plain [region] head (YOLOv2): the tiled kernel above; the direct-store warp-per-box kernel only for heads too wide for a tile
void launch_region_forward(TView in, float *out, int anchors, int classes, int coords, int softmax, cudaStream_t s)
{
    if (in.dtype == DT_F32 ? region_forward_tiled<float>(in, out, anchors, classes, coords, nullptr, nullptr, 1, softmax, s)
                           : region_forward_tiled<bf16>(in, out, anchors, classes, coords, nullptr, nullptr, 1, softmax, s)) return;
    const int HW = in.h * in.w;
    const long long boxes = (long long)in.n * anchors * HW;
    int grid = (int)((boxes + 7) / 8);
    if (grid > 148 * 16) grid = 148 * 16;
    if (in.dtype == DT_F32) region_forward_kernel<float><<<grid, kThreads, 0, s>>>((const float *)in.p, out, in.n, HW, in.ld, anchors, classes, coords, nullptr, nullptr, 1, softmax);
    else region_forward_kernel<bf16><<<grid, kThreads, 0, s>>>((const bf16 *)in.p, out, in.n, HW, in.ld, anchors, classes, coords, nullptr, nullptr, 1, softmax);
    B200_LAUNCHED();
}

// hierarchy_predictions (tree.c:37-51): predictions[j] *= predictions[parent[j]] for j ascending, i.e. class j ends up as the
// product of the conditional probabilities along its path, associated from the root down: rel[j] * (rel[parent] * (...)).
// One thread per (box, class) walks up to the root, then multiplies back down in that association — bit-identical to the
// serial in-place loop.  Out of place into tmp, then copied back (the walk reads the unmodified values).
#define B200_TREE_MAX_DEPTH 64
__global__ void region_hierarchy_kernel(const float *__restrict__ pred, float *__restrict__ tmp, int hw, int anchors, int classes, int coords,
                                        const int *__restrict__ parent)
{
    const int entries = coords + 1 + classes;
    const long long total = (long long)anchors * classes * hw;
    for (long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x; t < total; t += (long long)gridDim.x * blockDim.x) {
        const int loc = (int)(t % hw), j = (int)((t / hw) % classes), a = (int)(t / ((long long)hw * classes));
        const float *p = pred + ((size_t)a * entries + coords + 1) * hw + loc;
        int chain[B200_TREE_MAX_DEPTH], depth = 0;
        for (int c = j; c >= 0 && depth < B200_TREE_MAX_DEPTH; c = parent[c]) chain[depth++] = c;
        float v = p[(size_t)chain[depth - 1] * hw];
        for (int k = depth - 2; k >= 0; --k) v = __fmul_rn(p[(size_t)chain[k] * hw], v);
        tmp[t] = v;
    }
}

__global__ void region_hierarchy_store_kernel(float *__restrict__ pred, const float *__restrict__ tmp, int hw, int anchors, int classes, int coords)
{
    const int entries = coords + 1 + classes;
    const long long total = (long long)anchors * classes * hw;
    for (long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x; t < total; t += (long long)gridDim.x * blockDim.x) {
        const int loc = (int)(t % hw), j = (int)((t / hw) % classes), a = (int)(t / ((long long)hw * classes));
        pred[((size_t)a * entries + coords + 1 + j) * hw + loc] = tmp[t];
    }
}

void launch_region_hierarchy(float *item_out, float *tmp, int hw, int anchors, int classes, int coords, const int *parent, cudaStream_t s)
{
    const long long total = (long long)anchors * classes * hw;
    int grid = (int)((total + kThreads - 1) / kThreads);
    if (grid > 148 * 16) grid = 148 * 16;
    region_hierarchy_kernel<<<grid, kThreads, 0, s>>>(item_out, tmp, hw, anchors, classes, coords, parent);
    B200_LAUNCHED();
    region_hierarchy_store_kernel<<<grid, kThreads, 0, s>>>(item_out, tmp, hw, anchors, classes, coords);
    B200_LAUNCHED();
}
