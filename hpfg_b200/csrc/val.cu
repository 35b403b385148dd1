// Validation on the device (val.py:268-281 test_single_volume, SURVEY 8f.3): the order-0 resampling of
// scipy.ndimage.zoom and medpy 0.4.0's dc / hd95 (calculate_metric_percase, val.py:255-265), computed exactly.
//
//  zoom_nearest_kernel   scipy's order-0 rule per axis, index in fp64 as scipy computes it
//  border_count_kernel   |P|, |G|, |P n G| per class and the 6-neighbour borders of both volumes (border_value 0)
//  edt_w_kernel          exact squared EDT to one class's border, pass 1: 1-D distance along W
//  edt_env_kernel        passes 2 (H) and 3 (S): Felzenszwalb lower envelopes, separators compared as int64 cross-products;
//                        pass 3 samples d^2 at the other set's border voxels into one histogram per class
//  select_kernel         n and the d^2 at numpy.percentile(., 95)'s ranks lo / hi
#include <algorithm>

#include "common.cuh"

namespace hpfg {
namespace {

constexpr int kEdtInf = 0x7fffffff;   // "no border voxel on this line yet" (every finite d^2 is < 2^31, checked on the host)
constexpr int kCnt = 5;               // per-class counters: |P|, |G|, |P n G|, |border P|, |border G|

// ---- order-0 zoom --------------------------------------------------------------------------------------------------------
// scipy.ndimage.zoom(x, zoom, order=0, mode='constant', cval=0, grid_mode=False) on one axis: factor f = (in-1)/(out-1) (1 when
// out == 1), source coordinate c = k*f in fp64; c > in-1 gives cval, otherwise the source index is floor(c + 0.5).  The
// multiply and the add are separately rounded (no FMA contraction): 224 -> 216 gives c = 223.00000000000003 at the last index.
__device__ __forceinline__ int zoom_src(int k, double f, int in) {
    const double c = __dmul_rn((double)k, f);
    if (c > (double)(in - 1)) return -1;
    return (int)floor(__dadd_rn(c, 0.5));
}

template <typename T>
__global__ void __launch_bounds__(256) zoom_nearest_kernel(const T *__restrict__ in, int64_t n, int in_h, int in_w, int out_h,
                                                           int out_w, double fy, double fx, T *__restrict__ out) {
    pdl_prologue();
    const int64_t plane = (int64_t)out_h * out_w, total = n * plane;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t p = i / plane;
        const int r = (int)(i - p * plane), oy = r / out_w, ox = r - oy * out_w;
        const int sy = zoom_src(oy, fy, in_h), sx = zoom_src(ox, fx, in_w);
        out[i] = (sy < 0 || sx < 0) ? T(0) : in[(p * in_h + sy) * in_w + sx];
    }
}

// ---- metrics -----------------------------------------------------------------------------------------------------------
// border(X) = X ^ binary_erosion(X, generate_binary_structure(3, 1)) with border_value 0: a voxel of class c is a border voxel
// when one of its 6 neighbours is outside the volume or of another class.  flags bit 0: border of the prediction's class, bit 1:
// border of the label's class.  Counters of classes >= num_classes are not kept (calculate_metric_percase runs for 1..C-1).
__device__ __forceinline__ bool is_border(const uint8_t *__restrict__ v, int64_t i, int s, int h, int w, int S, int H, int W,
                                          int64_t hw, uint8_t c) {
    if (s == 0 || s == S - 1 || h == 0 || h == H - 1 || w == 0 || w == W - 1) return true;
    return v[i - 1] != c || v[i + 1] != c || v[i - W] != c || v[i + W] != c || v[i - hw] != c || v[i + hw] != c;
}

__global__ void __launch_bounds__(256) border_count_kernel(const uint8_t *__restrict__ pred, const uint8_t *__restrict__ label,
                                                           int S, int H, int W, int C, uint8_t *__restrict__ flags,
                                                           unsigned *__restrict__ counts) {
    extern __shared__ unsigned sc[];   // [C][kCnt]
    for (int i = threadIdx.x; i < C * kCnt; i += blockDim.x) sc[i] = 0;
    pdl_prologue();
    __syncthreads();
    const int64_t hw = (int64_t)H * W, total = hw * S;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int s = (int)(i / hw);
        const int r = (int)(i - s * hw), h = r / W, w = r - h * W;
        const uint8_t p = pred[i], g = label[i];
        uint8_t f = 0;
        if (p != 0 && p < C) {
            atomicAdd(&sc[p * kCnt + 0], 1u);
            if (g == p) atomicAdd(&sc[p * kCnt + 2], 1u);
            if (is_border(pred, i, s, h, w, S, H, W, hw, p)) {
                f |= 1;
                atomicAdd(&sc[p * kCnt + 3], 1u);
            }
        }
        if (g != 0 && g < C) {
            atomicAdd(&sc[g * kCnt + 1], 1u);
            if (is_border(label, i, s, h, w, S, H, W, hw, g)) {
                f |= 2;
                atomicAdd(&sc[g * kCnt + 4], 1u);
            }
        }
        flags[i] = f;
    }
    __syncthreads();
    for (int i = threadIdx.x; i < C * kCnt; i += blockDim.x)
        if (sc[i]) atomicAdd(&counts[i], sc[i]);
}

// Work item (class c = 1 + cd/2, direction d = cd&1).  d = 0: distances to border(G), sampled at border(P) (sd(P,G));
// d = 1: distances to border(P), sampled at border(G) (sd(G,P)).  Classes absent from either volume are skipped.
__device__ __forceinline__ bool cd_active(const unsigned *counts, int cd) {
    const int c = 1 + (cd >> 1);
    return counts[c * kCnt + 0] != 0 && counts[c * kCnt + 1] != 0;
}
__device__ __forceinline__ bool in_set(const uint8_t *pred, const uint8_t *label, const uint8_t *flags, int64_t i, int c, int bit) {
    return (flags[i] & (1 << bit)) && (bit == 0 ? pred[i] : label[i]) == c;
}

// Pass 1 (W): a[i] = (distance along the row to the nearest target voxel)^2, kEdtInf when the row has none.  One thread per row.
__global__ void __launch_bounds__(128) edt_w_kernel(const uint8_t *__restrict__ pred, const uint8_t *__restrict__ label,
                                                    const uint8_t *__restrict__ flags, const unsigned *__restrict__ counts,
                                                    int64_t rows, int W, int64_t voxels, int *__restrict__ a) {
    pdl_prologue();
    const int cd = blockIdx.y;
    if (!cd_active(counts, cd)) return;
    const int c = 1 + (cd >> 1), bit = (cd & 1) ? 0 : 1;        // target set: border(G) for d = 0, border(P) for d = 1
    int *ac = a + (int64_t)cd * voxels;
    for (int64_t row = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; row < rows; row += (int64_t)gridDim.x * blockDim.x) {
        const int64_t base = row * W;
        int last = -1;
        for (int x = 0; x < W; ++x) {                            // distance to the nearest target on the left (or none)
            if (in_set(pred, label, flags, base + x, c, bit)) last = x;
            ac[base + x] = last < 0 ? kEdtInf : x - last;
        }
        last = -1;
        for (int x = W - 1; x >= 0; --x) {                       // ... and on the right; store the square
            if (in_set(pred, label, flags, base + x, c, bit)) last = x;
            int d = ac[base + x];
            if (last >= 0 && last - x < d) d = last - x;
            ac[base + x] = d == kEdtInf ? kEdtInf : d * d;
        }
    }
}

// Lower envelope of the parabolas y = f(q) + (p - q)^2 over the finite f(q) of one line (Felzenszwalb & Huttenlocher 2012).  The
// intersection of the parabolas at q > v is s(q, v) = (f(q) + q^2 - f(v) - v^2) / (2 (q - v)); all comparisons of two such
// rationals (positive denominators) are done as int64 cross-products, so every d^2 is exact.
struct Sep {
    int64_t num, den;
};
__device__ __forceinline__ Sep sep(int q, int fq, int v, int fv) {
    return {(int64_t)fq + (int64_t)q * q - (int64_t)fv - (int64_t)v * v, 2 * (int64_t)(q - v)};
}

// Passes 2 (H) and 3 (S) over lines of `len` elements `stride` apart; line l starts at (l / inner) * len * inner + l % inner.
// in: the previous pass's d^2; env: scratch of the envelope's vertex positions (same layout).  SAMPLE = false: out = d^2;
// SAMPLE = true (the last pass): d^2 at the sample set's voxels goes to the class's histogram instead.
template <bool SAMPLE>
__global__ void __launch_bounds__(128) edt_env_kernel(const uint8_t *__restrict__ pred, const uint8_t *__restrict__ label,
                                                      const uint8_t *__restrict__ flags, const unsigned *__restrict__ counts,
                                                      int64_t lines, int len, int64_t inner, int64_t voxels,
                                                      const int *__restrict__ in, int *__restrict__ env, int *__restrict__ out,
                                                      unsigned *__restrict__ hist, int64_t nbins) {
    pdl_prologue();
    const int cd = blockIdx.y;
    if (!cd_active(counts, cd)) return;
    const int c = 1 + (cd >> 1), sample_bit = (cd & 1) ? 1 : 0;   // sample set: border(P) for d = 0, border(G) for d = 1
    const int *f = in + (int64_t)cd * voxels;
    int *v = env + (int64_t)cd * voxels;
    int *oc = SAMPLE ? nullptr : out + (int64_t)cd * voxels;
    unsigned *hc = hist + (int64_t)(cd >> 1) * nbins;
    for (int64_t l = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; l < lines; l += (int64_t)gridDim.x * blockDim.x) {
        const int64_t o = l / inner, base = o * len * inner + (l - o * inner);
        int k = -1;
        for (int q = 0; q < len; ++q) {
            const int fq = f[base + q * inner];
            if (fq == kEdtInf) continue;
            while (k > 0) {
                const int vk = v[base + k * inner], vk1 = v[base + (k - 1) * inner];
                const Sep a = sep(q, fq, vk, f[base + vk * inner]), b = sep(vk, f[base + vk * inner], vk1, f[base + vk1 * inner]);
                if (a.num * b.den <= b.num * a.den) --k;      // s(q, v_k) <= s(v_k, v_k-1): v_k is hidden
                else break;
            }
            ++k;
            v[base + k * inner] = q;
        }
        int j = 0;
        int vj = k >= 0 ? v[base] : 0, fj = k >= 0 ? f[base + vj * inner] : kEdtInf;
        for (int p = 0; p < len; ++p) {
            const int64_t i = base + p * inner;
            if (SAMPLE && !in_set(pred, label, flags, i, c, sample_bit)) continue;
            int d2 = kEdtInf;
            if (k >= 0) {
                while (j < k) {                               // advance while s(v_j+1, v_j) < p
                    const int vn = v[base + (j + 1) * inner], fn = f[base + vn * inner];
                    const Sep s = sep(vn, fn, vj, fj);
                    if (s.num < (int64_t)p * s.den) {
                        ++j;
                        vj = vn;
                        fj = fn;
                    } else {
                        break;
                    }
                }
                d2 = fj + (p - vj) * (p - vj);
            }
            if (SAMPLE) atomicAdd(&hc[d2], 1u);              // finite: the target set is not empty
            else oc[i] = d2;
        }
    }
}

// One block per class: n = |border P| + |border G|, vi = (n-1)*0.95 in fp64, lo = floor(vi), hi = min(lo+1, n-1) (numpy's
// 'linear' percentile), and the d^2 at ranks lo and hi of the class's histogram.  out[(c-1)*6..] = {|P|, |G|, |P n G|, n,
// d2_lo, d2_hi}; d2_lo = d2_hi = 0 for a class absent from either volume.
constexpr int kSelThreads = 512;
__global__ void __launch_bounds__(kSelThreads) select_kernel(const unsigned *__restrict__ counts, const unsigned *__restrict__ hist,
                                                             int64_t nbins4, int64_t *__restrict__ out) {
    __shared__ int64_t pre[kSelThreads];
    __shared__ int64_t res[2];
    pdl_prologue();
    const int c = 1 + blockIdx.x;
    const unsigned *cn = counts + c * kCnt;
    const int64_t n = (int64_t)cn[3] + cn[4];
    const bool active = cn[0] != 0 && cn[1] != 0;
    int64_t lo = 0, hi = 0;
    if (active) {
        const double vi = __dmul_rn((double)(n - 1), 0.95);
        lo = (int64_t)floor(vi);
        hi = lo + 1 < n - 1 ? lo + 1 : n - 1;
    }
    if (threadIdx.x < 2) res[threadIdx.x] = 0;
    const uint4 *h = reinterpret_cast<const uint4 *>(hist + (int64_t)blockIdx.x * nbins4 * 4);
    const int64_t chunk = (nbins4 + kSelThreads - 1) / kSelThreads, b0 = threadIdx.x * chunk;
    const int64_t b1 = b0 + chunk < nbins4 ? b0 + chunk : nbins4;
    int64_t sum = 0;
    if (active)
        for (int64_t b = b0; b < b1; ++b) {
            const uint4 q = h[b];
            sum += (int64_t)q.x + q.y + q.z + q.w;
        }
    pre[threadIdx.x] = sum;
    __syncthreads();
    for (int off = 1; off < kSelThreads; off <<= 1) {       // inclusive scan of the chunk sums
        const int64_t t = threadIdx.x >= off ? pre[threadIdx.x - off] : 0;
        __syncthreads();
        pre[threadIdx.x] += t;
        __syncthreads();
    }
    if (active) {
        int64_t acc = pre[threadIdx.x] - sum;               // values before this chunk
        if (sum > 0 && ((lo >= acc && lo < acc + sum) || (hi >= acc && hi < acc + sum))) {
            for (int64_t b = b0; b < b1; ++b) {
                const uint4 q = h[b];
                const unsigned cnt[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                    if (lo >= acc && lo < acc + cnt[e]) res[0] = b * 4 + e;
                    if (hi >= acc && hi < acc + cnt[e]) res[1] = b * 4 + e;
                    acc += cnt[e];
                }
            }
        }
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        int64_t *o = out + (int64_t)blockIdx.x * 6;
        o[0] = cn[0];
        o[1] = cn[1];
        o[2] = cn[2];
        o[3] = n;
        o[4] = res[0];
        o[5] = res[1];
    }
}

// ---- workspace -----------------------------------------------------------------------------------------------------------
struct MetricsLayout {
    int64_t voxels, nbins, nbins4, counts_off, flags_off, a_off, b_off, env_off, hist_off, total;
};
inline int64_t align256(int64_t v) { return (v + 255) & ~int64_t(255); }

int metrics_layout(int depth, int height, int width, int num_classes, MetricsLayout &m) {
    HPFG_REQUIRE(depth >= 1 && height >= 1 && width >= 1, "hpfg_volume_metrics: depth, height and width must be >= 1");
    HPFG_REQUIRE(num_classes >= 2 && num_classes <= 256, "hpfg_volume_metrics: num_classes must be in [2, 256] (uint8 labels)");
    m.voxels = (int64_t)depth * height * width;
    // the largest d^2 in the volume is (S-1)^2 + (H-1)^2 + (W-1)^2: one histogram bin per value
    m.nbins = (int64_t)(depth - 1) * (depth - 1) + (int64_t)(height - 1) * (height - 1) + (int64_t)(width - 1) * (width - 1) + 1;
    if (m.voxels >= (int64_t(1) << 31) || m.nbins >= kEdtInf) {
        set_error("hpfg_volume_metrics: volume " + std::to_string(depth) + "x" + std::to_string(height) + "x" +
                  std::to_string(width) + " has more than 2^31 voxels or a squared diameter that does not fit int32");
        return HPFG_ERR_UNSUPPORTED;
    }
    m.nbins4 = (m.nbins + 3) / 4;
    const int64_t cds = 2 * (int64_t)(num_classes - 1);
    m.counts_off = 0;
    m.flags_off = align256(num_classes * kCnt * 4);
    m.a_off = m.flags_off + align256(m.voxels);
    m.b_off = m.a_off + align256(cds * m.voxels * 4);
    m.env_off = m.b_off + align256(cds * m.voxels * 4);
    m.hist_off = m.env_off + align256(cds * m.voxels * 4);
    m.total = m.hist_off + align256((int64_t)(num_classes - 1) * m.nbins4 * 16);
    return HPFG_OK;
}

template <typename T>
int launch_zoom(const void *in, int64_t n, int in_h, int in_w, int out_h, int out_w, double fy, double fx, void *out,
                cudaStream_t st) {
    const int64_t total = n * out_h * out_w;
    const int grid = (int)std::min<int64_t>((total + 255) / 256, (int64_t)kNumSMs * 16);
    HPFG_CUDA_CHECK(launch_pdl(zoom_nearest_kernel<T>, dim3(grid), dim3(256), 0, st, static_cast<const T *>(in), n, in_h, in_w,
                               out_h, out_w, fy, fx, static_cast<T *>(out)));
    HPFG_LAUNCH_CHECK();
    return HPFG_OK;
}

}  // namespace
}  // namespace hpfg

using namespace hpfg;

// scipy.ndimage.zoom(plane, (out_h/in_h, out_w/in_w), order=0) for each of n planes (val.py:272 resamples every image slice to
// the patch size, val.py:277 the predicted labels back).
extern "C" int hpfg_zoom_nearest(const void *in, int64_t n, int in_h, int in_w, int out_h, int out_w, int elem_bytes, void *out,
                                 void *stream) {
    HPFG_REQUIRE(in && out, "hpfg_zoom_nearest: null buffer");
    HPFG_REQUIRE(n >= 1 && in_h >= 1 && in_w >= 1 && out_h >= 1 && out_w >= 1, "hpfg_zoom_nearest: sizes must be >= 1");
    HPFG_REQUIRE(n * out_h * out_w < (int64_t(1) << 40) && n * in_h * in_w < (int64_t(1) << 40), "hpfg_zoom_nearest: too large");
    // scipy: zoom = (in-1)/(out-1) per axis as one fp64 division, 1 where out == 1
    const double fy = out_h > 1 ? (double)(in_h - 1) / (double)(out_h - 1) : 1.0;
    const double fx = out_w > 1 ? (double)(in_w - 1) / (double)(out_w - 1) : 1.0;
    cudaStream_t st = (cudaStream_t)stream;
    switch (elem_bytes) {
        case 1: return launch_zoom<uint8_t>(in, n, in_h, in_w, out_h, out_w, fy, fx, out, st);
        case 4: return launch_zoom<uint32_t>(in, n, in_h, in_w, out_h, out_w, fy, fx, out, st);
        case 8: return launch_zoom<uint64_t>(in, n, in_h, in_w, out_h, out_w, fy, fx, out, st);
        default: set_error("hpfg_zoom_nearest: elem_bytes must be 1, 4 or 8"); return HPFG_ERR_INVALID;
    }
}

extern "C" int64_t hpfg_volume_metrics_workspace_bytes(int depth, int height, int width, int num_classes) {
    MetricsLayout m;
    if (metrics_layout(depth, height, width, num_classes, m) != HPFG_OK) return -1;
    return m.total;
}

// calculate_metric_percase (val.py:255-265) for every class 1..C-1 of one volume: medpy's dc (counts) and the integer parts of
// hd95 = percentile(hstack(sd(P,G), sd(G,P)), 95) with sd(A,B) = distance_transform_edt(~border(B))[border(A)]
// (medpy/metric/binary.py __surface_distances, connectivity 1, no voxel spacing).  The host finishes Dice and the lerp.
extern "C" int hpfg_volume_metrics(const uint8_t *pred_u8, const uint8_t *label_u8, int depth, int height, int width,
                                   int num_classes, int64_t *out, void *workspace, void *stream) {
    HPFG_REQUIRE(pred_u8 && label_u8 && out && workspace, "hpfg_volume_metrics: null buffer");
    MetricsLayout m;
    HPFG_RETURN_IF(metrics_layout(depth, height, width, num_classes, m));
    cudaStream_t st = (cudaStream_t)stream;
    ProfScope _prof(PROF_LOSS, st);
    char *ws = static_cast<char *>(workspace);
    unsigned *counts = reinterpret_cast<unsigned *>(ws + m.counts_off);
    uint8_t *flags = reinterpret_cast<uint8_t *>(ws + m.flags_off);
    int *a = reinterpret_cast<int *>(ws + m.a_off), *b = reinterpret_cast<int *>(ws + m.b_off);
    int *env = reinterpret_cast<int *>(ws + m.env_off);
    unsigned *hist = reinterpret_cast<unsigned *>(ws + m.hist_off);
    HPFG_CUDA_CHECK(cudaMemsetAsync(counts, 0, (size_t)num_classes * kCnt * 4, st));
    HPFG_CUDA_CHECK(cudaMemsetAsync(hist, 0, (size_t)(num_classes - 1) * m.nbins4 * 16, st));
    const int cds = 2 * (num_classes - 1);
    const int64_t hw = (int64_t)height * width;
    {
        const int grid = (int)std::min<int64_t>((m.voxels + 255) / 256, (int64_t)kNumSMs * 8);
        HPFG_CUDA_CHECK(launch_pdl(border_count_kernel, dim3(grid), dim3(256), (size_t)num_classes * kCnt * 4, st, pred_u8,
                                   label_u8, depth, height, width, num_classes, flags, counts));
        HPFG_LAUNCH_CHECK();
    }
    auto grid_x = [](int64_t lines) { return (int)std::min<int64_t>((lines + 127) / 128, 4096); };
    const int64_t rows = (int64_t)depth * height;
    HPFG_CUDA_CHECK(launch_pdl(edt_w_kernel, dim3(grid_x(rows), cds), dim3(128), 0, st, pred_u8, label_u8,
                               (const uint8_t *)flags, (const unsigned *)counts, rows, width, m.voxels, a));
    HPFG_LAUNCH_CHECK();
    // pass 2 (H): lines (s, w), elements W apart
    HPFG_CUDA_CHECK(launch_pdl(edt_env_kernel<false>, dim3(grid_x(depth * (int64_t)width), cds), dim3(128), 0, st, pred_u8,
                               label_u8, (const uint8_t *)flags, (const unsigned *)counts, depth * (int64_t)width, height,
                               (int64_t)width, m.voxels, (const int *)a, env, b, hist, m.nbins4 * 4));
    HPFG_LAUNCH_CHECK();
    // pass 3 (S): lines (h, w), elements H*W apart; samples into the histograms (the envelope scratch reuses pass 1's buffer)
    HPFG_CUDA_CHECK(launch_pdl(edt_env_kernel<true>, dim3(grid_x(hw), cds), dim3(128), 0, st, pred_u8, label_u8,
                               (const uint8_t *)flags, (const unsigned *)counts, hw, depth, hw, m.voxels, (const int *)b, a,
                               (int *)nullptr, hist, m.nbins4 * 4));
    HPFG_LAUNCH_CHECK();
    HPFG_CUDA_CHECK(launch_pdl(select_kernel, dim3(num_classes - 1), dim3(kSelThreads), 0, st, (const unsigned *)counts,
                               (const unsigned *)hist, m.nbins4, out));
    HPFG_LAUNCH_CHECK();
    return HPFG_OK;
}
