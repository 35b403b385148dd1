// UNet_Plus projection necks and Dense_Loss (SURVEY 8f.2): model/unet.py:120-152 (projection_conv), utils/loss/dense_loss.py:18-40.
//
// A neck sees a [N,C,H,W] fp32 NCHW map (the bottleneck feature, 256 x 14 x 14, or the logits, num_classes x 224 x 224) and
// returns a global vector mlp(avgpool(x)) [N,out] and a dense map mlp_conv(adaptive_pool_sxs(x)) [N,out,s*s].  Both branches
// are "rows x channels" problems once the pooling is done, so the layout is: ONE pooled matrix [N*(1+s*s), C] (rows 0..N-1
// the global means, then the s*s bins of every image), two fp32 GEMMs per branch with bias / ReLU in the epilogue, and the
// dense output stored transposed ([N,out,s*s]) by the epilogue's address map.  Everything is fp32 FMA on the CUDA cores:
// the reference computes these in fp32, the contrastive loss exponentiates 16/temperature, and all necks of a step are
// ~5 GFLOP next to the U-Nets' 550 -- not tensor-core work.
// Backward: the transposed GEMMs (weight gradients with the bias gradient as a by-product of the A-operand tiles, hidden
// gradient masked by ReLU in the epilogue, pooled gradient) and the adjoint of the two poolings in one pass over dx.
#include "common.cuh"

namespace hpfg {
namespace {

// ---------------------------------------------------------------------------------------------------------------------
// C[m,n] = epilogue( sum_k A(m,k) * B(n,k) ), 64x64 tile, 16-deep k steps, 4x4 outputs per thread, next tile prefetched
// into registers while the current one is multiplied.  A_K: A(m,k) = A[m*lda + k] (k contiguous) else A[k*lda + m];
// B_K likewise with n.  Epilogue: + bias[n], ReLU, * (mask[m,n] > 0) (mask in C's row-major layout), and either a
// row-major store (ldc) or, with dense_s > 0, the neck's [N,out,s*s] layout: row m = (image, position) -> C[(image*N + n)*s*s + position].
// colsum (optional, written by the n-tile-0 CTAs): colsum[m] = sum_k A(m,k) -- the bias gradient of a weight-gradient GEMM.
constexpr int BM = 64, BN = 64, BK = 16, PITCH = BM + 4, GEMM_THREADS = 256;

template <bool K_CONTIG>
__device__ __forceinline__ void gemm_fetch(const float *__restrict__ src, int ld, int row0, int rows, int k0, int K, int tid, float (&r)[4]) {
#pragma unroll
    for (int e = 0; e < 4; ++e) {
        const int idx = tid + e * GEMM_THREADS;
        const int k = K_CONTIG ? (idx & (BK - 1)) : (idx >> 6);
        const int m = K_CONTIG ? (idx >> 4) : (idx & (BM - 1));
        const bool ok = (row0 + m < rows) && (k0 + k < K);
        const int64_t off = K_CONTIG ? (int64_t)(row0 + m) * ld + (k0 + k) : (int64_t)(k0 + k) * ld + (row0 + m);
        r[e] = ok ? __ldg(src + off) : 0.f;
    }
}
template <bool K_CONTIG>
__device__ __forceinline__ void gemm_stage(float (*tile)[PITCH], int tid, const float (&r)[4]) {
#pragma unroll
    for (int e = 0; e < 4; ++e) {
        const int idx = tid + e * GEMM_THREADS;
        const int k = K_CONTIG ? (idx & (BK - 1)) : (idx >> 6);
        const int m = K_CONTIG ? (idx >> 4) : (idx & (BM - 1));
        tile[k][m] = r[e];
    }
}

template <bool A_K, bool B_K>
__global__ void __launch_bounds__(GEMM_THREADS)
neck_gemm_kernel(const float *__restrict__ A, int lda, const float *__restrict__ B, int ldb, float *__restrict__ C, int ldc, int M, int N,
                 int K, const float *__restrict__ bias, int relu, const float *__restrict__ mask, float *__restrict__ colsum, int dense_s) {
    __shared__ __align__(16) float As[BK][PITCH];
    __shared__ __align__(16) float Bs[BK][PITCH];
    const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
    const int m0 = blockIdx.y * BM, n0 = blockIdx.x * BN;
    const bool sum_rows = colsum != nullptr && blockIdx.x == 0 && tx == 0;
    float acc[4][4] = {};
    float cs[4] = {};
    float ra[4], rb[4];
    pdl_prologue();
    gemm_fetch<A_K>(A, lda, m0, M, 0, K, tid, ra);
    gemm_fetch<B_K>(B, ldb, n0, N, 0, K, tid, rb);
    for (int k0 = 0; k0 < K; k0 += BK) {
        gemm_stage<A_K>(As, tid, ra);
        gemm_stage<B_K>(Bs, tid, rb);
        __syncthreads();
        if (k0 + BK < K) {
            gemm_fetch<A_K>(A, lda, m0, M, k0 + BK, K, tid, ra);
            gemm_fetch<B_K>(B, ldb, n0, N, k0 + BK, K, tid, rb);
        }
#pragma unroll
        for (int k = 0; k < BK; ++k) {
            const float4 a4 = *reinterpret_cast<const float4 *>(&As[k][ty * 4]);
            const float4 b4 = *reinterpret_cast<const float4 *>(&Bs[k][tx * 4]);
            const float a[4] = {a4.x, a4.y, a4.z, a4.w}, b[4] = {b4.x, b4.y, b4.z, b4.w};
#pragma unroll
            for (int i = 0; i < 4; ++i) {
#pragma unroll
                for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
            }
            if (sum_rows) {
#pragma unroll
                for (int i = 0; i < 4; ++i) cs[i] += a[i];
            }
        }
        __syncthreads();
    }
    if (sum_rows) {
#pragma unroll
        for (int i = 0; i < 4; ++i)
            if (m0 + ty * 4 + i < M) colsum[m0 + ty * 4 + i] = cs[i];
    }
    const int positions = dense_s > 0 ? dense_s * dense_s : 1;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int m = m0 + ty * 4 + i;
        if (m >= M) continue;
        const int img = m / positions, pos = m - img * positions;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int n = n0 + tx * 4 + j;
            if (n >= N) continue;
            float v = acc[i][j];
            if (bias) v += __ldg(bias + n);
            if (relu) v = fmaxf(v, 0.f);
            if (mask) v = __ldg(mask + (int64_t)m * ldc + n) > 0.f ? v : 0.f;
            if (dense_s > 0)
                C[((int64_t)img * N + n) * positions + pos] = v;
            else
                C[(int64_t)m * ldc + n] = v;
        }
    }
}

struct GemmArgs {
    const float *A;
    int lda;
    const float *B;
    int ldb;
    float *C;
    int ldc;
    int M, N, K;
    const float *bias = nullptr;
    int relu = 0;
    const float *mask = nullptr;
    float *colsum = nullptr;
    int dense_s = 0;
};
template <bool A_K, bool B_K>
int launch_gemm(const GemmArgs &g, cudaStream_t st) {
    dim3 grid(ceil_div(g.N, BN), ceil_div(g.M, BM));
    HPFG_CUDA_CHECK(launch_pdl(neck_gemm_kernel<A_K, B_K>, grid, dim3(GEMM_THREADS), 0, st, g.A, g.lda, g.B, g.ldb, g.C, g.ldc, g.M, g.N,
                               g.K, g.bias, g.relu, g.mask, g.colsum, g.dense_s));
    HPFG_LAUNCH_CHECK();
    return HPFG_OK;
}

// ---------------------------------------------------------------------------------------------------------------------
// nn.AdaptiveAvgPool2d((1,1)) and ((s,s)) of one (image, channel) plane per CTA (model/unet.py:142,148): bin i of an axis of
// length L covers [floor(i*L/s), ceil((i+1)*L/s)) -- bins overlap when s does not divide L (14 -> 4).  Pass 1: one warp per
// row, lanes along w (coalesced), per-row sums of every column bin and of the whole row in shared memory; pass 2: one thread
// per bin adds its rows in order (deterministic).  pooled: [N*(1+s*s), C], rows 0..N-1 global means, row N + n*s*s + i*s + j the bins.
__device__ __forceinline__ int bin_lo(int i, int len, int s) { return (i * len) / s; }
__device__ __forceinline__ int bin_hi(int i, int len, int s) { return ((i + 1) * len + s - 1) / s; }

__global__ void neck_pool_kernel(const float *__restrict__ x, int n_img, int C, int H, int W, int s, float *__restrict__ pooled) {
    extern __shared__ float rowsum[];               // [H][s+1]: column-bin sums of each row, then the whole-row sum
    const int plane = blockIdx.x, n = plane / C, c = plane - n * C;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
    const float *src = x + (int64_t)plane * H * W;
    pdl_prologue();
    for (int h = warp; h < H; h += nwarps) {
        const float *row = src + (int64_t)h * W;
        float all = 0.f;
        for (int w = lane; w < W; w += 32) all += __ldg(row + w);
        all = warp_sum(all);
        if (lane == 0) rowsum[h * (s + 1) + s] = all;
        for (int j = 0; j < s; ++j) {
            const int lo = bin_lo(j, W, s), hi = bin_hi(j, W, s);
            float v = 0.f;
            for (int w = lo + lane; w < hi; w += 32) v += __ldg(row + w);
            v = warp_sum(v);
            if (lane == 0) rowsum[h * (s + 1) + j] = v;
        }
    }
    __syncthreads();
    for (int b = threadIdx.x; b <= s * s; b += blockDim.x) {
        if (b == s * s) {
            float v = 0.f;
            for (int h = 0; h < H; ++h) v += rowsum[h * (s + 1) + s];
            pooled[(int64_t)n * C + c] = v / (float)(H * W);
        } else {
            const int i = b / s, j = b - i * s;
            const int h0 = bin_lo(i, H, s), h1 = bin_hi(i, H, s);
            float v = 0.f;
            for (int h = h0; h < h1; ++h) v += rowsum[h * (s + 1) + j];
            const int cnt = (h1 - h0) * (bin_hi(j, W, s) - bin_lo(j, W, s));
            pooled[((int64_t)n_img + (int64_t)n * s * s + b) * C + c] = v / (float)cnt;
        }
    }
}

// adjoint of both poolings: dx[n,c,h,w] = dpooled_global[n,c]/(H*W) + sum over the bins that contain (h,w) of dpooled_bin/|bin|
__global__ void neck_pool_bwd_kernel(const float *__restrict__ dpooled, int n_img, int C, int H, int W, int s, float *__restrict__ dx, int64_t total) {
    pdl_prologue();
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
        const int w = (int)(e % W);
        const int64_t t = e / W;
        const int h = (int)(t % H);
        const int64_t plane = t / H;
        const int n = (int)(plane / C), c = (int)(plane - (int64_t)n * C);
        float g = __ldg(dpooled + (int64_t)n * C + c) / (float)(H * W);
        const float *bins = dpooled + ((int64_t)n_img + (int64_t)n * s * s) * C + c;
        for (int i = 0; i < s; ++i) {
            const int h0 = bin_lo(i, H, s), h1 = bin_hi(i, H, s);
            if (h < h0 || h >= h1) continue;
            for (int j = 0; j < s; ++j) {
                const int w0 = bin_lo(j, W, s), w1 = bin_hi(j, W, s);
                if (w < w0 || w >= w1) continue;
                g += __ldg(bins + (int64_t)(i * s + j) * C) / (float)((h1 - h0) * (w1 - w0));
            }
        }
        dx[e] = g;
    }
}

// d_dense [N,out,S] -> rows [(n,pos), out]: the A operand of the backward GEMMs
__global__ void neck_dense_to_rows_kernel(const float *__restrict__ d_dense, int out, int S, float *__restrict__ rows, int64_t total) {
    pdl_prologue();
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
        const int o = (int)(e % out);
        const int64_t r = e / out;
        const int n = (int)(r / S), pos = (int)(r - (int64_t)n * S);
        rows[e] = __ldg(d_dense + ((int64_t)n * out + o) * S + pos);
    }
}

// ---------------------------------------------------------------------------------------------------------------------
// Dense_Loss.contrastive_loss (utils/loss/dense_loss.py:18-34) on out_1, out_2 [B,D,S] (S = 1 for the global vectors):
// z = cat(normalize(out_1, dim=1).flatten(1), normalize(out_2, dim=1).flatten(1)); sim = exp(z z^T / t);
// loss = mean_i( -log( exp(<a_i,b_i>/t) / sum_{j != i} sim_ij ) ) over the 2B rows.  Three launches on 2B (or B) CTAs.
// batch = 1 (two rows, one off-diagonal entry each) gives exactly 0, as the formula does.
constexpr float kNormEps = 1e-12f;      // F.normalize default

// one CTA per row r of z: channel norms per spatial position (a warp each), z row, norms
__global__ void contrast_normalize_kernel(const float *__restrict__ out1, const float *__restrict__ out2, int B, int D, int S, float *__restrict__ z,
                                          float *__restrict__ norms) {
    const int r = blockIdx.x, lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
    const int64_t V = (int64_t)D * S;
    const float *src = r < B ? out1 + r * V : out2 + (r - B) * V;
    pdl_prologue();
    for (int s = warp; s < S; s += nwarps) {
        float ss = 0.f;
        for (int d = lane; d < D; d += 32) {
            const float v = __ldg(src + (int64_t)d * S + s);
            ss = fmaf(v, v, ss);
        }
        const float nrm = sqrtf(warp_sum(ss));
        const float inv = 1.f / fmaxf(nrm, kNormEps);
        for (int d = lane; d < D; d += 32) z[r * V + (int64_t)d * S + s] = __ldg(src + (int64_t)d * S + s) * inv;
        if (lane == 0) norms[r * S + s] = nrm;
    }
}

// one CTA per row i: the 2B similarities of the row (a warp per column, fp64 accumulation), taken RELATIVE to the positive pair:
// e_ij = exp((s_ij - s_i,pair)/t), so e_i,pair = 1 and the row's loss term -log(pos_i / sum_{j != i} sim_ij) = log1p(rest_i) with
// rest_i = sum_{j != i, pair} e_ij.  Same quantity as the reference's exp(s/t) ratios, but it neither overflows nor cancels when the
// pair dominates (16 positions: exp(16/0.7) against exp(~0), the usual state once the teacher tracks the student).
// P_ij = e_ij / (1 + rest_i) (0 on the diagonal) and miss_i = 1 - P_i,pair = rest_i / (1 + rest_i) go to the gradient kernel.
__global__ void contrast_rows_kernel(const float *__restrict__ z, int B, int V, float inv_t, float *__restrict__ P, float *__restrict__ miss,
                                     float *__restrict__ rowloss) {
    extern __shared__ float sm[];                   // z_i [V] | s_ij [2B] | {1 + rest}
    float *zi = sm, *sim = sm + V, *misc = sim + 2 * B;
    const int i = blockIdx.x, rows = 2 * B, pair = i < B ? i + B : i - B;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
    pdl_prologue();
    for (int v = threadIdx.x; v < V; v += blockDim.x) zi[v] = z[(int64_t)i * V + v];
    __syncthreads();
    for (int j = warp; j < rows; j += nwarps) {
        const float *zj = z + (int64_t)j * V;
        double dot = 0.0;
        for (int v = lane; v < V; v += 32) dot = fma((double)zi[v], (double)zj[v], dot);
        dot = warp_sum(dot);
        if (lane == 0) sim[j] = (float)dot;
    }
    __syncthreads();
    const float s_pair = sim[pair];
    __syncthreads();
    for (int j = threadIdx.x; j < rows; j += blockDim.x) sim[j] = (j == i) ? 0.f : (j == pair) ? 1.f : expf((sim[j] - s_pair) * inv_t);
    __syncthreads();
    if (threadIdx.x == 0) {
        float rest = 0.f;
        for (int j = 0; j < rows; ++j)
            if (j != i && j != pair) rest += sim[j];
        misc[0] = 1.f + rest;
        rowloss[i] = log1pf(rest);
        miss[i] = rest / (1.f + rest);
    }
    __syncthreads();
    const float denom = misc[0];
    for (int j = threadIdx.x; j < rows; j += blockDim.x) P[(int64_t)i * rows + j] = sim[j] / denom;
}

// CTA 0 writes loss = mean(rowloss).  With d_out1 != NULL, CTA k (< B): dL/dz_k = ((P_k. + P_.k) z - 2 z_pair) / (2B t) with the
// pair's coefficient P_k,pair + P_pair,k - 2 taken as -(miss_k + miss_pair), pulled back through the normalisation of out_1[k]:
// dx = (g - a <a,g>) / |x| per spatial position (g / eps where |x| < eps), times `out_scale` (from scale_dev when given) as a separate
// rounding, so that d_out1 is bit-identical to out_scale * (the unscaled gradient).
__global__ void contrast_grad_kernel(const float *__restrict__ z, const float *__restrict__ norms, const float *__restrict__ P,
                                     const float *__restrict__ miss, const float *__restrict__ rowloss, int B, int D, int S, float inv_t,
                                     float out_scale, const float *__restrict__ scale_dev, float *__restrict__ loss, float *__restrict__ d_out1) {
    extern __shared__ float sm[];                   // g [V] | coef [2B]
    const int k = blockIdx.x, rows = 2 * B, V = D * S;
    float *g = sm, *coef = sm + V;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
    pdl_prologue();
    if (k == 0 && threadIdx.x == 0) {
        float v = 0.f;
        for (int i = 0; i < rows; ++i) v += rowloss[i];
        *loss = v / (float)rows;
    }
    if (d_out1 == nullptr) return;
    if (scale_dev) out_scale = *scale_dev;
    for (int j = threadIdx.x; j < rows; j += blockDim.x)
        coef[j] = (j == k + B) ? -(miss[k] + miss[k + B]) : P[(int64_t)k * rows + j] + P[(int64_t)j * rows + k];
    __syncthreads();
    const float scale = inv_t / (float)rows;
    for (int v = threadIdx.x; v < V; v += blockDim.x) {
        float a = 0.f;
        for (int j = 0; j < rows; ++j) a = fmaf(coef[j], z[(int64_t)j * V + v], a);
        g[v] = a * scale;
    }
    __syncthreads();
    const float *zk = z + (int64_t)k * V;
    for (int s = warp; s < S; s += nwarps) {
        float dot = 0.f;
        for (int d = lane; d < D; d += 32) dot = fmaf(zk[d * S + s], g[d * S + s], dot);
        dot = warp_sum(dot);
        const float nrm = norms[k * S + s];
        const bool clamped = !(nrm > kNormEps);
        const float inv = 1.f / fmaxf(nrm, kNormEps);
        for (int d = lane; d < D; d += 32) {
            const float gv = g[d * S + s];
            d_out1[(int64_t)k * V + d * S + s] = __fmul_rn(out_scale, (clamped ? gv : gv - zk[d * S + s] * dot) * inv);
        }
    }
}

int pool_threads(int H) { return H >= 16 * 8 ? 512 : H >= 32 ? 256 : 128; }

}  // namespace
}  // namespace hpfg

using namespace hpfg;

extern "C" int hpfg_neck_forward(const float *x, int n, int channels, int height, int width, int s, int hid, int out,
                                 const float *const *params, float *pooled, float *hidden, float *out_global, float *out_dense,
                                 void *stream) {
    HPFG_REQUIRE(x && params && pooled && hidden && out_global && out_dense, "hpfg_neck_forward: null buffer");
    for (int i = 0; i < 8; ++i) HPFG_REQUIRE(params[i], "hpfg_neck_forward: null parameter tensor");
    HPFG_REQUIRE(n > 0 && channels > 0 && hid > 0 && out > 0, "hpfg_neck_forward: empty problem");
    HPFG_REQUIRE(s >= 1 && s <= height && s <= width, "hpfg_neck_forward: the dense branch needs 1 <= s <= H, W (s = 0 / no pooling is not supported)");
    const size_t pool_smem = (size_t)height * (s + 1) * sizeof(float);
    HPFG_REQUIRE(pool_smem <= 48 * 1024, "hpfg_neck_forward: H*(s+1) exceeds the pooling kernel's shared memory");
    HPFG_REQUIRE((int64_t)n * channels < (1ll << 31) && (int64_t)n * (1 + s * s) * (int64_t)(hid > channels ? hid : channels) < (1ll << 31),
                 "hpfg_neck_forward: problem too large");
    cudaStream_t st = (cudaStream_t)stream;
    const int S = s * s, rows_dense = n * S;
    {
        ProfScope _prof(PROF_GLUE, st);
        HPFG_CUDA_CHECK(launch_pdl(neck_pool_kernel, dim3(n * channels), dim3(pool_threads(height)), pool_smem, st, x, n, channels, height,
                                   width, s, pooled));
        HPFG_LAUNCH_CHECK();
    }
    ProfScope _prof(PROF_CONV_CUDA, st);
    GemmArgs g;
    // global branch: mlp = Linear -> ReLU -> Linear on rows 0..n-1 (model/unet.py:142-144)
    g = GemmArgs{pooled, channels, params[0], channels, hidden, hid, n, hid, channels, params[1], 1};
    HPFG_RETURN_IF((launch_gemm<true, true>(g, st)));
    g = GemmArgs{hidden, hid, params[2], hid, out_global, out, n, out, hid, params[3], 0};
    HPFG_RETURN_IF((launch_gemm<true, true>(g, st)));
    // dense branch: mlp_conv = 1x1 conv -> ReLU -> 1x1 conv on the s*s bins (model/unet.py:147-150), stored [N,out,s*s]
    const float *pd = pooled + (int64_t)n * channels;
    float *hd = hidden + (int64_t)n * hid;
    g = GemmArgs{pd, channels, params[4], channels, hd, hid, rows_dense, hid, channels, params[5], 1};
    HPFG_RETURN_IF((launch_gemm<true, true>(g, st)));
    g = GemmArgs{hd, hid, params[6], hid, out_dense, out, rows_dense, out, hid, params[7], 0, nullptr, nullptr, s};
    HPFG_RETURN_IF((launch_gemm<true, true>(g, st)));
    return HPFG_OK;
}

extern "C" int hpfg_neck_backward(const float *d_global, const float *d_dense, int n, int channels, int height, int width, int s,
                                  int hid, int out, const float *const *params, const float *pooled, const float *hidden,
                                  float *const *grads, float *dx, float *scratch, void *stream) {
    HPFG_REQUIRE(d_global && d_dense && params && pooled && hidden && grads && scratch, "hpfg_neck_backward: null buffer");
    for (int i = 0; i < 8; ++i) HPFG_REQUIRE(params[i] && grads[i], "hpfg_neck_backward: null parameter / gradient tensor");
    HPFG_REQUIRE(n > 0 && channels > 0 && hid > 0 && out > 0 && s >= 1 && s <= height && s <= width, "hpfg_neck_backward: bad shape");
    cudaStream_t st = (cudaStream_t)stream;
    const int S = s * s, rows_dense = n * S, rows = n + rows_dense;
    // scratch: d_dense as rows [n*S, out] | hidden gradient [rows, hid] | pooled gradient [rows, C]
    float *drows = scratch, *dhid = drows + (int64_t)rows_dense * out, *dpool = dhid + (int64_t)rows * hid;
    {
        ProfScope _prof(PROF_GLUE, st);
        const int64_t total = (int64_t)rows_dense * out;
        HPFG_CUDA_CHECK(launch_pdl(neck_dense_to_rows_kernel, dim3(ceil_div(total, 256)), dim3(256), 0, st, d_dense, out, S, drows, total));
        HPFG_LAUNCH_CHECK();
    }
    {
        ProfScope _prof(PROF_CONV_CUDA, st);
        for (int br = 0; br < 2; ++br) {
            const int r0 = br ? n : 0, nr = br ? rows_dense : n, p = br * 4;
            const float *dO = br ? drows : d_global;
            const float *hb = hidden + (int64_t)r0 * hid, *pb = pooled + (int64_t)r0 * channels;
            float *dh = dhid + (int64_t)r0 * hid, *dp = dpool + (int64_t)r0 * channels;
            GemmArgs g;
            // dW2[o,j] = sum_r dO[r,o] hidden[r,j], db2 = column sums of dO
            g = GemmArgs{dO, out, hb, hid, grads[p + 2], hid, out, hid, nr, nullptr, 0, nullptr, grads[p + 3]};
            HPFG_RETURN_IF((launch_gemm<false, false>(g, st)));
            // dhidden = (dO W2) * (hidden > 0)
            g = GemmArgs{dO, out, params[p + 2], hid, dh, hid, nr, hid, out, nullptr, 0, hb};
            HPFG_RETURN_IF((launch_gemm<true, false>(g, st)));
            // dW1[j,c] = sum_r dhidden[r,j] pooled[r,c], db1 = column sums of dhidden
            g = GemmArgs{dh, hid, pb, channels, grads[p + 0], channels, hid, channels, nr, nullptr, 0, nullptr, grads[p + 1]};
            HPFG_RETURN_IF((launch_gemm<false, false>(g, st)));
            if (dx) {
                g = GemmArgs{dh, hid, params[p + 0], channels, dp, channels, nr, channels, hid};
                HPFG_RETURN_IF((launch_gemm<true, false>(g, st)));
            }
        }
    }
    if (dx) {
        ProfScope _prof(PROF_GLUE, st);
        const int64_t total = (int64_t)n * channels * height * width;
        const int blocks = (int)(ceil_div(total, 256) < (int64_t)kNumSMs * 16 ? ceil_div(total, 256) : kNumSMs * 16);
        HPFG_CUDA_CHECK(launch_pdl(neck_pool_bwd_kernel, dim3(blocks), dim3(256), 0, st, dpool, n, channels, height, width, s, dx, total));
        HPFG_LAUNCH_CHECK();
    }
    return HPFG_OK;
}

extern "C" int64_t hpfg_dense_contrastive_workspace_floats(int batch, int dim, int positions) {
    const int64_t rows = 2ll * batch;
    return rows * dim * positions + rows * positions + rows * rows + 2 * rows;
}

extern "C" int hpfg_dense_contrastive_scaled(const float *out1, const float *out2, int batch, int dim, int positions, float temperature,
                                             float scale, const float *scale_dev, float *loss, float *d_out1, float *workspace,
                                             void *stream) {
    HPFG_REQUIRE(out1 && out2 && loss && workspace, "hpfg_dense_contrastive: null buffer");
    HPFG_REQUIRE(batch > 0 && dim > 0 && positions > 0, "hpfg_dense_contrastive: empty problem");
    HPFG_REQUIRE(temperature > 0.f, "hpfg_dense_contrastive: temperature must be positive");
    const int64_t V = (int64_t)dim * positions, rows = 2ll * batch;
    const size_t smem = (size_t)(V + rows + 2) * sizeof(float);
    HPFG_REQUIRE(smem <= 96 * 1024 && rows <= 4096, "hpfg_dense_contrastive: feature vector too long for one CTA's shared memory");
    cudaStream_t st = (cudaStream_t)stream;
    float *z = workspace, *norms = z + rows * V, *P = norms + rows * positions, *rowloss = P + rows * rows, *miss = rowloss + rows;
    ProfScope _prof(PROF_LOSS, st);
    if (smem > 48 * 1024) {
        HPFG_CUDA_CHECK(cudaFuncSetAttribute(contrast_rows_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 96 * 1024));
        HPFG_CUDA_CHECK(cudaFuncSetAttribute(contrast_grad_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 96 * 1024));
    }
    const float inv_t = 1.f / temperature;
    HPFG_CUDA_CHECK(launch_pdl(contrast_normalize_kernel, dim3((unsigned)rows), dim3(256), 0, st, out1, out2, batch, dim, positions, z, norms));
    HPFG_LAUNCH_CHECK();
    HPFG_CUDA_CHECK(launch_pdl(contrast_rows_kernel, dim3((unsigned)rows), dim3(256), smem, st, (const float *)z, batch, (int)V, inv_t, P, miss, rowloss));
    HPFG_LAUNCH_CHECK();
    HPFG_CUDA_CHECK(launch_pdl(contrast_grad_kernel, dim3(d_out1 ? batch : 1), dim3(256), smem, st, (const float *)z, (const float *)norms,
                               (const float *)P, (const float *)miss, (const float *)rowloss, batch, dim, positions, inv_t, scale, scale_dev,
                               loss, d_out1));
    HPFG_LAUNCH_CHECK();
    return HPFG_OK;
}

extern "C" int hpfg_dense_contrastive(const float *out1, const float *out2, int batch, int dim, int positions, float temperature,
                                      float *loss, float *d_out1, float *workspace, void *stream) {
    return hpfg_dense_contrastive_scaled(out1, out2, batch, dim, positions, temperature, 1.f, nullptr, loss, d_out1, workspace, stream);
}
