// Fused SSL loss: softmax, cross-entropy, batch-wide soft Dice, Mean-Teacher softmax-MSE consistency, CPS
// argmax pseudo-labelling and UAMT uncertainty masking, forward value AND d loss / d logits.
//   utils/loss/medloss.py:5-56 (Med_Sup_Loss, DiceLoss), utils/loss/diceloss.py:64-81,155-191,
//   2017_03_NIPS_Mean-Teacher_ACDC.py:97-106, 2021_06_CVPR_CPS_ACDC.py:99-111,
//   2019_07_MICCAI_Uncertainty_Aware_ACDC.py:145-162,
//   2022_02_ISBI_ICT-MedSeg_ACDC.py:111-137 (ICT: consistency against a per-sample mix of two teacher softmaxes),
//   2022_08_CVPR_S4CVNet_ACDC.py:124-156 (two students, Dice-only cross pseudo supervision + Mean-Teacher MSE).
// Dice is a ratio of batch-wide sums, so the gradient needs those sums first: phase 1 (reduce kernel) streams the logits that
// carry batch-wide sums and reduces with warp shuffles -> one double atomic per block per quantity; phase 2 (grad kernel)
// streams all logits (L2-resident: they are << 126 MB) and writes dlogits.  Only the LABELED images carry such sums in the
// SUP / Mean-Teacher / ICT modes (Dice and the CE normaliser); the consistency term's gradient 2w/M*(p-q) needs none, so
// its VALUE is accumulated by the gradient kernel itself and the last CTA to finish writes the loss scalars -- the reduce
// kernel then touches n_l of the n_l+n_u images.  CPS / S4CV (pseudo-label Dice over the unlabeled images) and UAMT
// (mask count) still reduce over the whole batch.  NCHW fp32, 4 consecutive pixels per thread, 128-bit loads per class plane.
// Mean-Teacher (the headline step) goes one step further: loss_mt_one_kernel does both phases in ONE launch on a co-resident
// grid with a grid barrier between the labeled sums and the labeled gradient (the unlabeled gradient runs in between); the
// two-launch path remains for the other modes and for the exact-global data-parallel mode (an all-reduce sits between the phases).
// Algorithmic bytes (MT): (n_l+n_u)*C*HW*4 read + n_u*C*HW*4 read + n_l*HW*8 read + (n_l+n_u)*C*HW*4 written.
#include "common.cuh"
#include <cstdlib>

#ifndef HPFG_LOSS_MT_MINBLOCKS
#define HPFG_LOSS_MT_MINBLOCKS 3
#endif

namespace hpfg {

constexpr int kMaxC = 8;
constexpr int kAccPerSet = 3 * kMaxC + 2;   // I[8] Z[8] Y[8] ce n_valid
constexpr int kAccMse = 4 * kAccPerSet;     // after the 4 (net,set) groups
constexpr int kAccMaskSum = kAccMse + 1;
constexpr int kAccMaskedDist = kAccMse + 2;
constexpr int kAccTotal = 128;
constexpr int kAccTicket = kAccTotal - 1;   // last slot, used as an unsigned block counter by the gradient kernel (MT / ICT)
constexpr float kDiceSmooth = 1e-5f;

struct LossArgs {
    int mode, n_l, n_u, hw, mc_passes;
    const float *student, *other, *mc;
    const float *mix;               // ICT: per-sample mix factor lambda[n_u] (device)
    const int64_t *labels;
    float cons_weight, uamt_threshold, ce_coef, dice_coef;
    float cons_weight2;             // S4CV: weight of the Mean-Teacher MSE terms (cons_weight = weight of the pseudo Dice terms)
    const float *cons_weight_dev;   // optional device scalar overriding cons_weight (CUDA-graph replays)
    const float *cons_weight2_dev;  // same for cons_weight2
    const float *uamt_threshold_dev;   // same for uamt_threshold
    float class_w[kMaxC];
    float *dstudent, *dother, *scalars;
    int64_t *pseudo1, *pseudo2;
    double *acc;
    uint8_t *aux;   // CPS: pl1 | pl2 (n_u*hw each); UAMT: mask (n_u*hw)
    int world;         // exact-global mode: number of ranks whose sums were all-reduced into acc (1 otherwise)
    int reduce_imgs;   // images the reduce kernel streams: n_l for SUP / MT / ICT (their global sums only involve labeled pixels)
    FastDiv qdiv;   // division by hw/4 without the 64-bit integer divide (quad index -> image, quad in image)
};

template <int C>
__device__ __forceinline__ void load4(const float *base, int64_t hw, float (&z)[C][4]) {
#pragma unroll
    for (int c = 0; c < C; ++c) {
        const float4 v = __ldg(reinterpret_cast<const float4 *>(base + (int64_t)c * hw));
        z[c][0] = v.x; z[c][1] = v.y; z[c][2] = v.z; z[c][3] = v.w;
    }
}

template <int C>
__device__ __forceinline__ void softmax4(const float (&z)[C][4], float (&p)[C][4], float (&lse)[4]) {
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        float m = z[0][j];
#pragma unroll
        for (int c = 1; c < C; ++c) m = fmaxf(m, z[c][j]);
        float s = 0.f;
#pragma unroll
        for (int c = 0; c < C; ++c) { p[c][j] = expf(z[c][j] - m); s += p[c][j]; }
        const float inv = 1.f / s;
#pragma unroll
        for (int c = 0; c < C; ++c) p[c][j] *= inv;
        lse[j] = m + logf(s);
    }
}

// Gradient kernel: probabilities only, exponentials through ex2.approx (FMUL + MUFU.EX2 instead of the ~8-instruction
// accurate expf; relative error ~1e-6, well inside the 1e-5 gradient bar; no argmax / pseudo-label is taken from these values
// and the loss VALUE and the batch-wide sums still come from the accurate softmax of the reduce kernel).
template <int C>
__device__ __forceinline__ void softmax4g(const float (&z)[C][4], float (&p)[C][4]) {
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        float m = z[0][j];
#pragma unroll
        for (int c = 1; c < C; ++c) m = fmaxf(m, z[c][j]);
        float s = 0.f;
#pragma unroll
        for (int c = 0; c < C; ++c) { p[c][j] = __expf(z[c][j] - m); s += p[c][j]; }
        const float inv = __fdividef(1.f, s);
#pragma unroll
        for (int c = 0; c < C; ++c) p[c][j] *= inv;
    }
}

template <int C>
__device__ __forceinline__ int argmax_first(const float (&p)[C][4], int j) {
    int best = 0;
    float bv = p[0][j];
#pragma unroll
    for (int c = 1; c < C; ++c)
        if (p[c][j] > bv) { bv = p[c][j]; best = c; }
    return best;
}

// accumulate CE + Dice partial sums of 4 pixels against labels lab[4] (255 -> ignored by CE, no class for Dice)
template <int C>
__device__ __forceinline__ void acc_sup(const float (&z)[C][4], const float (&p)[C][4], const float (&lse)[4],
                                        const int (&lab)[4], float (&a)[3 * C + 2]) {
#pragma unroll
    for (int j = 0; j < 4; ++j) {
#pragma unroll
        for (int c = 0; c < C; ++c) {
            const float t = (lab[j] == c) ? 1.f : 0.f;
            a[c] += p[c][j] * t;
            a[C + c] += p[c][j] * p[c][j];
            a[2 * C + c] += t;
            if (lab[j] == c) a[3 * C] += lse[j] - z[c][j];
        }
        if (lab[j] != 255) a[3 * C + 1] += 1.f;
    }
}

template <int N>
__device__ __forceinline__ void flush(float (&a)[N], double *dst_base, const int *slot, float *smem) {
    // warp reduce each accumulator, then cross-warp through shared memory, then one atomic per block
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarp = blockDim.x >> 5;
#pragma unroll
    for (int i = 0; i < N; ++i) {
        const float v = warp_sum(a[i]);
        if (lane == 0) smem[warp * N + i] = v;
    }
    __syncthreads();
    if (threadIdx.x < N) {
        double s = 0.0;
        for (int w = 0; w < nwarp; ++w) s += (double)smem[w * N + threadIdx.x];
        if (s != 0.0) atomicAdd(dst_base + slot[threadIdx.x], s);
    }
    __syncthreads();
}

__device__ __forceinline__ void load_labels4(const int64_t *p, int (&lab)[4]) {
    const longlong2 a = __ldg(reinterpret_cast<const longlong2 *>(p));
    const longlong2 b = __ldg(reinterpret_cast<const longlong2 *>(p + 2));
    lab[0] = (int)a.x; lab[1] = (int)a.y; lab[2] = (int)b.x; lab[3] = (int)b.y;
}

// ---------------------------------------------------------------------------------------------- phase 1
// MODE is a template parameter: the generic kernel carried four accumulator sets (177 registers, one CTA per SM, 12 %
// warps active in ncu); Mean-Teacher needs one.
template <int C, int MODE>
__global__ void __launch_bounds__(256, MODE == HPFG_LOSS_S4CV ? 1 : 2) loss_reduce_kernel(LossArgs A) {
    pdl_prologue();
    constexpr bool TWO = MODE == HPFG_LOSS_CPS || MODE == HPFG_LOSS_S4CV;   // two student networks
    if (MODE == HPFG_LOSS_UAMT && A.uamt_threshold_dev) A.uamt_threshold = *A.uamt_threshold_dev;
    constexpr int NS = 3 * C + 2;
    __shared__ float smem[8 * (2 * NS + 3)];
    __shared__ int slots[2 * NS + 3];
    const int64_t hw = A.hw, q_per_img = hw >> 2;
    const int64_t n_img = A.reduce_imgs;
    const int64_t total_q = n_img * q_per_img;
    constexpr int NSETS = TWO ? 2 : 1;
    float sl[NSETS][NS];   // labeled sums, net 0 / net 1 (CPS, S4CV)
    float su[NSETS][NS];   // CPS, S4CV: unlabeled sums wrt the peer's pseudo labels
    float misc[3] = {0.f, 0.f, 0.f};   // mse, mask_sum, masked_dist (S4CV: mse net 1, mse net 2)
#pragma unroll
    for (int i = 0; i < NS; ++i)
#pragma unroll
        for (int e = 0; e < NSETS; ++e) sl[e][i] = su[e][i] = 0.f;

    for (uint32_t q = blockIdx.x * blockDim.x + threadIdx.x; q < (uint32_t)total_q; q += gridDim.x * blockDim.x) {
        uint32_t img32, rem32;
        fast_divmod(q, A.qdiv, img32, rem32);
        const int64_t img = img32, pix = (int64_t)rem32 << 2;
        // every global load of this quad is issued before any math: one DRAM round trip per iteration instead of two or
        // three dependent ones (the loads sit behind warp-uniform branches, so the compiler cannot hoist them itself)
        const bool labeled = img < A.n_l;
        const int64_t u = img - A.n_l;
        float z[C][4], p[C][4], lse[4], z2[C][4], z3[C][4];
        int lab[4];
        load4<C>(A.student + (img * C) * hw + pix, hw, z);
        if (labeled) load_labels4(A.labels + img * hw + pix, lab);
        if (MODE != HPFG_LOSS_SUP && (TWO || !labeled))
            load4<C>(TWO ? A.other + (img * C) * hw + pix : A.other + (u * C) * hw + pix, hw, z2);
        if (MODE == HPFG_LOSS_ICT && !labeled) load4<C>(A.other + ((u + A.n_u) * C) * hw + pix, hw, z3);
        softmax4<C>(z, p, lse);
        if (labeled) {
            acc_sup<C>(z, p, lse, lab, sl[0]);
            if (TWO) {
                float p2[C][4], lse2[4];
                softmax4<C>(z2, p2, lse2);
                acc_sup<C>(z2, p2, lse2, lab, sl[NSETS - 1]);
            }
        } else if (MODE != HPFG_LOSS_SUP) {
            float p2[C][4], lse2[4];
            softmax4<C>(z2, p2, lse2);
            // (the MT and ICT branches below are kept for reference but no longer instantiated: launch_loss runs the SUP
            // instantiation over the labeled images for those modes and the gradient kernel sums the consistency value)
            if (MODE == HPFG_LOSS_MT) {
#pragma unroll
                for (int j = 0; j < 4; ++j)
#pragma unroll
                    for (int c = 0; c < C; ++c) { const float d = p[c][j] - p2[c][j]; misc[0] += d * d; }
            } else if (MODE == HPFG_LOSS_ICT) {   // target = (1-lambda)*softmax(teacher(ux0)) + lambda*softmax(teacher(ux1))
                float p3[C][4], lse3[4];
                softmax4<C>(z3, p3, lse3);
                const float lam = __ldg(A.mix + u), oml = 1.0f - lam;
#pragma unroll
                for (int j = 0; j < 4; ++j)
#pragma unroll
                    for (int c = 0; c < C; ++c) {
                        const float d = p[c][j] - (p2[c][j] * oml + p3[c][j] * lam);
                        misc[0] += d * d;
                    }
            } else if (TWO) {
                int pl1[4], pl2[4];
#pragma unroll
                for (int j = 0; j < 4; ++j) { pl1[j] = argmax_first<C>(p, j); pl2[j] = argmax_first<C>(p2, j); }
                acc_sup<C>(z, p, lse, pl2, su[0]);      // net 1 learns from net 2's labels
                acc_sup<C>(z2, p2, lse2, pl1, su[NSETS - 1]);   // and vice versa
                const int64_t o = u * hw + pix;
                *reinterpret_cast<uchar4 *>(A.aux + o) = make_uchar4(pl1[0], pl1[1], pl1[2], pl1[3]);
                *reinterpret_cast<uchar4 *>(A.aux + (int64_t)A.n_u * hw + o) = make_uchar4(pl2[0], pl2[1], pl2[2], pl2[3]);
                if (A.pseudo1)
                    for (int j = 0; j < 4; ++j) A.pseudo1[o + j] = pl1[j];
                if (A.pseudo2)
                    for (int j = 0; j < 4; ++j) A.pseudo2[o + j] = pl2[j];
                if (MODE == HPFG_LOSS_S4CV && A.mc) {   // both students against the one EMA teacher
                    float zt[C][4], pt[C][4], lt[4];
                    load4<C>(A.mc + (u * C) * hw + pix, hw, zt);
                    softmax4<C>(zt, pt, lt);
#pragma unroll
                    for (int j = 0; j < 4; ++j)
#pragma unroll
                        for (int c = 0; c < C; ++c) {
                            const float d1 = p[c][j] - pt[c][j], d2 = p2[c][j] - pt[c][j];
                            misc[0] += d1 * d1;
                            misc[1] += d2 * d2;
                        }
                }
            } else {   // UAMT: mean softmax of the T stochastic teacher passes -> entropy -> mask
                float mean[C][4];
#pragma unroll
                for (int c = 0; c < C; ++c)
#pragma unroll
                    for (int j = 0; j < 4; ++j) mean[c][j] = 0.f;
                for (int t = 0; t < A.mc_passes; ++t) {
                    float zm[C][4], pm[C][4], lm[4];
                    load4<C>(A.mc + (((int64_t)t * A.n_u + u) * C) * hw + pix, hw, zm);
                    softmax4<C>(zm, pm, lm);
#pragma unroll
                    for (int c = 0; c < C; ++c)
#pragma unroll
                        for (int j = 0; j < 4; ++j) mean[c][j] += pm[c][j];
                }
                const float invT = 1.f / (float)A.mc_passes;
                unsigned char mk[4];
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    float ent = 0.f, dist = 0.f;
#pragma unroll
                    for (int c = 0; c < C; ++c) {
                        const float m = mean[c][j] * invT;
                        ent -= m * logf(m + 1e-6f);
                        const float d = p[c][j] - p2[c][j];
                        dist += d * d;
                    }
                    mk[j] = ent < A.uamt_threshold ? 1 : 0;
                    if (mk[j]) { misc[1] += 1.f; misc[2] += dist; }
                }
                *reinterpret_cast<uchar4 *>(A.aux + u * hw + pix) = make_uchar4(mk[0], mk[1], mk[2], mk[3]);
            }
        }
    }
    // map compact per-thread accumulators to the global slots (class index padded to kMaxC)
    auto slot_of = [](int set_base, int i) {
        const int grp = i / C, c = i % C;
        return set_base + (grp < 3 ? grp * kMaxC + c : 3 * kMaxC + (i - 3 * C));
    };
    if (threadIdx.x < NS) slots[threadIdx.x] = slot_of(0, threadIdx.x);
    __syncthreads();
    flush<NS>(sl[0], A.acc + 0 * kAccPerSet, slots, smem);
    if (TWO) {
        flush<NS>(sl[NSETS - 1], A.acc + 2 * kAccPerSet, slots, smem);
        flush<NS>(su[0], A.acc + 1 * kAccPerSet, slots, smem);
        flush<NS>(su[NSETS - 1], A.acc + 3 * kAccPerSet, slots, smem);
    }
    if (MODE == HPFG_LOSS_MT || MODE == HPFG_LOSS_UAMT || MODE == HPFG_LOSS_ICT || MODE == HPFG_LOSS_S4CV) {
        if (threadIdx.x < 3) slots[threadIdx.x] = threadIdx.x;
        __syncthreads();
        flush<3>(misc, A.acc + kAccMse, slots, smem);
    }
}

// ---------------------------------------------------------------------------------------------- phase 2
// per-(net,set) coefficients derived from the global sums
struct SupCoef {
    float alpha[kMaxC], beta[kMaxC], inv_nv, ce, dice;
};

template <int C>
__device__ void make_coef(const double *acc, const float *cw, SupCoef &k) {
    double dice = 0.0;
    for (int c = 0; c < C; ++c) {
        const double I = acc[c], Z = acc[kMaxC + c], Y = acc[2 * kMaxC + c];
        const double D = Z + Y + (double)kDiceSmooth;
        const double num = 2.0 * I + (double)kDiceSmooth;
        dice += (1.0 - num / D) * (double)cw[c];
        k.alpha[c] = (float)(-2.0 * cw[c] / (C * D));
        k.beta[c] = (float)(2.0 * cw[c] * num / (C * D * D));
    }
    const double nv = acc[3 * kMaxC + 1];
    k.dice = (float)(dice / C);
    k.ce = (float)(acc[3 * kMaxC] / nv);
    k.inv_nv = (float)(1.0 / nv);
}

// gradient of coef_ce*CE + coef_dice*Dice wrt the logits of 4 pixels, times `scale`
template <int C>
__device__ __forceinline__ void grad_sup(const float (&p)[C][4], const int (&lab)[4], const SupCoef &k, float ce_coef,
                                         float dice_coef, float scale, float (&g)[C][4]) {
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        float a[C], dot = 0.f;
#pragma unroll
        for (int c = 0; c < C; ++c) {
            const float t = (lab[j] == c) ? 1.f : 0.f;
            a[c] = dice_coef * (k.alpha[c] * t + k.beta[c] * p[c][j]);
            dot += p[c][j] * a[c];
        }
        const float cev = (lab[j] != 255) ? ce_coef * k.inv_nv : 0.f;
#pragma unroll
        for (int c = 0; c < C; ++c) {
            const float t = (lab[j] == c) ? 1.f : 0.f;
            g[c][j] = scale * (p[c][j] * (a[c] - dot) + cev * (p[c][j] - t));
        }
    }
}

template <int C>
__device__ __forceinline__ void grad_mse(const float (&p)[C][4], const float (&q)[C][4], const float (&coef)[4],
                                         float (&g)[C][4], float *sq = nullptr) {
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        float a[C], dot = 0.f;
#pragma unroll
        for (int c = 0; c < C; ++c) {
            const float d = p[c][j] - q[c][j];
            if (sq) *sq += d * d;
            a[c] = coef[j] * d;
            dot += p[c][j] * a[c];
        }
#pragma unroll
        for (int c = 0; c < C; ++c) g[c][j] = p[c][j] * (a[c] - dot);
    }
}

template <int C>
__device__ __forceinline__ void store4(float *base, int64_t hw, const float (&g)[C][4]) {
#pragma unroll
    for (int c = 0; c < C; ++c)
        *reinterpret_cast<float4 *>(base + (int64_t)c * hw) = make_float4(g[c][0], g[c][1], g[c][2], g[c][3]);
}

// MODE: a compile-time copy of A.mode for the modes that get their own instantiation (Mean-Teacher: the headline step), -1 = read
// A.mode at run time.  Same expressions either way; the specialised kernel drops the CPS / S4CV / UAMT / ICT paths and their
// registers (128 -> see -Xptxas -v), so more CTAs are resident per SM and more loads are in flight.
template <int C, int MODE>
__global__ void __launch_bounds__(256, MODE == HPFG_LOSS_MT ? HPFG_LOSS_MT_MINBLOCKS : 1) loss_grad_kernel(LossArgs A) {
    pdl_prologue();
    if (MODE >= 0) A.mode = MODE;
    if (A.cons_weight_dev) A.cons_weight = *A.cons_weight_dev;
    if (A.cons_weight2_dev) A.cons_weight2 = *A.cons_weight2_dev;
    __shared__ SupCoef coef[4];   // [net*2 + set]
    __shared__ float s_cons;      // per-element consistency coefficient
    const bool s4cv = A.mode == HPFG_LOSS_S4CV;
    const bool cps = A.mode == HPFG_LOSS_CPS || s4cv;   // two student networks
    // Mean-Teacher / ICT: the consistency VALUE is accumulated here, next to its gradient, so the reduce kernel only has to
    // stream the labeled images (the Dice / CE sums); the last CTA to finish writes loss and consistency term
    const bool late_mse = A.mode == HPFG_LOSS_MT || A.mode == HPFG_LOSS_ICT;
    float mse_local = 0.f;
    // weights of the pseudo-label terms: CPS = Med_Sup_Loss on the peer's labels, S4CV = Dice only (2022_08...:139-140)
    const float ps_ce = s4cv ? 0.f : A.ce_coef, ps_dice = s4cv ? 1.f : A.dice_coef;
    if (threadIdx.x == 0) {
        make_coef<C>(A.acc + 0 * kAccPerSet, A.class_w, coef[0]);
        if (cps) {
            make_coef<C>(A.acc + 1 * kAccPerSet, A.class_w, coef[1]);
            make_coef<C>(A.acc + 2 * kAccPerSet, A.class_w, coef[2]);
            make_coef<C>(A.acc + 3 * kAccPerSet, A.class_w, coef[3]);
        }
        float cons = 0.f, cons_val = 0.f;
        const double M = (double)A.n_u * C * (double)A.hw * (double)A.world;      // elements of the consistency mean (all ranks)
        if (late_mse) {   // the squared distance is summed by THIS kernel (below); its gradient needs no global sum
            cons = (float)(2.0 * A.cons_weight / M);
        } else if (s4cv) {
            cons_val = (float)((A.acc[kAccMse] + A.acc[kAccMse + 1]) / M);   // consistency_loss1 + consistency_loss2
            cons = (float)(2.0 * A.cons_weight2 / M);
        } else if (A.mode == HPFG_LOSS_UAMT) {
            const double den = 2.0 * A.acc[kAccMaskSum] + 1e-16;
            cons_val = (float)(A.acc[kAccMaskedDist] / den);
            cons = (float)(2.0 * A.cons_weight / den);
        }
        s_cons = cons;
        if (blockIdx.x == 0) {
            const float sup0 = A.ce_coef * coef[0].ce + A.dice_coef * coef[0].dice;
            float sup = sup0, aux = cons_val;
            if (cps) {
                sup = sup0 + A.ce_coef * coef[2].ce + A.dice_coef * coef[2].dice;
                aux = ps_ce * coef[1].ce + ps_dice * coef[1].dice + ps_ce * coef[3].ce + ps_dice * coef[3].dice;
            }
            float loss = (A.mode == HPFG_LOSS_SUP) ? sup : sup + A.cons_weight * aux;
            float s6 = (float)A.acc[kAccMaskSum], s7 = 0.f;
            if (s4cv) {   // loss_semi = w_cps*(ps1+ps2) + w_mt*(cl1+cl2); scalars: [2] loss_semi, [6] ps1+ps2, [7] cl1+cl2
                const float semi = A.cons_weight * aux + A.cons_weight2 * cons_val;
                loss = sup + semi;
                s6 = aux;
                s7 = cons_val;
                aux = semi;
            }
            if (!late_mse) {
                A.scalars[0] = loss;
                A.scalars[2] = aux;
            }
            A.scalars[1] = sup;
            A.scalars[3] = coef[0].ce;
            A.scalars[4] = coef[0].dice;
            A.scalars[5] = (float)A.acc[3 * kMaxC + 1];
            A.scalars[6] = s6;
            A.scalars[7] = s7;
        }
    }
    __syncthreads();
    const int64_t hw = A.hw, q_per_img = hw >> 2;
    const int64_t total_q = (int64_t)(A.n_l + A.n_u) * q_per_img;
    for (uint32_t q = blockIdx.x * blockDim.x + threadIdx.x; q < (uint32_t)total_q; q += gridDim.x * blockDim.x) {
        uint32_t img32, rem32;
        fast_divmod(q, A.qdiv, img32, rem32);
        const int64_t img = img32, pix = (int64_t)rem32 << 2;
        const int64_t so = (img * C) * hw + pix;
        float z[C][4], p[C][4], g[C][4];
        if (img < A.n_l) {
            int lab[4];
            load_labels4(A.labels + img * hw + pix, lab);
            load4<C>(A.student + so, hw, z);
            softmax4g<C>(z, p);
            grad_sup<C>(p, lab, coef[0], A.ce_coef, A.dice_coef, 1.f, g);
            store4<C>(A.dstudent + so, hw, g);
            if (cps) {
                load4<C>(A.other + so, hw, z);
                softmax4g<C>(z, p);
                grad_sup<C>(p, lab, coef[2], A.ce_coef, A.dice_coef, 1.f, g);
                store4<C>(A.dother + so, hw, g);
            }
            continue;
        }
        const int64_t u = img - A.n_l;
        if (A.mode == HPFG_LOSS_SUP) {
#pragma unroll
            for (int c = 0; c < C; ++c)
#pragma unroll
                for (int j = 0; j < 4; ++j) g[c][j] = 0.f;
            store4<C>(A.dstudent + so, hw, g);
            continue;
        }
        float z2[C][4];      // second source (peer / teacher), requested before the student's softmax math
        load4<C>(A.student + so, hw, z);
        load4<C>(cps ? A.other + so : A.other + (u * C) * hw + pix, hw, z2);
        softmax4g<C>(z, p);
        if (cps) {
            const uchar4 a1 = *reinterpret_cast<const uchar4 *>(A.aux + u * hw + pix);
            const uchar4 a2 = *reinterpret_cast<const uchar4 *>(A.aux + (int64_t)A.n_u * hw + u * hw + pix);
            const int pl1[4] = {a1.x, a1.y, a1.z, a1.w}, pl2[4] = {a2.x, a2.y, a2.z, a2.w};
            float zt[C][4], pt[C][4], gm[C][4];
            const bool mse = s4cv && A.mc != nullptr;
            const float cf4[4] = {s_cons, s_cons, s_cons, s_cons};
            if (mse) {
                load4<C>(A.mc + (u * C) * hw + pix, hw, zt);
                softmax4g<C>(zt, pt);
            }
            grad_sup<C>(p, pl2, coef[1], ps_ce, ps_dice, A.cons_weight, g);
            if (mse) {
                grad_mse<C>(p, pt, cf4, gm);
#pragma unroll
                for (int c = 0; c < C; ++c)
#pragma unroll
                    for (int j = 0; j < 4; ++j) g[c][j] += gm[c][j];
            }
            store4<C>(A.dstudent + so, hw, g);
            softmax4g<C>(z2, p);
            grad_sup<C>(p, pl1, coef[3], ps_ce, ps_dice, A.cons_weight, g);
            if (mse) {
                grad_mse<C>(p, pt, cf4, gm);
#pragma unroll
                for (int c = 0; c < C; ++c)
#pragma unroll
                    for (int j = 0; j < 4; ++j) g[c][j] += gm[c][j];
            }
            store4<C>(A.dother + so, hw, g);
        } else {
            float q2[C][4], cf[4];
            softmax4g<C>(z2, q2);
            if (A.mode == HPFG_LOSS_ICT) {
                float z3[C][4], q3[C][4];
                load4<C>(A.other + ((u + A.n_u) * C) * hw + pix, hw, z3);
                softmax4g<C>(z3, q3);
                const float lam = __ldg(A.mix + u), oml = 1.0f - lam;
#pragma unroll
                for (int c = 0; c < C; ++c)
#pragma unroll
                    for (int j = 0; j < 4; ++j) q2[c][j] = q2[c][j] * oml + q3[c][j] * lam;
            }
            if (A.mode == HPFG_LOSS_UAMT) {
                const uchar4 mk = *reinterpret_cast<const uchar4 *>(A.aux + u * hw + pix);
                cf[0] = mk.x ? s_cons : 0.f; cf[1] = mk.y ? s_cons : 0.f;
                cf[2] = mk.z ? s_cons : 0.f; cf[3] = mk.w ? s_cons : 0.f;
            } else {
                cf[0] = cf[1] = cf[2] = cf[3] = s_cons;
            }
            grad_mse<C>(p, q2, cf, g, &mse_local);
            store4<C>(A.dstudent + so, hw, g);
        }
    }
    if (late_mse) {
        __shared__ float s_part[8];
        const float v = warp_sum(mse_local);
        if ((threadIdx.x & 31) == 0) s_part[threadIdx.x >> 5] = v;
        __syncthreads();
        if (threadIdx.x == 0) {
            double sum = 0.0;
            for (int w = 0; w < (int)(blockDim.x >> 5); ++w) sum += (double)s_part[w];
            atomicAdd(A.acc + kAccMse, sum);
            __threadfence();
            const unsigned ticket = atomicAdd(reinterpret_cast<unsigned *>(A.acc + kAccTicket), 1u);
            if (ticket == gridDim.x - 1) {      // every CTA's partial is in: finish the scalars
                __threadfence();
                const double total = atomicAdd(A.acc + kAccMse, 0.0);
                const float cons_val = (float)(total / ((double)A.n_u * C * (double)A.hw * (double)A.world));   // this rank's share
                const float sup = A.ce_coef * coef[0].ce + A.dice_coef * coef[0].dice;
                A.scalars[0] = sup + A.cons_weight * cons_val;
                A.scalars[2] = cons_val;
            }
        }
    }
}

// ------------------------------------------------------------------------------------ Mean-Teacher, one launch
// The Mean-Teacher step (2017_03_NIPS_Mean-Teacher_ACDC.py:97-106) in ONE launch on a co-resident grid:
//   phase A  Dice / CE sums of the labeled images (accurate softmax, as loss_reduce_kernel) -> double atomics, then ARRIVE;
//   phase B  gradient and value of the consistency term on the unlabeled images -- 3/4 of the bytes, needs no batch-wide sum,
//            so it runs while the other CTAs' phase-A atomics land;
//   barrier  wait until every CTA has arrived (all CTAs are resident: the host clamps the grid to the occupancy of this kernel,
//            and the dependent kernel is only released -- griddepcontrol.launch_dependents -- after the barrier, so its CTAs can
//            never hold the slots of CTAs the barrier is waiting for);
//   phase C  coefficients from the sums, gradient of the labeled images (their logits are L2 hits by now); the last CTA to finish
//            writes the scalars.
// Replaces the reduce launch (8.8 us for 9.6 MB: a latency-bound launch on the critical path) of the two-launch scheme.
constexpr int kAccBarrier = kAccTotal - 2;    // unsigned arrive counter of the grid barrier

template <int C>
__global__ void __launch_bounds__(256, 3) loss_mt_one_kernel(LossArgs A) {
    pdl_wait();
    if (A.cons_weight_dev) A.cons_weight = *A.cons_weight_dev;
    constexpr int NS = 3 * C + 2;
    __shared__ float smem[8 * NS];
    __shared__ int slots[NS];
    __shared__ SupCoef coef;
    __shared__ float s_part[8];
    const int64_t hw = A.hw, q_per_img = hw >> 2;
    const uint32_t lab_q = (uint32_t)(A.n_l * q_per_img), total_q = (uint32_t)((A.n_l + A.n_u) * q_per_img);
    const uint32_t tid0 = blockIdx.x * blockDim.x + threadIdx.x, stride = gridDim.x * blockDim.x;
    // ---- phase A
    {
        float sl[NS];
#pragma unroll
        for (int i = 0; i < NS; ++i) sl[i] = 0.f;
        for (uint32_t q = tid0; q < lab_q; q += stride) {
            uint32_t img32, rem32;
            fast_divmod(q, A.qdiv, img32, rem32);
            const int64_t img = img32, pix = (int64_t)rem32 << 2;
            float z[C][4], p[C][4], lse[4];
            int lab[4];
            load4<C>(A.student + (img * C) * hw + pix, hw, z);
            load_labels4(A.labels + img * hw + pix, lab);
            softmax4<C>(z, p, lse);
            acc_sup<C>(z, p, lse, lab, sl);
        }
        if (threadIdx.x < NS) {
            const int i = threadIdx.x, grp = i / C, c = i % C;
            slots[i] = grp < 3 ? grp * kMaxC + c : 3 * kMaxC + (i - 3 * C);
        }
        __syncthreads();
        flush<NS>(sl, A.acc, slots, smem);          // ends with __syncthreads(): this CTA's atomics are issued
    }
    unsigned *arrive = reinterpret_cast<unsigned *>(A.acc + kAccBarrier);
    if (threadIdx.x == 0) {
        __threadfence();
        atomicAdd(arrive, 1u);
    }
    // ---- phase B
    const float cons = (float)(2.0 * A.cons_weight / ((double)A.n_u * C * (double)A.hw));
    const float cf[4] = {cons, cons, cons, cons};
    float mse_local = 0.f;
    for (uint32_t q = lab_q + tid0; q < total_q; q += stride) {
        uint32_t img32, rem32;
        fast_divmod(q, A.qdiv, img32, rem32);
        const int64_t img = img32, pix = (int64_t)rem32 << 2, u = img - A.n_l;
        const int64_t so = (img * C) * hw + pix;
        float z[C][4], z2[C][4], p[C][4], q2[C][4], g[C][4];
        load4<C>(A.student + so, hw, z);
        load4<C>(A.other + (u * C) * hw + pix, hw, z2);
        softmax4g<C>(z, p);
        softmax4g<C>(z2, q2);
        grad_mse<C>(p, q2, cf, g, &mse_local);
        store4<C>(A.dstudent + so, hw, g);
    }
    // ---- barrier: every CTA's phase-A sums are in
    if (threadIdx.x == 0) {
        const long long t0 = clock64();
        while (*reinterpret_cast<volatile unsigned *>(arrive) < gridDim.x) {
            __nanosleep(40);
            if (clock64() - t0 > 6000000000LL) {      // bounded wait (~3 s): a protocol bug must trap, not hang the GPU
                printf("hpfg_b200: loss_mt_one_kernel grid barrier timed out (block %d of %d, arrived %u)\n", (int)blockIdx.x, (int)gridDim.x,
                       *reinterpret_cast<volatile unsigned *>(arrive));
                __trap();
            }
        }
        __threadfence();
        double acc[3 * kMaxC + 2];
        for (int i = 0; i < 3 * kMaxC + 2; ++i) acc[i] = __ldcg(A.acc + i);
        make_coef<C>(acc, A.class_w, coef);
        if (blockIdx.x == 0) {
            A.scalars[1] = A.ce_coef * coef.ce + A.dice_coef * coef.dice;
            A.scalars[3] = coef.ce;
            A.scalars[4] = coef.dice;
            A.scalars[5] = (float)acc[3 * kMaxC + 1];
            A.scalars[6] = 0.f;
            A.scalars[7] = 0.f;
        }
    }
    __syncthreads();
    pdl_launch_dependents();
    // ---- phase C
    for (uint32_t q = tid0; q < lab_q; q += stride) {
        uint32_t img32, rem32;
        fast_divmod(q, A.qdiv, img32, rem32);
        const int64_t img = img32, pix = (int64_t)rem32 << 2;
        const int64_t so = (img * C) * hw + pix;
        float z[C][4], p[C][4], g[C][4];
        int lab[4];
        load_labels4(A.labels + img * hw + pix, lab);
        load4<C>(A.student + so, hw, z);
        softmax4g<C>(z, p);
        grad_sup<C>(p, lab, coef, A.ce_coef, A.dice_coef, 1.f, g);
        store4<C>(A.dstudent + so, hw, g);
    }
    // ---- consistency value; the last CTA to finish writes loss and consistency term
    const float v = warp_sum(mse_local);
    if ((threadIdx.x & 31) == 0) s_part[threadIdx.x >> 5] = v;
    __syncthreads();
    if (threadIdx.x == 0) {
        double sum = 0.0;
        for (int w = 0; w < (int)(blockDim.x >> 5); ++w) sum += (double)s_part[w];
        atomicAdd(A.acc + kAccMse, sum);
        __threadfence();
        const unsigned ticket = atomicAdd(reinterpret_cast<unsigned *>(A.acc + kAccTicket), 1u);
        if (ticket == gridDim.x - 1) {
            __threadfence();
            const double total = atomicAdd(A.acc + kAccMse, 0.0);
            const float cons_val = (float)(total / ((double)A.n_u * C * (double)A.hw));
            const float sup = A.ce_coef * coef.ce + A.dice_coef * coef.dice;
            A.scalars[0] = sup + A.cons_weight * cons_val;
            A.scalars[2] = cons_val;
        }
    }
}

// -------------------------------------------------------------------------- stand-alone DiceLoss.forward
struct DiceArgs {
    const float *inputs;
    const int64_t *target;
    int n, hw, softmax;
    float class_w[kMaxC];
    float *dinputs, *scalars;
    double *acc;
};

template <int C>
__global__ void __launch_bounds__(256) dice_reduce_kernel(DiceArgs A) {
    pdl_prologue();
    constexpr int NS = 3 * C + 2;
    __shared__ float smem[8 * NS];
    __shared__ int slots[NS];
    const int64_t hw = A.hw, q_per_img = hw >> 2, total_q = (int64_t)A.n * q_per_img;
    float a[NS];
#pragma unroll
    for (int i = 0; i < NS; ++i) a[i] = 0.f;
    for (int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; q < total_q;
         q += (int64_t)gridDim.x * blockDim.x) {
        const int64_t img = q / q_per_img, pix = (q - img * q_per_img) << 2;
        float z[C][4], p[C][4], lse[4];
        int lab[4];
        load4<C>(A.inputs + (img * C) * hw + pix, hw, z);
        load_labels4(A.target + img * hw + pix, lab);
        if (A.softmax) {
            softmax4<C>(z, p, lse);
        } else {
#pragma unroll
            for (int c = 0; c < C; ++c)
#pragma unroll
                for (int j = 0; j < 4; ++j) p[c][j] = z[c][j];
            lse[0] = lse[1] = lse[2] = lse[3] = 0.f;
        }
        acc_sup<C>(z, p, lse, lab, a);
    }
    if (threadIdx.x < NS) {
        const int i = threadIdx.x, grp = i / C, c = i % C;
        slots[i] = grp < 3 ? grp * kMaxC + c : 3 * kMaxC + (i - 3 * C);
    }
    __syncthreads();
    flush<NS>(a, A.acc, slots, smem);
}

template <int C>
__global__ void __launch_bounds__(256) dice_grad_kernel(DiceArgs A) {
    pdl_prologue();
    __shared__ SupCoef k;
    if (threadIdx.x == 0) {
        make_coef<C>(A.acc, A.class_w, k);
        if (blockIdx.x == 0) {
            A.scalars[0] = k.dice;
            for (int c = 0; c < C; ++c) {
                const double I = A.acc[c], Z = A.acc[kMaxC + c], Y = A.acc[2 * kMaxC + c];
                A.scalars[1 + c] = (float)((2.0 * I + kDiceSmooth) / (Z + Y + kDiceSmooth));
            }
        }
    }
    __syncthreads();
    if (A.dinputs == nullptr) return;
    const int64_t hw = A.hw, q_per_img = hw >> 2, total_q = (int64_t)A.n * q_per_img;
    for (int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; q < total_q;
         q += (int64_t)gridDim.x * blockDim.x) {
        const int64_t img = q / q_per_img, pix = (q - img * q_per_img) << 2;
        float z[C][4], p[C][4], lse[4], g[C][4];
        int lab[4];
        load4<C>(A.inputs + (img * C) * hw + pix, hw, z);
        load_labels4(A.target + img * hw + pix, lab);
        if (A.softmax) {
            softmax4<C>(z, p, lse);
            grad_sup<C>(p, lab, k, 0.f, 1.f, 1.f, g);
        } else {
#pragma unroll
            for (int c = 0; c < C; ++c)
#pragma unroll
                for (int j = 0; j < 4; ++j)
                    g[c][j] = k.alpha[c] * ((lab[j] == c) ? 1.f : 0.f) + k.beta[c] * z[c][j];
        }
        store4<C>(A.dinputs + (img * C) * hw + pix, hw, g);
    }
}

static int loss_ctas_per_sm() {      // A/B knob (profiles/config_throughput.py): HPFG_LOSS_CTAS_PER_SM; default 2 = the resident CTAs per SM of both kernels (one wave, ~5 grid-stride iterations per thread: 52.6 -> 44.8 us per MT loss call, profiles/r01_loss_grid_ab.txt)
    static int v = [] {
        const char *e = getenv("HPFG_LOSS_CTAS_PER_SM");
        const int n = e ? atoi(e) : 0;
        return n > 0 ? n : 2;
    }();
    return v;
}

static int loss_mt_ctas_per_sm() {   // grid of the Mean-Teacher gradient kernel in CTAs per SM (its own instantiation, HPFG_LOSS_MT_MINBLOCKS resident)
    static int v = [] {
        const char *e = getenv("HPFG_LOSS_MT_CTAS_PER_SM");
        const int n = e ? atoi(e) : 0;
        return n > 0 ? n : HPFG_LOSS_MT_MINBLOCKS > 2 ? HPFG_LOSS_MT_MINBLOCKS : 2;
    }();
    return v;
}

static int loss_grid(int64_t quads, int ctas_per_sm = 0) {
    int64_t blocks = (quads + 255) / 256;
    const int64_t cap = (int64_t)kNumSMs * (ctas_per_sm > 0 ? ctas_per_sm : loss_ctas_per_sm());
    if (blocks > cap) blocks = cap;
    return (int)(blocks < 1 ? 1 : blocks);
}

static bool loss_mt_one_launch() {   // A/B knob: HPFG_LOSS_MT_ONE=0 keeps the reduce + gradient launches for Mean-Teacher
    static bool v = [] {
        const char *e = getenv("HPFG_LOSS_MT_ONE");
        return !(e && atoi(e) == 0);
    }();
    return v;
}

// co-resident CTA capacity of the one-launch kernel on the current device (its grid barrier needs every CTA resident)
template <int C>
static int loss_mt_one_capacity() {
    static int cap = [] {
        int dev = 0, sms = 0, per_sm = 0;
        if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess ||
            cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, loss_mt_one_kernel<C>, 256, 0) != cudaSuccess)
            return 0;
        if (per_sm > 3) per_sm = 3;
        return sms * per_sm;
    }();
    return cap;
}

template <int C>
static int launch_loss(const LossArgs &A, cudaStream_t st) {
    if (A.mode == HPFG_LOSS_MT && A.world == 1 && A.n_l > 0 && A.n_u > 0 && loss_mt_one_launch()) {
        const int cap = loss_mt_one_capacity<C>();
        if (cap > 0) {
            int64_t blocks = ((int64_t)A.n_u * (A.hw >> 2) + 255) / 256;     // at most one unlabeled quad per thread ...
            if (blocks > cap) blocks = cap;                                   // ... and never more CTAs than are resident at once
            HPFG_CUDA_CHECK(launch_pdl(loss_mt_one_kernel<C>, (int)blocks, 256, 0, st, A));
            HPFG_LAUNCH_CHECK();
            return HPFG_OK;
        }
    }
    const int grid = loss_grid((int64_t)(A.n_l + A.n_u) * (A.hw >> 2));
    const int rgrid = loss_grid((int64_t)A.reduce_imgs * (A.hw >> 2));
    switch (A.mode) {
        case HPFG_LOSS_SUP:      // SUP / MT / ICT: only the labeled images carry batch-wide sums (Dice, CE)
        case HPFG_LOSS_MT:
        case HPFG_LOSS_ICT: HPFG_CUDA_CHECK(launch_pdl(loss_reduce_kernel<C, HPFG_LOSS_SUP>, rgrid, 256, 0, st, A)); break;
        case HPFG_LOSS_CPS: HPFG_CUDA_CHECK(launch_pdl(loss_reduce_kernel<C, HPFG_LOSS_CPS>, rgrid, 256, 0, st, A)); break;
        case HPFG_LOSS_S4CV: HPFG_CUDA_CHECK(launch_pdl(loss_reduce_kernel<C, HPFG_LOSS_S4CV>, rgrid, 256, 0, st, A)); break;
        default: HPFG_CUDA_CHECK(launch_pdl(loss_reduce_kernel<C, HPFG_LOSS_UAMT>, rgrid, 256, 0, st, A)); break;
    }
    HPFG_LAUNCH_CHECK();
    // exact-global mode: Dice / CE / pseudo-label / mask sums over the batch of ALL ranks before any coefficient is formed
    // (the last slot is the gradient kernel's block counter: still zero everywhere, so it may take part)
    const bool mt = A.mode == HPFG_LOSS_MT;
    auto grad = mt ? loss_grad_kernel<C, HPFG_LOSS_MT> : loss_grad_kernel<C, -1>;
    const int ggrid = mt ? loss_grid((int64_t)(A.n_l + A.n_u) * (A.hw >> 2), loss_mt_ctas_per_sm()) : grid;
    if (A.world > 1) {
        HPFG_RETURN_IF(sync_allreduce(A.acc, kAccTotal, true, st));
        HPFG_CUDA_CHECK(launch_plain(grad, ggrid, 256, 0, st, A));     // (no programmatic launch across the collective)
    } else {
        HPFG_CUDA_CHECK(launch_pdl(grad, ggrid, 256, 0, st, A));
    }
    HPFG_LAUNCH_CHECK();
    return HPFG_OK;
}

template <int C>
static int launch_dice(const DiceArgs &A, cudaStream_t st) {
    const int grid = loss_grid((int64_t)A.n * (A.hw >> 2));
    HPFG_CUDA_CHECK(launch_pdl(dice_reduce_kernel<C>, grid, 256, 0, st, A));
    HPFG_LAUNCH_CHECK();
    HPFG_CUDA_CHECK(launch_pdl(dice_grad_kernel<C>, A.dinputs ? grid : 1, 256, 0, st, A));
    HPFG_LAUNCH_CHECK();
    return HPFG_OK;
}

}  // namespace hpfg

using namespace hpfg;

extern "C" int64_t hpfg_ssl_loss_workspace_bytes(int mode, int n_l, int n_u, int num_classes, int height,
                                                 int width) {
    (void)n_l; (void)num_classes;
    int64_t aux = 0;
    if (mode == HPFG_LOSS_CPS || mode == HPFG_LOSS_S4CV) aux = 2LL * n_u * height * width;
    if (mode == HPFG_LOSS_UAMT) aux = 1LL * n_u * height * width;
    return kAccTotal * (int64_t)sizeof(double) + ((aux + 255) / 256) * 256;
}

static int ssl_loss_impl(int mode, const float *student, const float *other, const float *mc_logits,
                         int mc_passes, const int64_t *labels, int n_l, int n_u, int num_classes, int height,
                         int width, float cons_weight, const float *cons_weight_dev, float uamt_threshold,
                         const float *class_weights_host, float ce_coef, float dice_coef, float *dstudent, float *dother,
                         float *scalars_out, int64_t *pseudo1, int64_t *pseudo2, void *workspace, void *stream,
                         const float *mix = nullptr, float cons_weight2 = 0.f, const float *cons_weight2_dev = nullptr,
                         const float *uamt_threshold_dev = nullptr) {
    HPFG_REQUIRE(mode >= HPFG_LOSS_SUP && mode <= HPFG_LOSS_S4CV, "hpfg_ssl_loss: unknown mode");
    HPFG_REQUIRE(student && dstudent && scalars_out && workspace, "hpfg_ssl_loss: null buffer");
    HPFG_REQUIRE(n_l >= 0 && n_u >= 0 && n_l + n_u > 0, "hpfg_ssl_loss: empty batch");
    HPFG_REQUIRE(n_l == 0 || labels, "hpfg_ssl_loss: labels required");
    HPFG_REQUIRE(num_classes >= 2 && num_classes <= kMaxC, "hpfg_ssl_loss: num_classes must be in [2,8]");
    HPFG_REQUIRE(((int64_t)height * width) % 4 == 0, "hpfg_ssl_loss: H*W must be a multiple of 4");
    if (mode != HPFG_LOSS_SUP && n_u > 0) HPFG_REQUIRE(other, "hpfg_ssl_loss: teacher/peer logits required");
    if (mode == HPFG_LOSS_CPS || mode == HPFG_LOSS_S4CV)
        HPFG_REQUIRE(dother && other, "hpfg_ssl_loss: CPS / S4CV need peer logits and dother");
    if (mode == HPFG_LOSS_ICT && n_u > 0) HPFG_REQUIRE(mix, "hpfg_ict_loss: mix_factors required");
    if (mode == HPFG_LOSS_UAMT) HPFG_REQUIRE(mc_logits && mc_passes > 0, "hpfg_ssl_loss: UAMT needs mc_logits");
    cudaStream_t st = (cudaStream_t)stream;
    LossArgs A{};
    HPFG_REQUIRE((int64_t)(n_l + n_u) * height * width / 4 < (1LL << 31), "hpfg_ssl_loss: batch too large for 32-bit quad indexing");
    A.mode = mode; A.n_l = n_l; A.n_u = n_u; A.hw = height * width; A.mc_passes = mc_passes;
    A.world = g_loss_global_sums ? sync_world() : 1;
    A.qdiv = make_fastdiv((uint32_t)(A.hw >> 2));
    A.reduce_imgs = (mode == HPFG_LOSS_SUP || mode == HPFG_LOSS_MT || mode == HPFG_LOSS_ICT) ? n_l : n_l + n_u;
    A.student = student; A.other = other; A.mc = mc_logits; A.labels = labels;
    A.mix = mix; A.cons_weight2 = cons_weight2; A.cons_weight2_dev = cons_weight2_dev;
    A.uamt_threshold_dev = uamt_threshold_dev;
    A.cons_weight = cons_weight; A.cons_weight_dev = cons_weight_dev; A.uamt_threshold = uamt_threshold; A.ce_coef = ce_coef; A.dice_coef = dice_coef;
    for (int c = 0; c < kMaxC; ++c) A.class_w[c] = (class_weights_host && c < num_classes) ? class_weights_host[c] : 1.f;
    A.dstudent = dstudent; A.dother = dother; A.scalars = scalars_out; A.pseudo1 = pseudo1; A.pseudo2 = pseudo2;
    A.acc = reinterpret_cast<double *>(workspace);
    A.aux = reinterpret_cast<uint8_t *>(workspace) + kAccTotal * sizeof(double);
    ProfScope _prof(PROF_LOSS, st);
    HPFG_CUDA_CHECK(cudaMemsetAsync(A.acc, 0, kAccTotal * sizeof(double), st));
    switch (num_classes) {
        case 2: return launch_loss<2>(A, st);
        case 3: return launch_loss<3>(A, st);
        case 4: return launch_loss<4>(A, st);
        case 5: return launch_loss<5>(A, st);
        case 6: return launch_loss<6>(A, st);
        case 7: return launch_loss<7>(A, st);
        default: return launch_loss<8>(A, st);
    }
}

extern "C" int hpfg_ssl_loss(int mode, const float *student, const float *other, const float *mc_logits,
                             int mc_passes, const int64_t *labels, int n_l, int n_u, int num_classes, int height,
                             int width, float cons_weight, float uamt_threshold, const float *class_weights_host,
                             float ce_coef, float dice_coef, float *dstudent, float *dother, float *scalars_out,
                             int64_t *pseudo1, int64_t *pseudo2, void *workspace, void *stream) {
    HPFG_REQUIRE(mode <= HPFG_LOSS_UAMT, "hpfg_ssl_loss: use hpfg_ict_loss / hpfg_s4cv_loss for the ICT / S4CV modes");
    return ssl_loss_impl(mode, student, other, mc_logits, mc_passes, labels, n_l, n_u, num_classes, height, width, cons_weight, nullptr,
                         uamt_threshold, class_weights_host, ce_coef, dice_coef, dstudent, dother, scalars_out, pseudo1, pseudo2,
                         workspace, stream);
}

extern "C" int hpfg_ssl_loss_dv(int mode, const float *student, const float *other, const float *mc_logits,
                                int mc_passes, const int64_t *labels, int n_l, int n_u, int num_classes, int height,
                                int width, const float *cons_weight_dev, float uamt_threshold,
                                const float *uamt_threshold_dev, const float *class_weights_host, float ce_coef,
                                float dice_coef, float *dstudent, float *dother, float *scalars_out, int64_t *pseudo1,
                                int64_t *pseudo2, void *workspace, void *stream) {
    HPFG_REQUIRE(cons_weight_dev, "hpfg_ssl_loss_dv: cons_weight_dev is null");
    HPFG_REQUIRE(mode <= HPFG_LOSS_UAMT, "hpfg_ssl_loss_dv: use hpfg_ict_loss / hpfg_s4cv_loss for the ICT / S4CV modes");
    return ssl_loss_impl(mode, student, other, mc_logits, mc_passes, labels, n_l, n_u, num_classes, height, width, 0.f, cons_weight_dev,
                         uamt_threshold, class_weights_host, ce_coef, dice_coef, dstudent, dother, scalars_out, pseudo1, pseudo2,
                         workspace, stream, nullptr, 0.f, nullptr, uamt_threshold_dev);
}

extern "C" int hpfg_dice_loss(const float *inputs, const int64_t *target, int n, int num_classes, int height,
                              int width, int softmax, const float *class_weights_host, float *dinputs,
                              float *scalars_out, void *workspace, void *stream) {
    HPFG_REQUIRE(inputs && target && scalars_out && workspace, "hpfg_dice_loss: null buffer");
    HPFG_REQUIRE(n > 0, "hpfg_dice_loss: empty batch");
    HPFG_REQUIRE(num_classes >= 2 && num_classes <= kMaxC, "hpfg_dice_loss: num_classes must be in [2,8]");
    HPFG_REQUIRE(((int64_t)height * width) % 4 == 0, "hpfg_dice_loss: H*W must be a multiple of 4");
    cudaStream_t st = (cudaStream_t)stream;
    DiceArgs A{};
    A.inputs = inputs; A.target = target; A.n = n; A.hw = height * width; A.softmax = softmax;
    for (int c = 0; c < kMaxC; ++c) A.class_w[c] = (class_weights_host && c < num_classes) ? class_weights_host[c] : 1.f;
    A.dinputs = dinputs; A.scalars = scalars_out; A.acc = reinterpret_cast<double *>(workspace);
    HPFG_CUDA_CHECK(cudaMemsetAsync(A.acc, 0, kAccTotal * sizeof(double), st));
    switch (num_classes) {
        case 2: return launch_dice<2>(A, st);
        case 3: return launch_dice<3>(A, st);
        case 4: return launch_dice<4>(A, st);
        case 5: return launch_dice<5>(A, st);
        case 6: return launch_dice<6>(A, st);
        case 7: return launch_dice<7>(A, st);
        default: return launch_dice<8>(A, st);
    }
}

// ---- ICT-MedSeg (2022_02_ISBI_ICT-MedSeg_ACDC.py:111-137) ---------------------------------------------------------
extern "C" int hpfg_ict_loss(const float *student, const float *teacher_u, const float *mix_factors,
                             const int64_t *labels, int n_l, int n_mixed, int num_classes, int height, int width,
                             float cons_weight, const float *cons_weight_dev, const float *class_weights_host,
                             float ce_coef, float dice_coef, float *dstudent, float *scalars_out, void *workspace,
                             void *stream) {
    return ssl_loss_impl(HPFG_LOSS_ICT, student, teacher_u, nullptr, 0, labels, n_l, n_mixed, num_classes, height, width,
                         cons_weight, cons_weight_dev, 0.f, class_weights_host, ce_coef, dice_coef, dstudent, nullptr,
                         scalars_out, nullptr, nullptr, workspace, stream, mix_factors);
}

// ---- S4CVNet (2022_08_CVPR_S4CVNet_ACDC.py:124-156) ----------------------------------------------------------------
extern "C" int hpfg_s4cv_loss(const float *logits1, const float *logits2, const float *teacher_u,
                              const int64_t *labels, int n_l, int n_u, int num_classes, int height, int width,
                              float cps_weight, float mt_weight, const float *weights_dev,
                              const float *class_weights_host, float ce_coef, float dice_coef, float *dlogits1,
                              float *dlogits2, float *scalars_out, int64_t *pseudo1, int64_t *pseudo2, void *workspace,
                              void *stream) {
    return ssl_loss_impl(HPFG_LOSS_S4CV, logits1, logits2, teacher_u, 0, labels, n_l, n_u, num_classes, height, width,
                         cps_weight, weights_dev, 0.f, class_weights_host, ce_coef, dice_coef, dlogits1, dlogits2,
                         scalars_out, pseudo1, pseudo2, workspace, stream, nullptr, mt_weight,
                         weights_dev ? weights_dev + 1 : nullptr);
}

namespace hpfg {
// out[u] = a[u]*(1-lambda_u) + b[u]*lambda_u over whole images (the ICT input mix, 2022_02...:115-117); 128-bit accesses.
__global__ void __launch_bounds__(256) ict_mix_kernel(const float4 *__restrict__ a, const float4 *__restrict__ b,
                                                      const float *__restrict__ lam, float4 *__restrict__ out,
                                                      int64_t quads_per_image, int64_t total_quads) {
    pdl_prologue();
    for (int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; q < total_quads; q += (int64_t)gridDim.x * blockDim.x) {
        const float l = __ldg(lam + q / quads_per_image), o = __fsub_rn(1.0f, l);
        const float4 x = __ldg(a + q), y = __ldg(b + q);
        // separate roundings (no FMA contraction): bit-identical to torch's a*(1-l) + b*l
        out[q] = make_float4(__fadd_rn(__fmul_rn(x.x, o), __fmul_rn(y.x, l)), __fadd_rn(__fmul_rn(x.y, o), __fmul_rn(y.y, l)),
                             __fadd_rn(__fmul_rn(x.z, o), __fmul_rn(y.z, l)), __fadd_rn(__fmul_rn(x.w, o), __fmul_rn(y.w, l)));
    }
}

// argmax over the class planes of NCHW fp32 logits, first maximum wins (torch.argmax; softmax is monotone, so
// argmax(softmax(z)) == argmax(z) up to fp32 ties, which are resolved on the softmax values exactly as the reference
// does: val.py:268-281 takes argmax(softmax(net(x)))).  4 pixels per thread, 128-bit loads per class plane.
template <int C>
__global__ void __launch_bounds__(256) argmax_kernel(const float *__restrict__ logits, int64_t hw, int64_t total_quads,
                                                     int64_t *__restrict__ out_i64, uint8_t *__restrict__ out_u8) {
    pdl_prologue();
    const int64_t q_per_img = hw >> 2;
    for (int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; q < total_quads; q += (int64_t)gridDim.x * blockDim.x) {
        const int64_t img = q / q_per_img, pix = (q - img * q_per_img) << 2;
        float z[C][4], p[C][4], lse[4];
        load4<C>(logits + (img * C) * hw + pix, hw, z);
        softmax4<C>(z, p, lse);
        int best[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) best[j] = argmax_first<C>(p, j);
        const int64_t o = img * hw + pix;
        if (out_i64) {
            *reinterpret_cast<longlong2 *>(out_i64 + o) = make_longlong2(best[0], best[1]);
            *reinterpret_cast<longlong2 *>(out_i64 + o + 2) = make_longlong2(best[2], best[3]);
        }
        if (out_u8) *reinterpret_cast<uchar4 *>(out_u8 + o) = make_uchar4(best[0], best[1], best[2], best[3]);
    }
}

template <int C>
static int launch_argmax(const float *logits, int64_t hw, int64_t quads, int64_t *o64, uint8_t *o8, cudaStream_t st) {
    HPFG_CUDA_CHECK(launch_pdl(argmax_kernel<C>, loss_grid(quads, 6), 256, 0, st, logits, hw, quads, o64, o8));
    HPFG_LAUNCH_CHECK();
    return HPFG_OK;
}

// softmax_mse_loss (utils/loss/diceloss.py:64-81): the UNREDUCED (softmax(a) - softmax(b))^2 map (or sigmoid), and its
// backward wrt a for an arbitrary upstream gradient: da_k = p_k * (u_k - sum_j u_j p_j), u_j = 2 gout_j (p_j - q_j).
// BWD = false: out = the map; BWD = true: out = da (gout read).  4 pixels per thread, 128-bit accesses per class plane.
template <int C, bool BWD, bool SIGMOID>
__global__ void __launch_bounds__(256) softmax_mse_kernel(const float *__restrict__ a, const float *__restrict__ b,
                                                          const float *__restrict__ gout, float *__restrict__ out, int64_t hw,
                                                          int64_t total_quads) {
    pdl_prologue();
    const int64_t q_per_img = hw >> 2;
    for (int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; q < total_quads; q += (int64_t)gridDim.x * blockDim.x) {
        const int64_t img = q / q_per_img, pix = (q - img * q_per_img) << 2;
        const int64_t o = (img * C) * hw + pix;
        float za[C][4], zb[C][4], pa[C][4], pb[C][4], g[C][4], l1[4], l2[4];
        load4<C>(a + o, hw, za);
        load4<C>(b + o, hw, zb);
        if (BWD) load4<C>(gout + o, hw, g);
        if (SIGMOID) {
#pragma unroll
            for (int c = 0; c < C; ++c)
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    pa[c][j] = 1.f / (1.f + expf(-za[c][j]));
                    pb[c][j] = 1.f / (1.f + expf(-zb[c][j]));
                }
        } else {
            softmax4<C>(za, pa, l1);
            softmax4<C>(zb, pb, l2);
        }
        float r[C][4];
        if (!BWD) {
#pragma unroll
            for (int c = 0; c < C; ++c)
#pragma unroll
                for (int j = 0; j < 4; ++j) { const float d = pa[c][j] - pb[c][j]; r[c][j] = d * d; }
        } else {
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                float u[C], dot = 0.f;
#pragma unroll
                for (int c = 0; c < C; ++c) { u[c] = 2.f * g[c][j] * (pa[c][j] - pb[c][j]); dot = fmaf(u[c], pa[c][j], dot); }
#pragma unroll
                for (int c = 0; c < C; ++c) r[c][j] = SIGMOID ? u[c] * pa[c][j] * (1.f - pa[c][j]) : pa[c][j] * (u[c] - dot);
            }
        }
        store4<C>(out + o, hw, r);
    }
}

template <int C>
static int launch_softmax_mse(const float *a, const float *b, const float *gout, float *out, int64_t hw, int64_t quads, bool sigmoid,
                              cudaStream_t st) {
    const int grid = loss_grid(quads, 6);
    if (gout) {
        if (sigmoid) HPFG_CUDA_CHECK(launch_pdl(softmax_mse_kernel<C, true, true>, grid, 256, 0, st, a, b, gout, out, hw, quads));
        else HPFG_CUDA_CHECK(launch_pdl(softmax_mse_kernel<C, true, false>, grid, 256, 0, st, a, b, gout, out, hw, quads));
    } else {
        if (sigmoid) HPFG_CUDA_CHECK(launch_pdl(softmax_mse_kernel<C, false, true>, grid, 256, 0, st, a, b, gout, out, hw, quads));
        else HPFG_CUDA_CHECK(launch_pdl(softmax_mse_kernel<C, false, false>, grid, 256, 0, st, a, b, gout, out, hw, quads));
    }
    HPFG_LAUNCH_CHECK();
    return HPFG_OK;
}
}  // namespace hpfg

extern "C" int hpfg_ict_mix(const float *a, const float *b, const float *mix_factors, int n, int64_t per_image,
                            float *out, void *stream) {
    HPFG_REQUIRE(a && b && mix_factors && out, "hpfg_ict_mix: null buffer");
    HPFG_REQUIRE(n > 0 && per_image > 0 && per_image % 4 == 0, "hpfg_ict_mix: per_image must be a positive multiple of 4");
    cudaStream_t st = (cudaStream_t)stream;
    const int64_t qpi = per_image / 4, total = qpi * n;
    ProfScope _prof(PROF_LOSS, st);
    HPFG_CUDA_CHECK(launch_pdl(ict_mix_kernel, loss_grid(total, 6), 256, 0, st, reinterpret_cast<const float4 *>(a),
                               reinterpret_cast<const float4 *>(b), mix_factors, reinterpret_cast<float4 *>(out), qpi, total));
    HPFG_LAUNCH_CHECK();
    return HPFG_OK;
}

extern "C" int hpfg_argmax_labels(const float *logits, int n, int num_classes, int height, int width,
                                  int64_t *labels_i64, uint8_t *labels_u8, void *stream) {
    HPFG_REQUIRE(logits && (labels_i64 || labels_u8), "hpfg_argmax_labels: null buffer");
    HPFG_REQUIRE(n > 0, "hpfg_argmax_labels: empty batch");
    HPFG_REQUIRE(num_classes >= 2 && num_classes <= kMaxC, "hpfg_argmax_labels: num_classes must be in [2,8]");
    const int64_t hw = (int64_t)height * width;
    HPFG_REQUIRE(hw % 4 == 0, "hpfg_argmax_labels: H*W must be a multiple of 4");
    cudaStream_t st = (cudaStream_t)stream;
    const int64_t quads = (hw >> 2) * n;
    ProfScope _prof(PROF_LOSS, st);
    switch (num_classes) {
        case 2: return launch_argmax<2>(logits, hw, quads, labels_i64, labels_u8, st);
        case 3: return launch_argmax<3>(logits, hw, quads, labels_i64, labels_u8, st);
        case 4: return launch_argmax<4>(logits, hw, quads, labels_i64, labels_u8, st);
        case 5: return launch_argmax<5>(logits, hw, quads, labels_i64, labels_u8, st);
        case 6: return launch_argmax<6>(logits, hw, quads, labels_i64, labels_u8, st);
        case 7: return launch_argmax<7>(logits, hw, quads, labels_i64, labels_u8, st);
        default: return launch_argmax<8>(logits, hw, quads, labels_i64, labels_u8, st);
    }
}

extern "C" int hpfg_softmax_mse(const float *input_logits, const float *target_logits, const float *grad_out, int n,
                                int num_classes, int height, int width, int sigmoid, float *out, void *stream) {
    HPFG_REQUIRE(input_logits && target_logits && out, "hpfg_softmax_mse: null buffer");
    HPFG_REQUIRE(n > 0, "hpfg_softmax_mse: empty batch");
    HPFG_REQUIRE(num_classes >= 1 && num_classes <= kMaxC, "hpfg_softmax_mse: num_classes must be in [1,8]");
    const int64_t hw = (int64_t)height * width;
    HPFG_REQUIRE(hw % 4 == 0, "hpfg_softmax_mse: H*W must be a multiple of 4");
    cudaStream_t st = (cudaStream_t)stream;
    const int64_t quads = (hw >> 2) * n;
    ProfScope _prof(PROF_LOSS, st);
    switch (num_classes) {
        case 1: return launch_softmax_mse<1>(input_logits, target_logits, grad_out, out, hw, quads, sigmoid != 0, st);
        case 2: return launch_softmax_mse<2>(input_logits, target_logits, grad_out, out, hw, quads, sigmoid != 0, st);
        case 3: return launch_softmax_mse<3>(input_logits, target_logits, grad_out, out, hw, quads, sigmoid != 0, st);
        case 4: return launch_softmax_mse<4>(input_logits, target_logits, grad_out, out, hw, quads, sigmoid != 0, st);
        case 5: return launch_softmax_mse<5>(input_logits, target_logits, grad_out, out, hw, quads, sigmoid != 0, st);
        case 6: return launch_softmax_mse<6>(input_logits, target_logits, grad_out, out, hw, quads, sigmoid != 0, st);
        case 7: return launch_softmax_mse<7>(input_logits, target_logits, grad_out, out, hw, quads, sigmoid != 0, st);
        default: return launch_softmax_mse<8>(input_logits, target_logits, grad_out, out, hw, quads, sigmoid != 0, st);
    }
}
