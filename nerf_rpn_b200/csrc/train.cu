// Training-step kernels around the three tcgen05 GEMMs (fprop, dgrad = fprop on mirrored weights, wgrad): everything of
// `loss.backward(); optimizer.step()` for the anchor RPN (SURVEY.md 8(a) a18, config 4) that is not a convolution.
//   BatchNorm3d in TRAIN mode  (feature_extractor.py:38-43,48-68 under model.train()): batch statistics, normalise (+ residual)
//                               (+ ReLU), running-stat update; backward = two per-channel reductions + one pointwise pass
//   F.max_pool3d(3,2,1)         forward with recorded argmax, backward as a deterministic gather (feature_extractor.py:219)
//   F.interpolate(nearest)+add  backward of the FPN top-down merge (feature_extractor.py:211-213)
//   stride-2 1^3 convolutions   sub-sample (forward operand of wgrad) / zero-stuff (dgrad) helpers
//   RPN losses                  BCE-with-logits + smooth-L1(beta 1/9) on the sampled anchors and their gradient w.r.t. the
//                               predictor output (rpn.py:372-417), box encoders (AABB_coder.py:14-56, midpoint_offset_coder.py:106-158)
//   optimiser                   weight packing fp32 -> 16-bit GEMM layouts, global gradient norm, fused clip + AdamW
//                               (run_rpn.py:345,390-395: AdamW, clip_grad_norm_)
// All bandwidth bound: one read (+ one write) of their tensors, 16-byte accesses, reductions in a fixed order (bit-reproducible).
#include <cstring>
#include "common.cuh"

namespace nrpn {

constexpr int kRedBlocks = 296;          // 2 per SM: partial sums of the per-channel reductions (592 measured slower: the three-operand backward pass loses more than the forward gains)

static inline unsigned grid1d(size_t total, int threads, int per_sm = 16) {
    size_t b = ceil_div(total, (size_t)threads);
    const size_t cap = (size_t)num_sms() * per_sm;
    return (unsigned)(b < cap ? (b ? b : 1) : cap);
}

// ---------------------------------------------------------------------------------------------- per-channel reductions
// MODE 0: s1 = sum y, s2 = sum y^2                       (batch statistics)
// MODE 1: g = dout * (out > 0 | 1); s1 = sum g, s2 = sum g * xhat,  xhat = (y - mean) * rstd     (BatchNorm backward)
// Thread (r, cg): channel group cg (8 channels) of rows r, r + R, ...; block partials in shared memory, then one fp32 pair per
// (block, channel) to global; the final kernel adds the block partials in fp64 in block order.
template <int MODE>
__global__ void __launch_bounds__(256) chan_reduce_kernel(const __nv_bfloat16* __restrict__ a, const __nv_bfloat16* __restrict__ act,
                                                          const __nv_bfloat16* __restrict__ y, long rows, int c, const float* __restrict__ stats,
                                                          int relu, int fp16, float* __restrict__ partial) {
    extern __shared__ float sm[];                       // [2][lanes][c] would be too big: reduce through warp-strided adds instead
    const int cgs = c >> 3;                             // channel groups
    const int lanes = 256 / cgs > 0 ? 256 / cgs : 1;    // rows processed per pass (cgs <= 256)
    const int cg = threadIdx.x % cgs, lane = threadIdx.x / cgs;
    float s1[8], s2[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) { s1[k] = 0.f; s2[k] = 0.f; }
    float mean[8], rstd[8];
    if (MODE == 1) {
#pragma unroll
        for (int k = 0; k < 8; ++k) { mean[k] = stats[cg * 8 + k]; rstd[k] = stats[c + cg * 8 + k]; }
    }
    if (lane < lanes) {
        const long per = ceil_div(rows, (long)gridDim.x);
        const long r0 = (long)blockIdx.x * per, r1 = min(rows, r0 + per);
#pragma unroll 4
        for (long r = r0 + lane; r < r1; r += lanes) {       // unrolled: four rows' loads in flight per thread
            const size_t off = (size_t)r * c + cg * 8;
            const uint4 av = __ldg(reinterpret_cast<const uint4*>(a + off));
            const uint32_t* aw = reinterpret_cast<const uint32_t*>(&av);
            if (MODE == 0) {
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    const float2 f = unpack_act2(aw[k], fp16);
                    s1[2 * k] += f.x; s2[2 * k] += f.x * f.x; s1[2 * k + 1] += f.y; s2[2 * k + 1] += f.y * f.y;
                }
            } else {
                const uint4 yv = __ldg(reinterpret_cast<const uint4*>(y + off));
                const uint32_t* yw = reinterpret_cast<const uint32_t*>(&yv);
                uint4 ov = make_uint4(0, 0, 0, 0);
                if (relu) ov = __ldg(reinterpret_cast<const uint4*>(act + off));
                const uint32_t* ow = reinterpret_cast<const uint32_t*>(&ov);
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    float2 g = unpack_act2(aw[k], fp16);
                    const float2 yy = unpack_act2(yw[k], fp16);
                    if (relu) { const float2 o = unpack_act2(ow[k], fp16); if (!(o.x > 0.f)) g.x = 0.f; if (!(o.y > 0.f)) g.y = 0.f; }
                    s1[2 * k] += g.x; s2[2 * k] += g.x * ((yy.x - mean[2 * k]) * rstd[2 * k]);
                    s1[2 * k + 1] += g.y; s2[2 * k + 1] += g.y * ((yy.y - mean[2 * k + 1]) * rstd[2 * k + 1]);
                }
            }
        }
    }
    // block reduction over `lanes` in a fixed order: lane l adds into shared memory in turn
    float* b1 = sm; float* b2 = sm + c;
    for (int i = threadIdx.x; i < 2 * c; i += blockDim.x) sm[i] = 0.f;
    __syncthreads();
    for (int l = 0; l < lanes; ++l) {
        if (lane == l) {
#pragma unroll
            for (int k = 0; k < 8; ++k) { b1[cg * 8 + k] += s1[k]; b2[cg * 8 + k] += s2[k]; }
        }
        __syncthreads();
    }
    for (int i = threadIdx.x; i < c; i += blockDim.x) {
        partial[((size_t)blockIdx.x * 2) * c + i] = b1[i];
        partial[((size_t)blockIdx.x * 2 + 1) * c + i] = b2[i];
    }
}

// MODE 0: stats = {mean[c], rstd[c], var_biased[c]}; optional running-stat update (momentum, unbiased variance) like nn.BatchNorm3d.
// MODE 1: sums = {sum g*xhat [c] (= dgamma), sum g [c] (= dbeta)}
template <int MODE>
__global__ void chan_reduce_final_kernel(const float* __restrict__ partial, int blocks, int c, long rows, float eps, float* __restrict__ out,
                                         float* __restrict__ running_mean, float* __restrict__ running_var, float momentum) {
    // 8 channels per CTA, 32 threads per channel: thread (kl, ch) sums the partials of blocks kl, kl + 32, ...; the 32 sums are added in a fixed
    // order (bit-reproducible).  (One thread per channel walked all 296 partials alone: 46 us per call, 106 calls per training step.)
    __shared__ double red[2][32][8];
    const int cl = threadIdx.x & 7, kl = threadIdx.x >> 3;
    const int ch = blockIdx.x * 8 + cl;
    double a = 0.0, b = 0.0;
    if (ch < c) {
#pragma unroll 5
        for (int k = kl; k < blocks; k += 32) { a += (double)partial[((size_t)k * 2) * c + ch]; b += (double)partial[((size_t)k * 2 + 1) * c + ch]; }
    }
    red[0][kl][cl] = a; red[1][kl][cl] = b;
    __syncthreads();
    if (kl != 0 || ch >= c) return;
    a = 0.0; b = 0.0;
#pragma unroll
    for (int k = 0; k < 32; ++k) { a += red[0][k][cl]; b += red[1][k][cl]; }
    if (MODE == 0) {
        const double mean = a / (double)rows;
        double var = b / (double)rows - mean * mean;
        if (var < 0.0) var = 0.0;
        out[ch] = (float)mean;
        out[c + ch] = (float)(1.0 / sqrt(var + (double)eps));
        out[2 * c + ch] = (float)var;
        if (running_mean) {
            const double unbiased = rows > 1 ? var * (double)rows / (double)(rows - 1) : var;
            running_mean[ch] = (float)((1.0 - momentum) * (double)running_mean[ch] + momentum * mean);
            running_var[ch] = (float)((1.0 - momentum) * (double)running_var[ch] + momentum * unbiased);
        }
    } else {
        out[ch] = (float)b;            // sum g * xhat = dgamma  (first, so that {dgamma, dbeta} lines up with [bn.weight.grad | bn.bias.grad])
        out[c + ch] = (float)a;        // sum g         = dbeta
    }
}

// out = act(gamma * (y - mean) * rstd + beta (+ res))
// When the number of 8-channel groups divides the block size (every power-of-two width of the path) a thread sees the SAME eight channels in every
// iteration of its grid-stride loop: the per-channel constants are loaded once (the first version fetched 32 / 40 scalars and ran a 64-bit modulo per
// 16 bytes of data: 1.36 / 1.73 ms per training step against 0.6 / 1.2 ms of HBM time).
__global__ void __launch_bounds__(256) bn_apply_kernel(const __nv_bfloat16* __restrict__ y, const __nv_bfloat16* __restrict__ res,
                                                       __nv_bfloat16* __restrict__ out, size_t chunks, int c, const float* __restrict__ stats,
                                                       const float* __restrict__ gamma, const float* __restrict__ beta, int relu, int fp16) {
    const int cgs = c >> 3;
    const bool fixed = (256 % cgs) == 0;
    float mean[8], rstd[8], gam[8], bet[8];
    auto consts = [&](int c0) {
#pragma unroll
        for (int k = 0; k < 8; ++k) { mean[k] = stats[c0 + k]; rstd[k] = stats[c + c0 + k]; gam[k] = gamma[c0 + k]; bet[k] = beta[c0 + k]; }
    };
    if (fixed) consts((int)(threadIdx.x % cgs) * 8);
#pragma unroll 2
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < chunks; i += (size_t)gridDim.x * blockDim.x) {
        if (!fixed) consts((int)(i % cgs) * 8);
        const uint4 yv = __ldg(reinterpret_cast<const uint4*>(y) + i);
        const uint32_t* yw = reinterpret_cast<const uint32_t*>(&yv);
        uint4 rv = make_uint4(0, 0, 0, 0);
        if (res) rv = __ldg(reinterpret_cast<const uint4*>(res) + i);
        const uint32_t* rw = reinterpret_cast<const uint32_t*>(&rv);
        uint32_t o[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const float2 f = unpack_act2(yw[k], fp16);
            float va = (f.x - mean[2 * k]) * rstd[2 * k] * gam[2 * k] + bet[2 * k];
            float vb = (f.y - mean[2 * k + 1]) * rstd[2 * k + 1] * gam[2 * k + 1] + bet[2 * k + 1];
            if (res) { const float2 r = unpack_act2(rw[k], fp16); va += r.x; vb += r.y; }
            if (relu) { va = fmaxf(va, 0.f); vb = fmaxf(vb, 0.f); }
            o[k] = pack_act2(va, vb, fp16);
        }
        reinterpret_cast<uint4*>(out)[i] = make_uint4(o[0], o[1], o[2], o[3]);
    }
}

// dy = gamma * rstd * (g - s1/M - xhat * s2/M),  g = dout * (out > 0 | 1);  dres = g (gradient of the skip connection)
__global__ void __launch_bounds__(256) bn_backward_apply_kernel(const __nv_bfloat16* __restrict__ dout, const __nv_bfloat16* __restrict__ act,
                                                                const __nv_bfloat16* __restrict__ y, __nv_bfloat16* __restrict__ dy,
                                                                __nv_bfloat16* __restrict__ dres, size_t chunks, int c, long rows,
                                                                const float* __restrict__ stats, const float* __restrict__ gamma,
                                                                const float* __restrict__ sums, int relu, int fp16) {
    const int cgs = c >> 3;
    const float inv_m = 1.0f / (float)rows;
    const bool fixed = (256 % cgs) == 0;
    float mean[8], rstd[8], gam[8], s1[8], s2[8];              // s1 = sum(g xhat) / M (dgamma / M), s2 = sum(g) / M (dbeta / M)
    auto consts = [&](int c0) {
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            mean[k] = stats[c0 + k]; rstd[k] = stats[c + c0 + k]; gam[k] = gamma[c0 + k];
            s1[k] = sums[c0 + k] * inv_m; s2[k] = sums[c + c0 + k] * inv_m;
        }
    };
    if (fixed) consts((int)(threadIdx.x % cgs) * 8);
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < chunks; i += (size_t)gridDim.x * blockDim.x) {
        if (!fixed) consts((int)(i % cgs) * 8);
        const uint4 gv = __ldg(reinterpret_cast<const uint4*>(dout) + i);
        const uint4 yv = __ldg(reinterpret_cast<const uint4*>(y) + i);
        uint4 ov = make_uint4(0, 0, 0, 0);
        if (relu) ov = __ldg(reinterpret_cast<const uint4*>(act) + i);
        const uint32_t* gw = reinterpret_cast<const uint32_t*>(&gv);
        const uint32_t* yw = reinterpret_cast<const uint32_t*>(&yv);
        const uint32_t* ow = reinterpret_cast<const uint32_t*>(&ov);
        uint32_t o[4], gm[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            float2 g = unpack_act2(gw[k], fp16);
            const float2 yy = unpack_act2(yw[k], fp16);
            if (relu) { const float2 a = unpack_act2(ow[k], fp16); if (!(a.x > 0.f)) g.x = 0.f; if (!(a.y > 0.f)) g.y = 0.f; }
            const int ka = 2 * k, kb = ka + 1;
            const float xa = (yy.x - mean[ka]) * rstd[ka], xb = (yy.y - mean[kb]) * rstd[kb];
            const float da = gam[ka] * rstd[ka] * (g.x - s2[ka] - xa * s1[ka]);
            const float db = gam[kb] * rstd[kb] * (g.y - s2[kb] - xb * s1[kb]);
            o[k] = pack_act2(da, db, fp16);
            gm[k] = pack_act2(g.x, g.y, fp16);
        }
        reinterpret_cast<uint4*>(dy)[i] = make_uint4(o[0], o[1], o[2], o[3]);
        if (dres) reinterpret_cast<uint4*>(dres)[i] = make_uint4(gm[0], gm[1], gm[2], gm[3]);
    }
}

// ---------------------------------------------------------------------------------------------- max-pool (3,2,1) with argmax
// Forward: out = max over the 3^3 window; idx = window position (dx+1)*9 + (dy+1)*3 + (dz+1) of the FIRST maximum in scan order
// (x outer, z inner; padded taps skipped), or of the LAST NaN, which then is the output -- the element torch's
// max_pool3d_with_indices records (its test is `val > max || isnan(val)`).
__global__ void __launch_bounds__(256) maxpool_k3s2_argmax_kernel(const __nv_bfloat16* __restrict__ in, int n, int X, int Y, int Z, int C, int Xo, int Yo,
                                                                  int Zo, __nv_bfloat16* __restrict__ out, uint8_t* __restrict__ idx, int fp16) {
    const int cg = C >> 3;
    const size_t total = (size_t)n * Xo * Yo * Zo * cg;
    for (size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (size_t)gridDim.x * blockDim.x) {
        const int g = (int)(t % cg); size_t v = t / cg;
        const int k = (int)(v % Zo); v /= Zo;
        const int j = (int)(v % Yo); v /= Yo;
        const int i = (int)(v % Xo); const int b = (int)(v / Xo);
        float m[8]; int am[8];
#pragma unroll
        for (int q = 0; q < 8; ++q) { m[q] = -INFINITY; am[q] = 13; }
        const __nv_bfloat16* base = in + (size_t)b * X * Y * Z * C + g * 8;
        for (int dx = -1; dx <= 1; ++dx) {
            const int x = 2 * i + dx; if (x < 0 || x >= X) continue;
            for (int dy = -1; dy <= 1; ++dy) {
                const int y = 2 * j + dy; if (y < 0 || y >= Y) continue;
                for (int dz = -1; dz <= 1; ++dz) {
                    const int z = 2 * k + dz; if (z < 0 || z >= Z) continue;
                    const uint4 raw = __ldg(reinterpret_cast<const uint4*>(base + (((size_t)x * Y + y) * Z + z) * C));
                    const uint32_t* h = reinterpret_cast<const uint32_t*>(&raw);
                    const int code = (dx + 1) * 9 + (dy + 1) * 3 + (dz + 1);
#pragma unroll
                    for (int q = 0; q < 4; ++q) {
                        const float2 f = unpack_act2(h[q], fp16);
                        if (f.x > m[2 * q] || isnan(f.x)) { m[2 * q] = f.x; am[2 * q] = code; }
                        if (f.y > m[2 * q + 1] || isnan(f.y)) { m[2 * q + 1] = f.y; am[2 * q + 1] = code; }
                    }
                }
            }
        }
        uint32_t o[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) o[q] = pack_act2(m[2 * q], m[2 * q + 1], fp16);
        const size_t off = ((((size_t)b * Xo + i) * Yo + j) * Zo + k) * C + g * 8;
        *reinterpret_cast<uint4*>(out + off) = make_uint4(o[0], o[1], o[2], o[3]);
        *reinterpret_cast<uint2*>(idx + off) = make_uint2((uint32_t)am[0] | ((uint32_t)am[1] << 8) | ((uint32_t)am[2] << 16) | ((uint32_t)am[3] << 24),
                                                          (uint32_t)am[4] | ((uint32_t)am[5] << 8) | ((uint32_t)am[6] << 16) | ((uint32_t)am[7] << 24));
    }
}

// Backward as a gather: input voxel (x,y,z) belongs to the windows of outputs i with |x - 2i| <= 1 (<= 2 per axis); it receives
// dy of every window whose recorded argmax is its own position.  Fixed summation order (i, j, k ascending): deterministic.
__global__ void __launch_bounds__(256) maxpool_k3s2_backward_kernel(const __nv_bfloat16* __restrict__ dy, const uint8_t* __restrict__ idx, int n, int X, int Y,
                                                                    int Z, int C, int Xo, int Yo, int Zo, __nv_bfloat16* __restrict__ dx, int fp16) {
    const int cg = C >> 3;
    const size_t total = (size_t)n * X * Y * Z * cg;
    for (size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (size_t)gridDim.x * blockDim.x) {
        const int g = (int)(t % cg); size_t v = t / cg;
        const int z = (int)(v % Z); v /= Z;
        const int y = (int)(v % Y); v /= Y;
        const int x = (int)(v % X); const int b = (int)(v / X);
        float acc[8];
#pragma unroll
        for (int q = 0; q < 8; ++q) acc[q] = 0.f;
        for (int i = (x > 0 ? (x - 1 + 1) / 2 : 0); i <= (x + 1) / 2 && i < Xo; ++i) {
            const int ddx = x - 2 * i; if (ddx < -1 || ddx > 1) continue;
            for (int j = (y > 0 ? y / 2 : 0); j <= (y + 1) / 2 && j < Yo; ++j) {
                const int ddy = y - 2 * j; if (ddy < -1 || ddy > 1) continue;
                for (int k = (z > 0 ? z / 2 : 0); k <= (z + 1) / 2 && k < Zo; ++k) {
                    const int ddz = z - 2 * k; if (ddz < -1 || ddz > 1) continue;
                    const int code = (ddx + 1) * 9 + (ddy + 1) * 3 + (ddz + 1);
                    const size_t off = ((((size_t)b * Xo + i) * Yo + j) * Zo + k) * C + g * 8;
                    const uint2 iv = __ldg(reinterpret_cast<const uint2*>(idx + off));
                    const uint4 gv = __ldg(reinterpret_cast<const uint4*>(dy + off));
                    const uint32_t* gw = reinterpret_cast<const uint32_t*>(&gv);
#pragma unroll
                    for (int q = 0; q < 4; ++q) {
                        const float2 f = unpack_act2(gw[q], fp16);
                        const uint32_t word = q < 2 ? iv.x : iv.y;
                        const int ia = (word >> (16 * (q & 1))) & 0xFF, ib = (word >> (16 * (q & 1) + 8)) & 0xFF;
                        if (ia == code) acc[2 * q] += f.x;
                        if (ib == code) acc[2 * q + 1] += f.y;
                    }
                }
            }
        }
        uint32_t o[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) o[q] = pack_act2(acc[2 * q], acc[2 * q + 1], fp16);
        *reinterpret_cast<uint4*>(dx + ((((size_t)b * X + x) * Y + y) * Z + z) * C + g * 8) = make_uint4(o[0], o[1], o[2], o[3]);
    }
}

// ---------------------------------------------------------------------------------------------- nearest up-sampling, backward
// Forward (conv epilogue): fine[f] += coarse[min(floor(f * in/out), in-1)].  Backward: dcoarse[cidx] (+)= sum of dfine[f] over the
// fine voxels that map to cidx, evaluated with the SAME float expression as the forward epilogue.
__device__ __forceinline__ int up_src(int g, float rs, int in) { return min((int)floorf((float)g * rs), in - 1); }

__global__ void __launch_bounds__(256) upsample_nearest_backward_kernel(const __nv_bfloat16* __restrict__ dfine, int n, int Xf, int Yf, int Zf, int Xc, int Yc,
                                                                        int Zc, int C, __nv_bfloat16* __restrict__ dcoarse, int accumulate, int fp16) {
    const int cg = C >> 3;
    const float rsx = (float)Xc / (float)Xf, rsy = (float)Yc / (float)Yf, rsz = (float)Zc / (float)Zf;
    const size_t total = (size_t)n * Xc * Yc * Zc * cg;
    for (size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (size_t)gridDim.x * blockDim.x) {
        const int g = (int)(t % cg); size_t v = t / cg;
        const int z = (int)(v % Zc); v /= Zc;
        const int y = (int)(v % Yc); v /= Yc;
        const int x = (int)(v % Xc); const int b = (int)(v / Xc);
        float acc[8];
#pragma unroll
        for (int q = 0; q < 8; ++q) acc[q] = 0.f;
        __nv_bfloat16* dst = dcoarse + ((((size_t)b * Xc + x) * Yc + y) * Zc + z) * C + g * 8;
        if (accumulate) {
            const uint4 cur = *reinterpret_cast<const uint4*>(dst);
            const uint32_t* cw = reinterpret_cast<const uint32_t*>(&cur);
#pragma unroll
            for (int q = 0; q < 4; ++q) { const float2 f = unpack_act2(cw[q], fp16); acc[2 * q] = f.x; acc[2 * q + 1] = f.y; }
        }
        // candidate fine indices: the pre-image of a coarse index under floor(f * in/out) is an interval around x * out/in
        const int fx0 = max(0, (int)((float)x / rsx) - 2), fx1 = min(Xf - 1, (int)((float)(x + 1) / rsx) + 2);
        const int fy0 = max(0, (int)((float)y / rsy) - 2), fy1 = min(Yf - 1, (int)((float)(y + 1) / rsy) + 2);
        const int fz0 = max(0, (int)((float)z / rsz) - 2), fz1 = min(Zf - 1, (int)((float)(z + 1) / rsz) + 2);
        for (int fx = fx0; fx <= fx1; ++fx) {
            if (up_src(fx, rsx, Xc) != x) continue;
            for (int fy = fy0; fy <= fy1; ++fy) {
                if (up_src(fy, rsy, Yc) != y) continue;
                for (int fz = fz0; fz <= fz1; ++fz) {
                    if (up_src(fz, rsz, Zc) != z) continue;
                    const uint4 gv = __ldg(reinterpret_cast<const uint4*>(dfine + ((((size_t)b * Xf + fx) * Yf + fy) * Zf + fz) * C + g * 8));
                    const uint32_t* gw = reinterpret_cast<const uint32_t*>(&gv);
#pragma unroll
                    for (int q = 0; q < 4; ++q) { const float2 f = unpack_act2(gw[q], fp16); acc[2 * q] += f.x; acc[2 * q + 1] += f.y; }
                }
            }
        }
        uint32_t o[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) o[q] = pack_act2(acc[2 * q], acc[2 * q + 1], fp16);
        *reinterpret_cast<uint4*>(dst) = make_uint4(o[0], o[1], o[2], o[3]);
    }
}

// ---------------------------------------------------------------------------------------------- stride-2 helpers (1^3 s2 convs)
// gather: dst[(i,j,k)] = src[(2i,2j,2k)]; scatter: dst[(x,y,z)] = (x,y,z all even) ? src[(x/2,y/2,z/2)] : 0 (full overwrite)
__global__ void __launch_bounds__(256) stride2_kernel(const uint4* __restrict__ src, uint4* __restrict__ dst, int n, int X, int Y, int Z, int Xo, int Yo, int Zo,
                                                      int cg, int scatter) {
    const size_t total = scatter ? (size_t)n * X * Y * Z * cg : (size_t)n * Xo * Yo * Zo * cg;
    for (size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (size_t)gridDim.x * blockDim.x) {
        const int g = (int)(t % cg); size_t v = t / cg;
        if (scatter) {
            const int z = (int)(v % Z); v /= Z;
            const int y = (int)(v % Y); v /= Y;
            const int x = (int)(v % X); const int b = (int)(v / X);
            uint4 val = make_uint4(0, 0, 0, 0);
            if (!((x | y | z) & 1)) val = __ldg(src + ((((size_t)b * Xo + (x >> 1)) * Yo + (y >> 1)) * Zo + (z >> 1)) * cg + g);
            dst[t] = val;
        } else {
            const int k = (int)(v % Zo); v /= Zo;
            const int j = (int)(v % Yo); v /= Yo;
            const int i = (int)(v % Xo); const int b = (int)(v / Xo);
            dst[t] = __ldg(src + ((((size_t)b * X + 2 * i) * Y + 2 * j) * Z + 2 * k) * cg + g);
        }
    }
}

// a (+)= b on 16-bit tensors (gradient accumulation at branch points)
__global__ void __launch_bounds__(256) add_inplace_kernel(__nv_bfloat16* __restrict__ a, const __nv_bfloat16* __restrict__ b, size_t chunks, int fp16) {
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < chunks; i += (size_t)gridDim.x * blockDim.x) {
        uint4 av = reinterpret_cast<const uint4*>(a)[i];
        const uint4 bv = __ldg(reinterpret_cast<const uint4*>(b) + i);
        uint32_t* aw = reinterpret_cast<uint32_t*>(&av);
        const uint32_t* bw = reinterpret_cast<const uint32_t*>(&bv);
#pragma unroll
        for (int k = 0; k < 4; ++k) { const float2 x = unpack_act2(aw[k], fp16), y = unpack_act2(bw[k], fp16); aw[k] = pack_act2(x.x + y.x, x.y + y.y, fp16); }
        reinterpret_cast<uint4*>(a)[i] = av;
    }
}

// ---------------------------------------------------------------------------------------------- RPN losses
struct LossDev {
    int n_levels, A, code, rotated;
    float* pred[NRPN_RPN_MAX_LEVELS];              // fp32 (voxels, 128) rows [A logits | A*code deltas | pad]
    __nv_bfloat16* dpred[NRPN_RPN_MAX_LEVELS];     // 16-bit (voxels, 128), zero-filled by the caller
    int gx[NRPN_RPN_MAX_LEVELS], gy[NRPN_RPN_MAX_LEVELS], gz[NRPN_RPN_MAX_LEVELS];
    int sx[NRPN_RPN_MAX_LEVELS], sy[NRPN_RPN_MAX_LEVELS], sz[NRPN_RPN_MAX_LEVELS];
    long begin[NRPN_RPN_MAX_LEVELS + 1];           // first flat anchor index of each level
    float cell[NRPN_RPN_MAX_LEVELS][16][6];
};

__device__ __forceinline__ void anchor_of(const LossDev& P, long flat, int& l, long& vox, int& a, float* an) {
    l = 0;
#pragma unroll
    for (int i = 1; i < NRPN_RPN_MAX_LEVELS; ++i) if (i < P.n_levels && flat >= P.begin[i]) l = i;
    const long r = flat - P.begin[l];
    a = (int)(r % P.A); vox = r / P.A;
    long v = vox;
    const int z = (int)(v % P.gz[l]); v /= P.gz[l];
    const int y = (int)(v % P.gy[l]); const int x = (int)(v / P.gy[l]);
    const float fx = (float)(x * P.sx[l]), fy = (float)(y * P.sy[l]), fz = (float)(z * P.sz[l]);
    an[0] = fx + P.cell[l][a][0]; an[1] = fy + P.cell[l][a][1]; an[2] = fz + P.cell[l][a][2];
    an[3] = fx + P.cell[l][a][3]; an[4] = fy + P.cell[l][a][4]; an[5] = fz + P.cell[l][a][5];
}

// encode_boxes_3d (AABB_coder.py:14-56): target deltas of gt (x1..z2) w.r.t. anchor
__device__ __forceinline__ void encode_aabb(const float* an, const float* gt, float* t) {
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        const float es = an[3 + k] - an[k], ec = an[k] + 0.5f * es;
        const float gs = gt[3 + k] - gt[k], gc = gt[k] + 0.5f * gs;
        t[k] = (gc - ec) / es;
        t[3 + k] = logf(gs / es);
    }
}

// bbox2delta_sp (midpoint_offset_coder.py:106-158): gt (x,y,z,w,h,d,theta) w.r.t. anchor -> (dx,dy,dz,dw,dh,dd,da,db)
__device__ __forceinline__ void encode_obb(const float* an, const float* gt, float* t) {
    const float px = (an[0] + an[3]) * 0.5f, py = (an[1] + an[4]) * 0.5f, pz = (an[2] + an[5]) * 0.5f;
    const float pw = an[3] - an[0], ph = an[4] - an[1], pd = an[5] - an[2];
    const float x = gt[0], y = gt[1], w = gt[3], h = gt[4], th = gt[6];
    const float co = cosf(th), si = sinf(th);
    const float xb = fabsf(w / 2.f * co) + fabsf(h / 2.f * si), yb = fabsf(w / 2.f * si) + fabsf(h / 2.f * co);      // obb2hbb
    const float gx = ((x - xb) + (x + xb)) * 0.5f, gy = ((y - yb) + (y + yb)) * 0.5f;
    const float gw = (x + xb) - (x - xb), gh = (y + yb) - (y - yb);
    const float v1x = w / 2.f * co, v1y = -w / 2.f * si, v2x = -h / 2.f * si, v2y = -h / 2.f * co;                     // obb2poly
    const float pxs[4] = {x + v1x + v2x, x + v1x - v2x, x - v1x - v2x, x - v1x + v2x};
    const float pys[4] = {y + v1y + v2y, y + v1y - v2y, y - v1y - v2y, y - v1y + v2y};
    float ymin = pys[0], xmax = pxs[0];
#pragma unroll
    for (int k = 1; k < 4; ++k) { ymin = fminf(ymin, pys[k]); xmax = fmaxf(xmax, pxs[k]); }
    float ga = -INFINITY, gb = -INFINITY;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        ga = fmaxf(ga, fabsf(pys[k] - ymin) > 0.1f ? -1000.f : pxs[k]);
        gb = fmaxf(gb, fabsf(pxs[k] - xmax) > 0.1f ? -1000.f : pys[k]);
    }
    t[0] = (gx - px) / pw; t[1] = (gy - py) / ph; t[2] = (gt[2] - pz) / pd;
    t[3] = logf(gw / pw); t[4] = logf(gh / ph); t[5] = logf(gt[5] / pd);
    t[6] = (ga - gx) / gw; t[7] = (gb - gy) / gh;
}

// One block.  Thread i < n_pos: positive sample i (label 1: BCE + smooth-L1); n_pos <= i < n_pos + n_neg: negative sample (label 0).
// losses[0] += BCE sum / norm, losses[1] += smooth-L1 sum / norm  (norm = number of sampled anchors of the whole batch: F.binary_
// cross_entropy_with_logits is a mean over them, the box loss is divided by sampled_inds.numel(), rpn.py:401-417).
// dpred gets d(w_obj * L_obj + w_reg * L_reg)/d(pred) * grad_scale.
__global__ void __launch_bounds__(256) rpn_loss_kernel(const LossDev P, const long* __restrict__ pos, int n_pos, const long* __restrict__ neg, int n_neg,
                                                       const float* __restrict__ gt_pos, float norm, float w_obj, float w_reg, float grad_scale,
                                                       float* __restrict__ losses, float* __restrict__ targets_out, int fp16) {
    __shared__ double s_obj[256], s_reg[256];
    double l_obj = 0.0, l_reg = 0.0;
    const float inv = 1.0f / norm;
    for (int i = threadIdx.x; i < n_pos + n_neg; i += blockDim.x) {
        const bool is_pos = i < n_pos;
        const long flat = is_pos ? pos[i] : neg[i - n_pos];
        int l, a; long vox; float an[6];
        anchor_of(P, flat, l, vox, a, an);
        const float* row = P.pred[l] + (size_t)vox * 128;
        __nv_bfloat16* drow = P.dpred[l] + (size_t)vox * 128;
        const float xl = row[a], yl = is_pos ? 1.f : 0.f;
        l_obj += (double)(fmaxf(xl, 0.f) - xl * yl + log1pf(expf(-fabsf(xl))));
        const float sg = 1.f / (1.f + expf(-xl));
        store_act(drow + a, (sg - yl) * inv * w_obj * grad_scale, fp16);
        if (is_pos) {
            float t[8];
            if (P.rotated) encode_obb(an, gt_pos + (size_t)i * 7, t); else encode_aabb(an, gt_pos + (size_t)i * 6, t);
            const float beta = 1.0f / 9.0f;
            for (int j = 0; j < P.code; ++j) {
                const float p = row[P.A + a * P.code + j];
                const float d = p - t[j], ad = fabsf(d);
                l_reg += (double)(ad < beta ? 0.5f * d * d / beta : ad - 0.5f * beta);
                const float gr = ad < beta ? d / beta : (d > 0.f ? 1.f : (d < 0.f ? -1.f : 0.f));
                store_act(drow + P.A + a * P.code + j, gr * inv * w_reg * grad_scale, fp16);
                if (targets_out) targets_out[(size_t)i * P.code + j] = t[j];
            }
        }
    }
    s_obj[threadIdx.x] = l_obj; s_reg[threadIdx.x] = l_reg;
    __syncthreads();
    if (threadIdx.x == 0) {
        double a = 0.0, b = 0.0;
        for (int i = 0; i < 256; ++i) { a += s_obj[i]; b += s_reg[i]; }
        losses[0] += (float)(a / (double)norm);
        losses[1] += (float)(b / (double)norm);
    }
}

// ---------------------------------------------------------------------------------------------- optimiser side
// fp32 master weights (Cout, Cin, taps) -> 16-bit GEMM operands: fwd (taps, CoutPad, CinPad) [co][ci], and (optional) the
// backward-data operand (taps mirrored, matrices transposed) (taps, CinPadN, CoutPadK) [ci][co].  Pad rows / columns are never
// written: the buffers are zero-filled once at allocation.
__global__ void __launch_bounds__(256) pack_weights_kernel(const float* __restrict__ w, int cout, int cin, int taps, __nv_bfloat16* __restrict__ fwd,
                                                           int fwd_rows, int fwd_cols, __nv_bfloat16* __restrict__ bwd, int bwd_rows, int bwd_cols, int fp16) {
    // A 16 (co) x 16 (ci) x taps tile through shared memory: the master weight is read in runs of 16 * taps contiguous floats, both operands are
    // written in runs of 16 contiguous 16-bit values (one 32-byte sector).  (One thread per master-weight element wrote 2-byte values `rows * cols`
    // apart: 1.1 ms per training step for 184 MB.)
    extern __shared__ float tile[];                         // [16 co][16 ci][taps]
    const int co0 = blockIdx.y * 16, ci0 = blockIdx.x * 16;
    const int run = 16 * taps;
    for (int i = threadIdx.x; i < 16 * run; i += blockDim.x) {
        const int co = i / run, r = i - co * run;            // r = ci_local * taps + t
        const int ci = r / taps;
        tile[i] = (co0 + co < cout && ci0 + ci < cin) ? w[((size_t)(co0 + co) * cin + ci0) * taps + r] : 0.f;
    }
    __syncthreads();
    for (int i = threadIdx.x; i < 16 * run; i += blockDim.x) {
        const int ci = i & 15, co = (i >> 4) & 15, t = i >> 8;
        if (co0 + co < cout && ci0 + ci < cin)
            store_act(fwd + ((size_t)t * fwd_rows + co0 + co) * fwd_cols + ci0 + ci, tile[(co * 16 + ci) * taps + t], fp16);
    }
    if (bwd) {
        for (int i = threadIdx.x; i < 16 * run; i += blockDim.x) {
            const int co = i & 15, ci = (i >> 4) & 15, t = i >> 8;
            if (co0 + co < cout && ci0 + ci < cin)
                store_act(bwd + ((size_t)(taps - 1 - t) * bwd_rows + ci0 + ci) * bwd_cols + co0 + co, tile[(co * 16 + ci) * taps + t], fp16);
        }
    }
}

// out[i] = idx[i] >= 0 ? src[idx[i]] : 0, converted to 16 bits (stem weight packing through a host-built index table) or kept fp32
__global__ void gather_pack_kernel(const float* __restrict__ src, const int* __restrict__ idx, size_t n, __nv_bfloat16* __restrict__ out16,
                                   float* __restrict__ out32, float scale, int fp16) {
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        const int k = idx[i];
        const float v = k >= 0 ? src[k] * scale : 0.f;
        if (out16) store_act(out16 + i, v, fp16); else out32[i] = v;
    }
}

__global__ void __launch_bounds__(256) sumsq_partial_kernel(const float* __restrict__ g, size_t n, double* __restrict__ partial) {
    __shared__ double sh[256];
    double s = 0.0;
    const size_t per = ceil_div(n, (size_t)gridDim.x);
    const size_t i0 = (size_t)blockIdx.x * per, i1 = i0 + per < n ? i0 + per : n;
    // 128-bit loads over the 16-byte aligned middle of the block's range (fp64 accumulation per thread), scalars at the ragged ends
    const size_t a0 = (i0 + 3) & ~(size_t)3, a1 = i1 & ~(size_t)3;
    if (a0 < a1 && !(reinterpret_cast<uintptr_t>(g) & 15)) {
        for (size_t i = i0 + threadIdx.x; i < a0; i += blockDim.x) { const double v = (double)g[i]; s += v * v; }
        for (size_t i = a0 / 4 + threadIdx.x; i < a1 / 4; i += blockDim.x) {
            const float4 q = __ldg(reinterpret_cast<const float4*>(g) + i);
            s += (double)q.x * (double)q.x + (double)q.y * (double)q.y + (double)q.z * (double)q.z + (double)q.w * (double)q.w;
        }
        for (size_t i = a1 + threadIdx.x; i < i1; i += blockDim.x) { const double v = (double)g[i]; s += v * v; }
    } else {
        for (size_t i = i0 + threadIdx.x; i < i1; i += blockDim.x) { const double v = (double)g[i]; s += v * v; }
    }
    sh[threadIdx.x] = s;
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) { if (threadIdx.x < o) sh[threadIdx.x] += sh[threadIdx.x + o]; __syncthreads(); }
    if (threadIdx.x == 0) partial[blockIdx.x] = sh[0];
}

__global__ void sumsq_final_kernel(const double* __restrict__ partial, int blocks, float inv_scale, float* __restrict__ norm_out) {
    double s = 0.0;
    for (int i = 0; i < blocks; ++i) s += partial[i];
    norm_out[0] = (float)(sqrt(s) * (double)inv_scale);
}

// torch.nn.utils.clip_grad_norm_ (coefficient clamp(max_norm / (norm + 1e-6), max 1)) fused with torch.optim.AdamW's update
__global__ void __launch_bounds__(256) adamw_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m, float* __restrict__ v, size_t n,
                                                    const float* __restrict__ norm, float max_norm, float inv_scale, float lr, float beta1, float beta2,
                                                    float eps, float wd, float bc1, float bc2_sqrt) {
    float coef = inv_scale;
    if (max_norm > 0.f) { const float c = max_norm / (norm[0] + 1e-6f); coef *= c < 1.f ? c : 1.f; }
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        const float gi = g[i] * coef;
        float pi = p[i] * (1.f - lr * wd);
        const float mi = beta1 * m[i] + (1.f - beta1) * gi;
        const float vi = beta2 * v[i] + (1.f - beta2) * gi * gi;
        const float denom = sqrtf(vi) / bc2_sqrt + eps;
        pi -= (lr / bc1) * (mi / denom);
        p[i] = pi; m[i] = mi; v[i] = vi;
    }
}

}  // namespace nrpn

using namespace nrpn;

extern "C" {
#pragma GCC visibility push(default)

size_t nrpn_chan_reduce_workspace_bytes(int c) { return c < 1 ? 0 : (size_t)kRedBlocks * 2 * c * sizeof(float) + 256; }

static int chan_reduce_check(const void* a, long rows, int c, void* ws, size_t ws_bytes) {
    if (!a || !ws || rows < 1 || c < 8 || c % 8 != 0 || c > 2048) return NRPN_ERR_INVALID;
    if (reinterpret_cast<uintptr_t>(a) % 16 != 0) return NRPN_ERR_INVALID;
    if (ws_bytes < nrpn_chan_reduce_workspace_bytes(c)) return NRPN_ERR_WORKSPACE;
    return NRPN_OK;
}

int nrpn_bn_stats(const void* y, long rows, int c, int act_fp16, float eps, float* stats, float* running_mean, float* running_var,
                  float momentum, void* workspace, size_t workspace_bytes, nrpn_stream_t stream) {
    { const int rc = chan_reduce_check(y, rows, c, workspace, workspace_bytes); if (rc) return rc; }
    if (!stats || (running_mean == nullptr) != (running_var == nullptr)) return NRPN_ERR_INVALID;
    float* partial = reinterpret_cast<float*>(align_up((size_t)workspace, 256));
    const int blocks = rows < kRedBlocks ? (int)rows : kRedBlocks;
    cudaStream_t st = (cudaStream_t)stream;
    chan_reduce_kernel<0><<<blocks, 256, 2 * c * sizeof(float), st>>>(reinterpret_cast<const __nv_bfloat16*>(y), nullptr, nullptr, rows, c, nullptr, 0,
                                                                     act_fp16 ? 1 : 0, partial);
    NRPN_LAUNCH_CHECK();
    chan_reduce_final_kernel<0><<<ceil_div(c, 8), 256, 0, st>>>(partial, blocks, c, rows, eps, stats, running_mean, running_var, momentum);
    NRPN_LAUNCH_CHECK();
    return NRPN_OK;
}

int nrpn_bn_apply(const void* y, const void* res, void* out, long rows, int c, const float* stats, const float* gamma, const float* beta,
                  int relu, int act_fp16, nrpn_stream_t stream) {
    if (!y || !out || !stats || !gamma || !beta || rows < 1 || c < 8 || c % 8 != 0) return NRPN_ERR_INVALID;
    const size_t chunks = (size_t)rows * (c / 8);
    bn_apply_kernel<<<grid1d(chunks, 256), 256, 0, (cudaStream_t)stream>>>(reinterpret_cast<const __nv_bfloat16*>(y), reinterpret_cast<const __nv_bfloat16*>(res),
                                                                           reinterpret_cast<__nv_bfloat16*>(out), chunks, c, stats, gamma, beta, relu ? 1 : 0,
                                                                           act_fp16 ? 1 : 0);
    NRPN_LAUNCH_CHECK();
    return NRPN_OK;
}

int nrpn_bn_backward(const void* dout, const void* act, const void* y, void* dy, void* dres, long rows, int c, const float* stats,
                     const float* gamma, float* sums, int relu, int act_fp16, void* workspace, size_t workspace_bytes, nrpn_stream_t stream) {
    { const int rc = chan_reduce_check(dout, rows, c, workspace, workspace_bytes); if (rc) return rc; }
    if (!y || !dy || !stats || !gamma || !sums || (relu && !act)) return NRPN_ERR_INVALID;
    float* partial = reinterpret_cast<float*>(align_up((size_t)workspace, 256));
    const int blocks = rows < kRedBlocks ? (int)rows : kRedBlocks;
    cudaStream_t st = (cudaStream_t)stream;
    const int f = act_fp16 ? 1 : 0;
    chan_reduce_kernel<1><<<blocks, 256, 2 * c * sizeof(float), st>>>(reinterpret_cast<const __nv_bfloat16*>(dout), reinterpret_cast<const __nv_bfloat16*>(act),
                                                                     reinterpret_cast<const __nv_bfloat16*>(y), rows, c, stats, relu ? 1 : 0, f, partial);
    NRPN_LAUNCH_CHECK();
    chan_reduce_final_kernel<1><<<ceil_div(c, 8), 256, 0, st>>>(partial, blocks, c, rows, 0.f, sums, nullptr, nullptr, 0.f);
    NRPN_LAUNCH_CHECK();
    const size_t chunks = (size_t)rows * (c / 8);
    bn_backward_apply_kernel<<<grid1d(chunks, 256), 256, 0, st>>>(reinterpret_cast<const __nv_bfloat16*>(dout), reinterpret_cast<const __nv_bfloat16*>(act),
                                                                  reinterpret_cast<const __nv_bfloat16*>(y), reinterpret_cast<__nv_bfloat16*>(dy),
                                                                  reinterpret_cast<__nv_bfloat16*>(dres), chunks, c, rows, stats, gamma, sums, relu ? 1 : 0, f);
    NRPN_LAUNCH_CHECK();
    return NRPN_OK;
}

int nrpn_maxpool3d_k3s2_argmax(const void* in, int n, int x, int y, int z, int c, void* out, uint8_t* idx, int act_fp16, nrpn_stream_t stream) {
    if (!in || !out || !idx || n < 1 || x < 1 || y < 1 || z < 1 || c < 8 || c % 8 != 0) return NRPN_ERR_INVALID;
    const int Xo = (x - 1) / 2 + 1, Yo = (y - 1) / 2 + 1, Zo = (z - 1) / 2 + 1;
    const size_t total = (size_t)n * Xo * Yo * Zo * (c / 8);
    maxpool_k3s2_argmax_kernel<<<grid1d(total, 256), 256, 0, (cudaStream_t)stream>>>(reinterpret_cast<const __nv_bfloat16*>(in), n, x, y, z, c, Xo, Yo, Zo,
                                                                                     reinterpret_cast<__nv_bfloat16*>(out), idx, act_fp16 ? 1 : 0);
    NRPN_LAUNCH_CHECK();
    return NRPN_OK;
}

int nrpn_maxpool3d_k3s2_backward(const void* dy, const uint8_t* idx, int n, int x, int y, int z, int c, void* dx, int act_fp16, nrpn_stream_t stream) {
    if (!dy || !dx || !idx || n < 1 || x < 1 || y < 1 || z < 1 || c < 8 || c % 8 != 0) return NRPN_ERR_INVALID;
    const int Xo = (x - 1) / 2 + 1, Yo = (y - 1) / 2 + 1, Zo = (z - 1) / 2 + 1;
    const size_t total = (size_t)n * x * y * z * (c / 8);
    maxpool_k3s2_backward_kernel<<<grid1d(total, 256), 256, 0, (cudaStream_t)stream>>>(reinterpret_cast<const __nv_bfloat16*>(dy), idx, n, x, y, z, c, Xo, Yo, Zo,
                                                                                       reinterpret_cast<__nv_bfloat16*>(dx), act_fp16 ? 1 : 0);
    NRPN_LAUNCH_CHECK();
    return NRPN_OK;
}

int nrpn_upsample_nearest_backward(const void* dfine, int n, int xf, int yf, int zf, int xc, int yc, int zc, int c, void* dcoarse, int accumulate,
                                   int act_fp16, nrpn_stream_t stream) {
    if (!dfine || !dcoarse || n < 1 || xf < 1 || yf < 1 || zf < 1 || xc < 1 || yc < 1 || zc < 1 || c < 8 || c % 8 != 0) return NRPN_ERR_INVALID;
    const size_t total = (size_t)n * xc * yc * zc * (c / 8);
    upsample_nearest_backward_kernel<<<grid1d(total, 256), 256, 0, (cudaStream_t)stream>>>(reinterpret_cast<const __nv_bfloat16*>(dfine), n, xf, yf, zf, xc, yc, zc, c,
                                                                                           reinterpret_cast<__nv_bfloat16*>(dcoarse), accumulate ? 1 : 0,
                                                                                           act_fp16 ? 1 : 0);
    NRPN_LAUNCH_CHECK();
    return NRPN_OK;
}

int nrpn_stride2(const void* src, void* dst, int n, int x, int y, int z, int c, int scatter, nrpn_stream_t stream) {
    if (!src || !dst || n < 1 || x < 1 || y < 1 || z < 1 || c < 8 || c % 8 != 0) return NRPN_ERR_INVALID;
    const int Xo = (x + 1) / 2, Yo = (y + 1) / 2, Zo = (z + 1) / 2;
    const size_t total = scatter ? (size_t)n * x * y * z * (c / 8) : (size_t)n * Xo * Yo * Zo * (c / 8);
    stride2_kernel<<<grid1d(total, 256), 256, 0, (cudaStream_t)stream>>>(reinterpret_cast<const uint4*>(src), reinterpret_cast<uint4*>(dst), n, x, y, z, Xo, Yo, Zo,
                                                                         c / 8, scatter ? 1 : 0);
    NRPN_LAUNCH_CHECK();
    return NRPN_OK;
}

int nrpn_add_inplace(void* a, const void* b, size_t elements, int act_fp16, nrpn_stream_t stream) {
    if (!a || !b || elements < 8 || elements % 8 != 0) return NRPN_ERR_INVALID;
    add_inplace_kernel<<<grid1d(elements / 8, 256), 256, 0, (cudaStream_t)stream>>>(reinterpret_cast<__nv_bfloat16*>(a), reinterpret_cast<const __nv_bfloat16*>(b),
                                                                                    elements / 8, act_fp16 ? 1 : 0);
    NRPN_LAUNCH_CHECK();
    return NRPN_OK;
}

int nrpn_rpn_loss(const nrpn_rpn_desc* d, void* const* dpred, const int64_t* pos_idx, int n_pos, const int64_t* neg_idx, int n_neg,
                  const float* gt_pos, float norm, float w_obj, float w_reg, float grad_scale, float* losses, float* targets_out,
                  int act_fp16, nrpn_stream_t stream) {
    if (!d || !dpred || !losses || d->n_levels < 1 || d->n_levels > NRPN_RPN_MAX_LEVELS || d->num_anchors < 1 || d->num_anchors > 16) return NRPN_ERR_INVALID;
    if (n_pos < 0 || n_neg < 0 || (n_pos > 0 && (!pos_idx || !gt_pos)) || (n_neg > 0 && !neg_idx) || !(norm > 0.f)) return NRPN_ERR_INVALID;
    const int code = d->rotated ? 8 : 6;
    if (d->num_anchors * (1 + code) > 128) return NRPN_ERR_UNSUPPORTED;
    if (n_pos + n_neg == 0) return NRPN_OK;
    LossDev P;
    memset(&P, 0, sizeof(P));
    P.n_levels = d->n_levels; P.A = d->num_anchors; P.code = code; P.rotated = d->rotated;
    long begin = 0;
    for (int l = 0; l < d->n_levels; ++l) {
        const nrpn_rpn_level& L = d->level[l];
        if (!L.pred || !dpred[l] || L.ld != 128) return NRPN_ERR_INVALID;
        P.pred[l] = const_cast<float*>(L.pred); P.dpred[l] = reinterpret_cast<__nv_bfloat16*>(dpred[l]);
        P.gx[l] = L.gx; P.gy[l] = L.gy; P.gz[l] = L.gz; P.sx[l] = L.sx; P.sy[l] = L.sy; P.sz[l] = L.sz;
        P.begin[l] = begin;
        begin += (long)L.gx * L.gy * L.gz * d->num_anchors;
        for (int a = 0; a < d->num_anchors; ++a) for (int k = 0; k < 6; ++k) P.cell[l][a][k] = d->cell_anchors[l][a][k];
    }
    P.begin[d->n_levels] = begin;
    rpn_loss_kernel<<<1, 256, 0, (cudaStream_t)stream>>>(P, reinterpret_cast<const long*>(pos_idx), n_pos, reinterpret_cast<const long*>(neg_idx), n_neg, gt_pos,
                                                         norm, w_obj, w_reg, grad_scale, losses, targets_out, act_fp16 ? 1 : 0);
    NRPN_LAUNCH_CHECK();
    return NRPN_OK;
}

int nrpn_pack_weights(const float* w, int cout, int cin, int taps, void* fwd, int fwd_rows, int fwd_cols, void* bwd, int bwd_rows, int bwd_cols,
                      int act_fp16, nrpn_stream_t stream) {
    if (!w || !fwd || cout < 1 || cin < 1 || taps < 1 || fwd_rows < cout || fwd_cols < cin) return NRPN_ERR_INVALID;
    if (bwd && (bwd_rows < cin || bwd_cols < cout)) return NRPN_ERR_INVALID;
    const size_t total = (size_t)cout * cin * taps;
    (void)total;
    const dim3 grid((unsigned)ceil_div(cin, 16), (unsigned)ceil_div(cout, 16));
    const size_t smem = (size_t)256 * taps * sizeof(float);
    if (grid.y > 65535 || smem > 48 * 1024) return NRPN_ERR_UNSUPPORTED;        // taps <= 48 (3^3 = 27; the 7^3 stem goes through nrpn_gather_pack)
    pack_weights_kernel<<<grid, 256, smem, (cudaStream_t)stream>>>(w, cout, cin, taps, reinterpret_cast<__nv_bfloat16*>(fwd), fwd_rows, fwd_cols,
                                                                   reinterpret_cast<__nv_bfloat16*>(bwd), bwd_rows, bwd_cols, act_fp16 ? 1 : 0);
    NRPN_LAUNCH_CHECK();
    return NRPN_OK;
}

int nrpn_gather_pack(const float* src, const int32_t* idx, size_t n, void* out16, float* out32, float scale, int act_fp16, nrpn_stream_t stream) {
    if (!src || !idx || n < 1 || ((out16 == nullptr) == (out32 == nullptr))) return NRPN_ERR_INVALID;
    gather_pack_kernel<<<grid1d(n, 256), 256, 0, (cudaStream_t)stream>>>(src, idx, n, reinterpret_cast<__nv_bfloat16*>(out16), out32, scale, act_fp16 ? 1 : 0);
    NRPN_LAUNCH_CHECK();
    return NRPN_OK;
}

size_t nrpn_grad_norm_workspace_bytes(void) { return (size_t)kRedBlocks * sizeof(double) + 256; }

int nrpn_grad_norm(const float* g, size_t n, float inv_scale, float* norm_out, void* workspace, size_t workspace_bytes, nrpn_stream_t stream) {
    if (!g || !norm_out || !workspace || n < 1) return NRPN_ERR_INVALID;
    if (workspace_bytes < nrpn_grad_norm_workspace_bytes()) return NRPN_ERR_WORKSPACE;
    double* partial = reinterpret_cast<double*>(align_up((size_t)workspace, 256));
    cudaStream_t st = (cudaStream_t)stream;
    sumsq_partial_kernel<<<kRedBlocks, 256, 0, st>>>(g, n, partial);
    NRPN_LAUNCH_CHECK();
    sumsq_final_kernel<<<1, 1, 0, st>>>(partial, kRedBlocks, inv_scale, norm_out);
    NRPN_LAUNCH_CHECK();
    return NRPN_OK;
}

int nrpn_adamw_step(float* p, const float* g, float* m, float* v, size_t n, const float* norm, float max_norm, float inv_scale, float lr, float beta1,
                    float beta2, float eps, float weight_decay, int step, nrpn_stream_t stream) {
    if (!p || !g || !m || !v || n < 1 || step < 1 || (max_norm > 0.f && !norm)) return NRPN_ERR_INVALID;
    const float bc1 = 1.0f - powf(beta1, (float)step);
    const float bc2s = sqrtf(1.0f - powf(beta2, (float)step));
    adamw_kernel<<<grid1d(n, 256), 256, 0, (cudaStream_t)stream>>>(p, g, m, v, n, norm, max_norm, inv_scale, lr, beta1, beta2, eps, weight_decay, bc1, bc2s);
    NRPN_LAUNCH_CHECK();
    return NRPN_OK;
}

#pragma GCC visibility pop
}  // extern "C"

// ---------------------------------------------------------------------------------------------- training-time scene augmentation
// BaseDataset.augment_rpn_inputs + rotate_and_scale_scene (datasets.py:109-163, 290-329) on the device, on the grid in its on-disk
// channels-last order (X, Y, Z, 4): one thread per output voxel, one 128-bit access per source voxel.
//   step 1 (optional) rot90 about z:   out1[i][j] = in[j][X1 - 1 - i]          (torch.transpose(1, 2) then flip(1); extents swap)
//   step 2 (optional) flips along x/y: out2[i][j] = out1[X2-1-i or i][Y2-1-j or j]
//   step 3 (optional) rotate + scale:  F.grid_sample(trilinear, zeros padding, align_corners=True) at the source point the reference's
//                                      grid construction yields: p = scale * R(angle) (c - centre) + centre in normalised units
namespace nrpn {

struct AugParams { int X, Y, Z, Xo, Yo, rot90, flipx, flipy, resample; float c00, c01, c10, c11, s; };

__device__ __forceinline__ float4 aug_fetch(const float4* __restrict__ in, const AugParams& P, int i, int j, int k) {
    // (i, j, k) index the grid AFTER rot90 / flips (extent Xo x Yo x Z); map back to the stored grid (X x Y x Z)
    if (i < 0 || j < 0 || k < 0 || i >= P.Xo || j >= P.Yo || k >= P.Z) return make_float4(0.f, 0.f, 0.f, 0.f);
    if (P.flipx) i = P.Xo - 1 - i;
    if (P.flipy) j = P.Yo - 1 - j;
    int si = i, sj = j;
    if (P.rot90) { si = j; sj = P.Y - 1 - i; }          // out1[i][j] = in[j][Y_in - 1 - i] with out1 extents (Y_in, X_in)
    return __ldg(in + ((size_t)si * P.Y + sj) * P.Z + k);
}

__global__ void __launch_bounds__(256) augment_scene_kernel(const float4* __restrict__ in, float4* __restrict__ out, const AugParams P) {
    const size_t total = (size_t)P.Xo * P.Yo * P.Z;
    for (size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (size_t)gridDim.x * blockDim.x) {
        const int k = (int)(t % P.Z); size_t v = t / P.Z;
        const int j = (int)(v % P.Yo); const int i = (int)(v / P.Yo);
        if (!P.resample) { out[t] = aug_fetch(in, P, i, j, k); continue; }
        // reference: x = linspace(-1, 1, res) * res / 2 (voxel i -> (2 i / (res - 1) - 1) * res / 2), grid = [x y z] @ xform^T, then divided by
        // res / 2 per axis -> normalised coordinates; align_corners=True: pixel = (g + 1) / 2 * (res - 1)
        const float hx = 0.5f * (float)P.Xo, hy = 0.5f * (float)P.Yo;
        const float x = (P.Xo > 1 ? (2.0f * (float)i / (float)(P.Xo - 1) - 1.0f) : -1.0f) * hx;
        const float y = (P.Yo > 1 ? (2.0f * (float)j / (float)(P.Yo - 1) - 1.0f) : -1.0f) * hy;
        const float gx = (P.c00 * x + P.c01 * y) / hx, gy = (P.c10 * x + P.c11 * y) / hy;
        const float gz = (P.Z > 1 ? (2.0f * (float)k / (float)(P.Z - 1) - 1.0f) : -1.0f) * P.s;
        const float fx = (gx + 1.0f) * 0.5f * (float)(P.Xo - 1), fy = (gy + 1.0f) * 0.5f * (float)(P.Yo - 1), fz = (gz + 1.0f) * 0.5f * (float)(P.Z - 1);
        const int x0 = (int)floorf(fx), y0 = (int)floorf(fy), z0 = (int)floorf(fz);
        const float tx = fx - (float)x0, ty = fy - (float)y0, tz = fz - (float)z0;
        float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
        for (int c = 0; c < 8; ++c) {
            const int dx = c & 1, dy = (c >> 1) & 1, dz = c >> 2;
            const float w = (dx ? tx : 1.0f - tx) * (dy ? ty : 1.0f - ty) * (dz ? tz : 1.0f - tz);
            const float4 q = aug_fetch(in, P, x0 + dx, y0 + dy, z0 + dz);
            acc.x += w * q.x; acc.y += w * q.y; acc.z += w * q.z; acc.w += w * q.w;
        }
        out[t] = acc;
    }
}

}  // namespace nrpn

extern "C" {
#pragma GCC visibility push(default)

int nrpn_augment_scene(const float* grid_xyzc, int x, int y, int z, float* out_xyzc, int rot90, int flip_x, int flip_y, int resample,
                       float angle, float scale, nrpn_stream_t stream) {
    if (!grid_xyzc || !out_xyzc || x < 1 || y < 1 || z < 1 || grid_xyzc == out_xyzc) return NRPN_ERR_INVALID;
    if (reinterpret_cast<uintptr_t>(grid_xyzc) % 16 != 0 || reinterpret_cast<uintptr_t>(out_xyzc) % 16 != 0) return NRPN_ERR_INVALID;
    nrpn::AugParams P;
    P.X = x; P.Y = y; P.Z = z; P.rot90 = rot90 ? 1 : 0; P.flipx = flip_x ? 1 : 0; P.flipy = flip_y ? 1 : 0; P.resample = resample ? 1 : 0;
    P.Xo = rot90 ? y : x; P.Yo = rot90 ? x : y;
    // xform = [[cos, -sin, 0], [sin, cos, 0], [0, 0, 1]] * scale (datasets.py:293-297, fp32)
    P.c00 = (float)cos((double)angle) * scale; P.c01 = -(float)sin((double)angle) * scale;
    P.c10 = (float)sin((double)angle) * scale; P.c11 = (float)cos((double)angle) * scale; P.s = scale;
    const size_t total = (size_t)P.Xo * P.Yo * z;
    nrpn::augment_scene_kernel<<<nrpn::grid1d(total, 256), 256, 0, (cudaStream_t)stream>>>(reinterpret_cast<const float4*>(grid_xyzc),
                                                                                          reinterpret_cast<float4*>(out_xyzc), P);
    NRPN_LAUNCH_CHECK();
    return NRPN_OK;
}

#pragma GCC visibility pop
}  // extern "C"
