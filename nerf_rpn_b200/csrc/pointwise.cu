// Bandwidth-bound helpers around the convolutions (HBM roofline kernels; 16-byte coalesced accesses).
#include "common.cuh"

namespace nrpn {

// fp32 NCDHW grid (N,4,X,Y,Z) -> bf16 (N, X2, Y2, Z2+1, 64), X2 = ceil(X/2) etc.
// Row (i,j,k) holds two 2x2x2 space-to-depth blocks: channels [0,32) = block (i,j,k-1), [32,64) = block (i,j,k);
// inside a block channel = ((rx*2+ry)*2+rz)*4 + c for input voxel (2i+rx, 2j+ry, 2k'+rz), zero outside the grid.
// With this layout the reference's stem Conv3d(4,64,k=7,s=2,p=3) (feature_extractor.py:163) is a stride-1
// implicit GEMM with 4x4x2 taps of K = 64 (see nerf_rpn_b200/engine.py: pack_stem_weight).
// One thread writes one 16-byte chunk (8 channels); 8 consecutive lanes cover one 128-byte row.
// density_to_alpha (datasets.py:165-167, applied by the reference's dataset on the host when --normalize_density is set):
// alpha = clip(1 - exp(-exp(sigma) / 100), 0, 1) on the last channel, fp32 like numpy computes it on a float32 array.
__device__ __forceinline__ float density_to_alpha(float sigma) {
    const float a = 1.0f - expf(-__fdiv_rn(expf(sigma), 100.0f));
    return fminf(fmaxf(a, 0.0f), 1.0f);
}

__global__ void pack_stem_kernel(const float* __restrict__ grid, int n, int X, int Y, int Z, int X2, int Y2, int Z2,
                                 __nv_bfloat16* __restrict__ out, int fp16, int alpha) {
    const size_t total = (size_t)n * X2 * Y2 * (Z2 + 1) * 8;
    for (size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (size_t)gridDim.x * blockDim.x) {
        const int s = (int)(t & 7);
        size_t v = t >> 3;
        const int k = (int)(v % (Z2 + 1)); v /= (Z2 + 1);
        const int j = (int)(v % Y2); v /= Y2;
        const int i = (int)(v % X2); const int b = (int)(v / X2);
        const int half = s >> 2, rx = (s >> 1) & 1, ry = s & 1;
        const int kk = k - 1 + half;                    // s2d block index along z
        const int x = 2 * i + rx, y = 2 * j + ry, z = 2 * kk;
        float val[8];                                   // order: rz major, c minor
#pragma unroll
        for (int q = 0; q < 8; ++q) val[q] = 0.f;
        if (kk >= 0 && kk < Z2 && x < X && y < Y) {
#pragma unroll
            for (int c = 0; c < 4; ++c) {
                const float* p = grid + ((((size_t)b * 4 + c) * X + x) * Y + y) * Z + z;
                val[c] = p[0];
                if (z + 1 < Z) val[4 + c] = p[1];
            }
            if (alpha) { val[3] = density_to_alpha(val[3]); if (z + 1 < Z) val[7] = density_to_alpha(val[7]); }
        }
        uint32_t h[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) h[q] = pack_act2(val[2 * q], val[2 * q + 1], fp16);
        *reinterpret_cast<uint4*>(out + (t << 3)) = make_uint4(h[0], h[1], h[2], h[3]);
    }
}

// Same packing from the grid as it is stored on disk and handed over by the reference's dataset (datasets.py:49-57: a
// (4,W,L,H) VIEW of the (W,L,H,4) array): one 128-bit load per voxel instead of four scalar loads from four channel planes.
__global__ void pack_stem_cl_kernel(const float4* __restrict__ grid, int n, int X, int Y, int Z, int X2, int Y2, int Z2,
                                    __nv_bfloat16* __restrict__ out, int fp16, int alpha) {
    const size_t total = (size_t)n * X2 * Y2 * (Z2 + 1) * 8;
    for (size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (size_t)gridDim.x * blockDim.x) {
        const int s = (int)(t & 7);
        size_t v = t >> 3;
        const int k = (int)(v % (Z2 + 1)); v /= (Z2 + 1);
        const int j = (int)(v % Y2); v /= Y2;
        const int i = (int)(v % X2); const int b = (int)(v / X2);
        const int half = s >> 2, rx = (s >> 1) & 1, ry = s & 1;
        const int kk = k - 1 + half;
        const int x = 2 * i + rx, y = 2 * j + ry, z = 2 * kk;
        float4 a = make_float4(0.f, 0.f, 0.f, 0.f), c = a;
        if (kk >= 0 && kk < Z2 && x < X && y < Y) {
            const float4* p = grid + (((size_t)b * X + x) * Y + y) * Z + z;
            a = __ldg(p);
            if (z + 1 < Z) c = __ldg(p + 1);
            if (alpha) { a.w = density_to_alpha(a.w); if (z + 1 < Z) c.w = density_to_alpha(c.w); }
        }
        const uint32_t h0 = pack_act2(a.x, a.y, fp16), h1 = pack_act2(a.z, a.w, fp16);
        const uint32_t h2 = pack_act2(c.x, c.y, fp16), h3 = pack_act2(c.z, c.w, fp16);
        *reinterpret_cast<uint4*>(out + (t << 3)) = make_uint4(h0, h1, h2, h3);
    }
}

// uint8 grids (datasets.py:59-61 normalises them with .float() / 255.0 on the host): the raw (N,X,Y,Z,4) bytes are copied to the
// device (a quarter of the fp32 H2D traffic) and normalised here, one 32-bit load per voxel; the division is the same correctly
// rounded fp32 x / 255 the reference performs.
__global__ void pack_stem_cl_u8_kernel(const uint32_t* __restrict__ grid, int n, int X, int Y, int Z, int X2, int Y2, int Z2,
                                       __nv_bfloat16* __restrict__ out, int fp16) {
    const size_t total = (size_t)n * X2 * Y2 * (Z2 + 1) * 8;
    for (size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (size_t)gridDim.x * blockDim.x) {
        const int s = (int)(t & 7);
        size_t v = t >> 3;
        const int k = (int)(v % (Z2 + 1)); v /= (Z2 + 1);
        const int j = (int)(v % Y2); v /= Y2;
        const int i = (int)(v % X2); const int b = (int)(v / X2);
        const int half = s >> 2, rx = (s >> 1) & 1, ry = s & 1;
        const int kk = k - 1 + half;
        const int x = 2 * i + rx, y = 2 * j + ry, z = 2 * kk;
        uint32_t a = 0u, c = 0u;
        if (kk >= 0 && kk < Z2 && x < X && y < Y) {
            const uint32_t* p = grid + (((size_t)b * X + x) * Y + y) * Z + z;
            a = __ldg(p);
            if (z + 1 < Z) c = __ldg(p + 1);
        }
        auto f = [](uint32_t w, int byte) { return __fdiv_rn((float)((w >> (8 * byte)) & 0xFFu), 255.0f); };
        const uint32_t h0 = pack_act2(f(a, 0), f(a, 1), fp16), h1 = pack_act2(f(a, 2), f(a, 3), fp16);
        const uint32_t h2 = pack_act2(f(c, 0), f(c, 1), fp16), h3 = pack_act2(f(c, 2), f(c, 3), fp16);
        *reinterpret_cast<uint4*>(out + (t << 3)) = make_uint4(h0, h1, h2, h3);
    }
}

// F.max_pool3d(k=3, s=2, p=1) on channels-last bf16; one thread per (output voxel, 8 channels).  A NaN in the window makes
// the output NaN, as in torch.
__global__ void maxpool_k3s2_kernel(const __nv_bfloat16* __restrict__ in, int n, int X, int Y, int Z, int C, int Xo, int Yo,
                                    int Zo, __nv_bfloat16* __restrict__ out, int fp16) {
    const int cg = C >> 3;
    const size_t total = (size_t)n * Xo * Yo * Zo * cg;
    for (size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (size_t)gridDim.x * blockDim.x) {
        const int g = (int)(t % cg); size_t v = t / cg;
        const int k = (int)(v % Zo); v /= Zo;
        const int j = (int)(v % Yo); v /= Yo;
        const int i = (int)(v % Xo); const int b = (int)(v / Xo);
        float m[8];
#pragma unroll
        for (int q = 0; q < 8; ++q) m[q] = -INFINITY;
        // out-of-range taps are clamped onto the border voxel instead of skipped: a maximum ignores duplicates, and the 27
        // loads become branch-free and independent (all in flight at once)
        const __nv_bfloat16* base = in + (size_t)b * X * Y * Z * C + g * 8;
#pragma unroll
        for (int dx = -1; dx <= 1; ++dx) {
            const int x = min(max(2 * i + dx, 0), X - 1);
#pragma unroll
            for (int dy = -1; dy <= 1; ++dy) {
                const int y = min(max(2 * j + dy, 0), Y - 1);
                uint4 raw[3];
#pragma unroll
                for (int dz = -1; dz <= 1; ++dz) {
                    const int z = min(max(2 * k + dz, 0), Z - 1);
                    raw[dz + 1] = __ldg(reinterpret_cast<const uint4*>(base + (((size_t)x * Y + y) * Z + z) * C));
                }
#pragma unroll
                for (int dz = 0; dz < 3; ++dz) {
                    const uint32_t* h = reinterpret_cast<const uint32_t*>(&raw[dz]);
#pragma unroll
                    for (int q = 0; q < 4; ++q) { const float2 f = unpack_act2(h[q], fp16); m[2 * q] = max_nan(m[2 * q], f.x); m[2 * q + 1] = max_nan(m[2 * q + 1], f.y); }
                }
            }
        }
        uint32_t o[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) o[q] = pack_act2(m[2 * q], m[2 * q + 1], fp16);
        *reinterpret_cast<uint4*>(out + ((((size_t)b * Xo + i) * Yo + j) * Zo + k) * C + g * 8) = make_uint4(o[0], o[1], o[2], o[3]);
    }
}

// nn.MaxPool3d(kernel 2, stride 2, ceil_mode=True) on channels-last bf16 (VGG stages, feature_extractor.py:347):
// output extent ceil(in/2); the last window is clipped at the border.  NaN propagates, as in torch.
__global__ void maxpool_k2s2_ceil_kernel(const __nv_bfloat16* __restrict__ in, int n, int X, int Y, int Z, int C, int Xo, int Yo,
                                         int Zo, __nv_bfloat16* __restrict__ out, int fp16) {
    const int cg = C >> 3;
    const size_t total = (size_t)n * Xo * Yo * Zo * cg;
    for (size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (size_t)gridDim.x * blockDim.x) {
        const int g = (int)(t % cg); size_t v = t / cg;
        const int k = (int)(v % Zo); v /= Zo;
        const int j = (int)(v % Yo); v /= Yo;
        const int i = (int)(v % Xo); const int b = (int)(v / Xo);
        float m[8];
#pragma unroll
        for (int q = 0; q < 8; ++q) m[q] = -INFINITY;
#pragma unroll
        for (int dx = 0; dx < 2; ++dx) {
            const int x = 2 * i + dx; if (x >= X) continue;
#pragma unroll
            for (int dy = 0; dy < 2; ++dy) {
                const int y = 2 * j + dy; if (y >= Y) continue;
#pragma unroll
                for (int dz = 0; dz < 2; ++dz) {
                    const int z = 2 * k + dz; if (z >= Z) continue;
                    const uint4 raw = __ldg(reinterpret_cast<const uint4*>(in + ((((size_t)b * X + x) * Y + y) * Z + z) * C + g * 8));
                    const uint32_t* h = reinterpret_cast<const uint32_t*>(&raw);
#pragma unroll
                    for (int q = 0; q < 4; ++q) { const float2 f = unpack_act2(h[q], fp16); m[2 * q] = max_nan(m[2 * q], f.x); m[2 * q + 1] = max_nan(m[2 * q + 1], f.y); }
                }
            }
        }
        uint32_t o[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) o[q] = pack_act2(m[2 * q], m[2 * q + 1], fp16);
        *reinterpret_cast<uint4*>(out + ((((size_t)b * Xo + i) * Yo + j) * Zo + k) * C + g * 8) = make_uint4(o[0], o[1], o[2], o[3]);
    }
}

// Stride-1 stem packing (VGG_FPN for grids < 160: Conv3d(4,64,k=7,s=1,p=3), feature_extractor.py:341):
// fp32 NCDHW (N,4,X,Y,Z) -> bf16 (N, X, Y+1, Z, 64).  Row (x, yp, z) holds, for the two input rows y = yp-1 and yp, the seven
// z-neighbours z-3..z+3 of all 4 channels: channel = ((yy*7 + zz)*4 + c), 56 used + 8 zero.  The 7^3 conv becomes a
// 7 (dx) x 4 (y pairs) tap implicit GEMM with K = 64 per tap (packing.pack_stem_s1_weight).
__global__ void pack_stem_s1_kernel(const float* __restrict__ grid, int n, int X, int Y, int Z, __nv_bfloat16* __restrict__ out, int fp16) {
    const size_t total = (size_t)n * X * (Y + 1) * Z * 8;
    for (size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (size_t)gridDim.x * blockDim.x) {
        const int s = (int)(t & 7);
        size_t v = t >> 3;
        const int z = (int)(v % Z); v /= Z;
        const int yp = (int)(v % (Y + 1)); v /= (Y + 1);
        const int x = (int)(v % X); const int b = (int)(v / X);
        float val[8];
#pragma unroll
        for (int e = 0; e < 8; ++e) {
            const int ch = s * 8 + e;
            float f = 0.f;
            if (ch < 56) {
                const int c = ch & 3, zz = (ch >> 2) % 7, yy = (ch >> 2) / 7;
                const int y = yp - 1 + yy, zi = z + zz - 3;
                if (y >= 0 && y < Y && zi >= 0 && zi < Z) f = grid[((((size_t)b * 4 + c) * X + x) * Y + y) * Z + zi];
            }
            val[e] = f;
        }
        uint32_t h[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) h[q] = pack_act2(val[2 * q], val[2 * q + 1], fp16);
        *reinterpret_cast<uint4*>(out + (t << 3)) = make_uint4(h[0], h[1], h[2], h[3]);
    }
}

static inline unsigned grid_for(size_t total, int block) {
    size_t g = (total + block - 1) / block;
    const size_t cap = (size_t)num_sms() * 16;
    return (unsigned)(g < cap ? (g ? g : 1) : cap);
}

}  // namespace nrpn

using namespace nrpn;

extern "C" {
#pragma GCC visibility push(default)

int nrpn_pack_stem_input_ex(const float* grid, int n, int x, int y, int z, void* packed, int act_fp16, int channels_last, int density_to_alpha,
                            nrpn_stream_t stream) {
    const int alpha = density_to_alpha ? 1 : 0;
    if (!grid || !packed || n < 1 || x < 1 || y < 1 || z < 1) return NRPN_ERR_INVALID;
    const int X2 = (x + 1) / 2, Y2 = (y + 1) / 2, Z2 = (z + 1) / 2;
    const size_t total = (size_t)n * X2 * Y2 * (Z2 + 1) * 8;
    if (channels_last) {
        if (reinterpret_cast<uintptr_t>(grid) % 16 != 0) return NRPN_ERR_INVALID;
        pack_stem_cl_kernel<<<grid_for(total, 256), 256, 0, (cudaStream_t)stream>>>(reinterpret_cast<const float4*>(grid), n, x, y, z, X2, Y2, Z2,
                                                                                   reinterpret_cast<__nv_bfloat16*>(packed), act_fp16 ? 1 : 0, alpha);
        NRPN_LAUNCH_CHECK();
        return NRPN_OK;
    }
    pack_stem_kernel<<<grid_for(total, 256), 256, 0, (cudaStream_t)stream>>>(grid, n, x, y, z, X2, Y2, Z2,
                                                                            reinterpret_cast<__nv_bfloat16*>(packed), act_fp16 ? 1 : 0, alpha);
    NRPN_LAUNCH_CHECK();
    return NRPN_OK;
}

int nrpn_pack_stem_input(const float* grid, int n, int x, int y, int z, void* packed, int act_fp16, int channels_last, nrpn_stream_t stream) {
    return nrpn_pack_stem_input_ex(grid, n, x, y, z, packed, act_fp16, channels_last, 0, stream);
}

int nrpn_pack_stem_input_u8(const uint8_t* grid, int n, int x, int y, int z, void* packed, int act_fp16, nrpn_stream_t stream) {
    if (!grid || !packed || n < 1 || x < 1 || y < 1 || z < 1) return NRPN_ERR_INVALID;
    if (reinterpret_cast<uintptr_t>(grid) % 4 != 0) return NRPN_ERR_INVALID;
    const int X2 = (x + 1) / 2, Y2 = (y + 1) / 2, Z2 = (z + 1) / 2;
    const size_t total = (size_t)n * X2 * Y2 * (Z2 + 1) * 8;
    pack_stem_cl_u8_kernel<<<grid_for(total, 256), 256, 0, (cudaStream_t)stream>>>(reinterpret_cast<const uint32_t*>(grid), n, x, y, z, X2, Y2, Z2,
                                                                                  reinterpret_cast<__nv_bfloat16*>(packed), act_fp16 ? 1 : 0);
    NRPN_LAUNCH_CHECK();
    return NRPN_OK;
}

int nrpn_maxpool3d_k3s2(const void* in, int n, int x, int y, int z, int c, void* out, int act_fp16, nrpn_stream_t stream) {
    if (!in || !out || n < 1 || x < 1 || y < 1 || z < 1 || c < 8 || c % 8 != 0) return NRPN_ERR_INVALID;
    const int Xo = (x - 1) / 2 + 1, Yo = (y - 1) / 2 + 1, Zo = (z - 1) / 2 + 1;
    const size_t total = (size_t)n * Xo * Yo * Zo * (c / 8);
    maxpool_k3s2_kernel<<<grid_for(total, 256), 256, 0, (cudaStream_t)stream>>>(
        reinterpret_cast<const __nv_bfloat16*>(in), n, x, y, z, c, Xo, Yo, Zo, reinterpret_cast<__nv_bfloat16*>(out), act_fp16 ? 1 : 0);
    NRPN_LAUNCH_CHECK();
    return NRPN_OK;
}

int nrpn_maxpool3d_k2s2_ceil(const void* in, int n, int x, int y, int z, int c, void* out, int act_fp16, nrpn_stream_t stream) {
    if (!in || !out || n < 1 || x < 1 || y < 1 || z < 1 || c < 8 || c % 8 != 0) return NRPN_ERR_INVALID;
    const int Xo = (x + 1) / 2, Yo = (y + 1) / 2, Zo = (z + 1) / 2;
    const size_t total = (size_t)n * Xo * Yo * Zo * (c / 8);
    maxpool_k2s2_ceil_kernel<<<grid_for(total, 256), 256, 0, (cudaStream_t)stream>>>(
        reinterpret_cast<const __nv_bfloat16*>(in), n, x, y, z, c, Xo, Yo, Zo, reinterpret_cast<__nv_bfloat16*>(out), act_fp16 ? 1 : 0);
    NRPN_LAUNCH_CHECK();
    return NRPN_OK;
}

int nrpn_pack_stem_input_s1(const float* grid, int n, int x, int y, int z, void* packed, int act_fp16, nrpn_stream_t stream) {
    if (!grid || !packed || n < 1 || x < 1 || y < 1 || z < 1) return NRPN_ERR_INVALID;
    const size_t total = (size_t)n * x * (y + 1) * z * 8;
    pack_stem_s1_kernel<<<grid_for(total, 256), 256, 0, (cudaStream_t)stream>>>(grid, n, x, y, z, reinterpret_cast<__nv_bfloat16*>(packed), act_fp16 ? 1 : 0);
    NRPN_LAUNCH_CHECK();
    return NRPN_OK;
}

int nrpn_version(void) { return 100; }

const char* nrpn_status_string(int status) {
    switch (status) {
        case NRPN_OK: return "ok";
        case NRPN_ERR_INVALID: return "invalid argument";
        case NRPN_ERR_UNSUPPORTED: return "unsupported shape";
        case NRPN_ERR_WORKSPACE: return "workspace too small";
        case NRPN_ERR_CUDA: return "CUDA error";
        case NRPN_ERR_NO_DEVICE: return "no sm_100 device / driver entry point";
        default: return "unknown status";
    }
}

int nrpn_last_cuda_error(void) { return g_last_cuda_error; }

unsigned long long nrpn_launch_count(void) { return g_launch_count.load(); }

#pragma GCC visibility pop
}  // extern "C"
