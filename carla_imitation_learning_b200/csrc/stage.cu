// K0: fused frame staging  rgb u8 (n,H,W,3) -> gray planes f32/bf16 (n,H,W).
// Replaces the per-sample numpy work of SequentialTorchDataset._load_file
// (/root/reference/src/dataset/imitation_dataset.py:120-121,130):
//     np.dot(images, [0.299, 0.587, 0.114]) / 255.0  ->  float32
// The kernel reproduces the numpy result bit for bit for ALL 2^24 (R,G,B) triples (see gray_px below;
// tests/test_gpu_parity.py::test_stage_gray_bit_exact_all_rgb proves it on the device, tests/test_stage_model.py
// on a host model of the same three f32 operations).
// HBM-bound: 3 B read + 4 B (f32) or 2 B (bf16) written per pixel; no reuse, so no smem.
#include "bc_common.cuh"

namespace {

// The reference evaluates (R*.299 + G*.587 + B*.114) / 255.0 in f64 and casts to f32. For every one of the 2^24 (R,G,B)
// triples that f32 value depends only on the integer s = 299R + 587G + 114B (<= 255000) and equals the CORRECTLY ROUNDED
// f32 quotient s / 255000 (the f64 chain's error, ~1e-16 relative, is far below the distance of any s/255000 to an f32
// rounding boundary: >= 1e-13 relative). A correctly rounded quotient needs no FP64: q0 = s*r, rem = fma(-q0, 255000, s)
// (exact), q = fma(rem, r, q0) with r = rn(1/255000) -- three f32 instructions, verified against numpy for all 247,023
// distinct s on the host and for all 2^24 triples on the device (tests/test_gpu_parity.py::test_stage_gray_bit_exact_all_rgb).
// (The first versions of this kernel ran the f64 chain itself and were FP64-pipe bound at 62 % of the HBM copy rate.)
__device__ __forceinline__ float gray_px(uint32_t r, uint32_t g, uint32_t b) {
    const float s = (float)(299u * r + 587u * g + 114u * b);          // exact: s < 2^24
    const float rcp = 1.0f / 255000.0f;
    const float q0 = __fmul_rn(s, rcp);
    const float rem = __fmaf_rn(-q0, 255000.0f, s);
    return __fmaf_rn(rem, rcp, q0);
}

// gray values of PX consecutive pixels (3 * PX bytes, 4 B aligned)
template <int PX>
__device__ __forceinline__ void gray_group(const uint32_t* __restrict__ src, float (&v)[PX]) {
    uint32_t w[3 * PX / 4];
#pragma unroll
    for (int i = 0; i < 3 * PX / 4; ++i) w[i] = __ldg(src + i);
#pragma unroll
    for (int p = 0; p < PX; ++p) {
        uint32_t c[3];
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            const int byte = 3 * p + k;
            c[k] = (w[byte >> 2] >> (8 * (byte & 3))) & 0xffu;
        }
        v[p] = gray_px(c[0], c[1], c[2]);
    }
}

// PX pixels per thread: 4 for f32 output (one 16 B store), 8 for bf16 output (one 16 B store).
template <int PX, typename TOUT>
__global__ void __launch_bounds__(256) stage_gray_kernel(const uint8_t* __restrict__ rgb,
                                                         TOUT* __restrict__ out, int64_t n_groups) {
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; g < n_groups; g += stride) {
        float v[PX];
        gray_group<PX>(reinterpret_cast<const uint32_t*>(rgb + g * (3 * PX)), v);
        if constexpr (sizeof(TOUT) == 4) {
            float4* dst = reinterpret_cast<float4*>(out + g * PX);
#pragma unroll
            for (int i = 0; i < PX / 4; ++i) dst[i] = make_float4(v[4 * i], v[4 * i + 1], v[4 * i + 2], v[4 * i + 3]);
        } else {
            uint32_t pk[PX / 2];
#pragma unroll
            for (int i = 0; i < PX / 2; ++i) {
                __nv_bfloat162 h = __floats2bfloat162_rn(v[2 * i], v[2 * i + 1]);
                pk[i] = *reinterpret_cast<uint32_t*>(&h);
            }
            uint4* dst = reinterpret_cast<uint4*>(out + g * PX);
#pragma unroll
            for (int i = 0; i < PX / 8; ++i) dst[i] = make_uint4(pk[4 * i], pk[4 * i + 1], pk[4 * i + 2], pk[4 * i + 3]);
        }
    }
}

// ---- "Toeplitz-ready" (TP) bf16 planes: the layout conv1's tcgen05 kernels consume without any repack.
// conv1 is a 7x7 stride-3 convolution evaluated as D[(oy,g),(j,co)] = sum A[(oy,g),(ci,ky,p)] * Wt (conv1_tc.cu):
// row (oy,g) of the A operand for kernel row ky is the 16-pixel segment [12g, 12g+16) of image row 3*oy+ky.
// A plane is therefore stored as  TP[c = R%3][h = half of the segment][q = R/3][g = 0..20][8 px]  (R = image
// row): for a fixed (c,h) consecutive (q,g) are 16 B apart, which IS the UMMA no-swizzle canonical layout
// (8 rows x 16 B core matrices, SBO 128 B; the two K halves of a row are one piece stride apart = LBO), both
// K-major (forward) and MN-major (wgrad). 1.32x the bytes of the plain plane (segments overlap by 4 px);
// rows R = 256, 257 (q = 85 of classes 1, 2) are zero.
constexpr int TP_NG = 21, TP_NQ = 86;

template <typename LOADER>
__device__ __forceinline__ void tp_write(LOADER&& load16, __nv_bfloat16* __restrict__ out, int64_t u) {
    const int g = (int)(u % TP_NG), q = (int)((u / TP_NG) % TP_NQ), c = (int)((u / (TP_NG * TP_NQ)) % 3);
    const int64_t plane = u / (TP_NG * TP_NQ * 3);
    const int R = 3 * q + c;
    uint32_t pk[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    if (R < BC_H) load16(plane, R, 12 * g, pk);
    __nv_bfloat16* dst = out + plane * BC_TP_PLANE_ELEMS + ((int64_t)(c * 2) * TP_NQ + q) * (TP_NG * 8) + g * 8;
    *reinterpret_cast<uint4*>(dst) = make_uint4(pk[0], pk[1], pk[2], pk[3]);
    *reinterpret_cast<uint4*>(dst + TP_NQ * TP_NG * 8) = make_uint4(pk[4], pk[5], pk[6], pk[7]);
}

__device__ __forceinline__ uint32_t pack_bf16(float a, float b) {
    __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
    return *reinterpret_cast<uint32_t*>(&h);
}

// Every pixel is converted ONCE: unit (R, g'), g' = 0..21, owns the 12 pixels [12g', 12g'+12) of image row R (g' = 21: the
// last 4) and writes them where they belong -- pixels 0..7 as the h=0 chunk and 8..11 as the first half of the h=1 chunk of
// segment g', pixels 0..3 also as the second half of the h=1 chunk of segment g'-1 (the 4-pixel overlap of neighbouring
// segments). Every pixel is converted once (12 conversions per thread, not 16).
// `plain` (optional): the same gray values also as plain (n,256,256) bf16 planes.
constexpr int TP_NU = TP_NG + 1;

// The bf16 value of a pixel, bf16_rn(f32 gray), needs less than the correctly rounded f32 quotient: s * r followed by one
// compensation step fma(s, r_lo, .) (r + r_lo = 1/255000 to 2^-48) lands on the same side of every bf16 rounding boundary as
// the exact quotient for all 247,023 distinct s (a single FMUL fails for s = 106333, 180791, 212666, 244541, which lie within
// 2^-25 of a bf16 midpoint) -- host-checked exhaustively (tests/test_stage_model.py) and on the device for all 2^24 triples
// (tests/test_gpu_parity.py). s itself is two dp4a over the pixel's bytes (R, G, B, G) gathered by ONE byte permute,
// 299 = 255 + 44, 587 = 255 + 255 + 77, 114 = 114, accumulated on top of the bit pattern of 2^23: the integer sum IS the float
// 2^23 + s, and one FADD makes it s (no I2F on the quarter-rate XU pipe, no shift / mask pairs). The first version of this
// kernel spent 25 instructions per pixel (11 of them 64-bit unit-index arithmetic) and was issue-bound at 42 % of the copy
// rate on the DRAM bytes it moves; this one spends about 10.
__device__ __forceinline__ float gray_px_bf16_exact(uint32_t px /* bytes R, G, B, G */) {
    uint32_t acc = __dp4a(px, 0xFF72FFFFu, 0x4B000000u);       // 255 R + 255 G + 114 B + 255 G + bits(2^23)
    acc = __dp4a(px, 0x00004D2Cu, acc);                        //  44 R +  77 G
    const float s = __uint_as_float(acc) - 8388608.0f;         // exact: s <= 255000 < 2^23
    constexpr float r = 1.0f / 255000.0f;
    constexpr float r_lo = (float)(1.0 / 255000.0 - (double)r);
    return __fmaf_rn(s, r_lo, __fmul_rn(s, r));
}

// The 12 gray values of TP unit (R, g') as bf16 pairs: src = the unit's first pixel (4 B aligned); g' = 21 has 4 pixels.
template <typename I>
__device__ __forceinline__ void tp_gray_unit(const uint32_t* __restrict__ src, I g, uint32_t (&pk)[6]) {
    uint32_t w[10];
#pragma unroll
    for (int i = 0; i < 9; ++i) w[i] = (g < TP_NG || i < 3) ? __ldg(src + i) : 0u;     // g' = 21 has 4 pixels = 12 bytes left
    w[9] = 0u;
    float v[12];
#pragma unroll
    for (int p = 0; p < 12; ++p) {
        constexpr uint32_t sel[4] = {0x1210u, 0x2321u, 0x3432u, 0x4543u};               // bytes o, o+1, o+2, o+1 = R, G, B, G
        const int o = (3 * p) & 3, i = (3 * p) >> 2;
        v[p] = gray_px_bf16_exact(__byte_perm(w[i], w[i + 1], sel[o]));
    }
#pragma unroll
    for (int i = 0; i < 6; ++i) pk[i] = pack_bf16(v[2 * i], v[2 * i + 1]);
}

// Where TP unit (R, g') goes: row0 = the plane's (c = R%3, h = 0, q = R/3) row; pixels 0..7 to segment g' h=0, 8..11 to the
// first half of its h=1 chunk, 0..3 also to the second half of segment g'-1's h=1 chunk.
template <typename I>
__device__ __forceinline__ void tp_store_unit(__nv_bfloat16* row0, I g, const uint32_t (&pk)[6]) {
    __nv_bfloat16* row1 = row0 + TP_NQ * TP_NG * 8;                                                             // (c, h=1, q)
    if (g < TP_NG) {
        *reinterpret_cast<uint4*>(row0 + g * 8) = make_uint4(pk[0], pk[1], pk[2], pk[3]);
        *reinterpret_cast<uint2*>(row1 + g * 8) = make_uint2(pk[4], pk[5]);
    }
    if (g > 0) *reinterpret_cast<uint2*>(row1 + (g - 1) * 8 + 4) = make_uint2(pk[0], pk[1]);
}

__global__ void __launch_bounds__(256) stage_gray_tp_kernel(const uint8_t* __restrict__ rgb, __nv_bfloat16* __restrict__ out,
                                                            __nv_bfloat16* __restrict__ plain, uint32_t n_units) {
    bc::pdl_wait();          // the previous step's kernels still read the planes this one overwrites
    bc::pdl_trigger();
    const uint32_t stride = gridDim.x * blockDim.x;
    for (uint32_t u = blockIdx.x * blockDim.x + threadIdx.x; u < n_units; u += stride) {      // 32-bit unit arithmetic
        const uint32_t t1 = u / TP_NU, g = u - t1 * TP_NU;
        const uint32_t t2 = t1 / TP_NQ, q = t1 - t2 * TP_NQ;
        const uint32_t plane = t2 / 3u, c = t2 - plane * 3u;
        const uint32_t R = 3u * q + c;
        uint32_t pk[6] = {0, 0, 0, 0, 0, 0};                 // 12 gray values as bf16 pairs; rows R >= 256 stay zero
        if (R < BC_H) {
            tp_gray_unit(reinterpret_cast<const uint32_t*>(rgb + ((size_t)plane * (BC_H * BC_W) + R * BC_W + 12u * g) * 3), g, pk);
            if (plain) {
                uint2* dst = reinterpret_cast<uint2*>(plain + ((size_t)plane * BC_H + R) * BC_W + 12u * g);
                dst[0] = make_uint2(pk[0], pk[1]);
                if (g < TP_NG) { dst[1] = make_uint2(pk[2], pk[3]); dst[2] = make_uint2(pk[4], pk[5]); }
            }
        }
        tp_store_unit(out + (size_t)plane * BC_TP_PLANE_ELEMS + ((c * 2u) * TP_NQ + q) * (TP_NG * 8), g, pk);
    }
}

// plain planes (f32 or bf16, rows contiguous, `plane_stride` elements apart) -> TP planes
template <typename TIN>
__global__ void __launch_bounds__(256) planes_to_tp_kernel(const TIN* __restrict__ in, int64_t plane_stride, __nv_bfloat16* __restrict__ out, int64_t n_units) {
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t u = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; u < n_units; u += stride)
        tp_write([&](int64_t plane, int R, int px0, uint32_t (&pk)[8]) {
            const TIN* src = in + plane * plane_stride + R * BC_W + px0;
            if constexpr (sizeof(TIN) == 4) {
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    const float4 f = __ldg(reinterpret_cast<const float4*>(src) + i);
                    pk[2 * i] = pack_bf16(f.x, f.y); pk[2 * i + 1] = pack_bf16(f.z, f.w);
                }
            } else {
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    const uint2 w = __ldg(reinterpret_cast<const uint2*>(src) + i);
                    pk[2 * i] = w.x; pk[2 * i + 1] = w.y;
                }
            }
        }, out, u);
}

// ---- EXTENSION (no counterpart in the reference; oracle/ext_oracle.py::stage_augmented): crop + colour jitter + normalise fused
// into the staging pass. Per frame one row of `table` = {crop_y, crop_x, brightness, contrast, saturation, mean, 1/std, -}
// (generated on the host from a seed: data.augment_table). Every step is a single-rounded f32 operation in the oracle's order
// (no FMA contraction), so the f32 output is bit-identical to the numpy specification and the bf16 output is its rounding.
struct AugRow { float cy, cx, br, ct, sa, mean, istd, pad; };
__device__ __forceinline__ float clamp255(float v) { return fminf(fmaxf(v, 0.f), 255.f); }
__device__ __forceinline__ float luma(float r, float g, float b) {
    return __fadd_rn(__fadd_rn(__fmul_rn(0.299f, r), __fmul_rn(0.587f, g)), __fmul_rn(0.114f, b));
}
__device__ __forceinline__ float aug_px(const uint8_t* __restrict__ px, const AugRow& t) {
    float c[3];
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        float v = clamp255(__fmul_rn((float)__ldg(px + k), t.br));
        c[k] = clamp255(__fadd_rn(__fmul_rn(__fadd_rn(v, -127.5f), t.ct), 127.5f));
    }
    const float y = luma(c[0], c[1], c[2]);
#pragma unroll
    for (int k = 0; k < 3; ++k) c[k] = clamp255(__fadd_rn(y, __fmul_rn(__fadd_rn(c[k], -y), t.sa)));
    const float g = __fmul_rn(luma(c[0], c[1], c[2]), 1.0f / 255.0f);
    return __fmul_rn(__fadd_rn(g, -t.mean), t.istd);
}

// The 12 augmented values of TP unit (R, g'): src = the unit's first source pixel; g' = 21 has 4 pixels (the rest are 0).
__device__ __forceinline__ void tp_aug_unit(const uint8_t* __restrict__ src, int g, const AugRow& t, float (&v)[12]) {
    const int npx = g < TP_NG ? 12 : 4;
#pragma unroll
    for (int p = 0; p < 12; ++p) v[p] = p < npx ? aug_px(src + 3 * p, t) : 0.f;
}

// 4 augmented values of one row: src = the first source pixel
__device__ __forceinline__ float4 aug4(const uint8_t* __restrict__ src, const AugRow& t) {
    float4 v;
    v.x = aug_px(src, t); v.y = aug_px(src + 3, t); v.z = aug_px(src + 6, t); v.w = aug_px(src + 9, t);
    return v;
}

// plain f32 planes (n,256,256): one thread = 4 pixels
__global__ void __launch_bounds__(256) stage_aug_f32_kernel(const uint8_t* __restrict__ rgb, int src_h, int src_w, const AugRow* __restrict__ table,
                                                            float* __restrict__ out, int64_t n_groups) {
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t u = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; u < n_groups; u += stride) {
        const int x4 = (int)(u % (BC_W / 4)), R = (int)((u / (BC_W / 4)) % BC_H);
        const int64_t plane = u / ((BC_W / 4) * BC_H);
        const AugRow t = table[plane];
        const uint8_t* src = rgb + ((plane * src_h + (int)t.cy + R) * (int64_t)src_w + (int)t.cx + 4 * x4) * 3;
        reinterpret_cast<float4*>(out)[u] = aug4(src, t);
    }
}

// Toeplitz-ready bf16 planes: the unit decomposition of stage_gray_tp_kernel (12 pixels per thread)
__global__ void __launch_bounds__(256) stage_aug_tp_kernel(const uint8_t* __restrict__ rgb, int src_h, int src_w, const AugRow* __restrict__ table,
                                                           __nv_bfloat16* __restrict__ out, int64_t n_units) {
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t u = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; u < n_units; u += stride) {
        const int g = (int)(u % TP_NU), q = (int)((u / TP_NU) % TP_NQ), c = (int)((u / (TP_NU * TP_NQ)) % 3);
        const int64_t plane = u / (TP_NU * TP_NQ * 3);
        const int R = 3 * q + c;
        uint32_t pk[6] = {0, 0, 0, 0, 0, 0};
        if (R < BC_H) {
            const AugRow t = table[plane];
            float v[12];
            tp_aug_unit(rgb + ((plane * src_h + (int)t.cy + R) * (int64_t)src_w + (int)t.cx + 12 * g) * 3, g, t, v);
#pragma unroll
            for (int i = 0; i < 6; ++i) pk[i] = pack_bf16(v[2 * i], v[2 * i + 1]);
        }
        tp_store_unit(out + plane * BC_TP_PLANE_ELEMS + ((int64_t)(c * 2) * TP_NQ + q) * (TP_NG * 8), g, pk);
    }
}

// ---- EXTENSION: per-agent frame history for closed-loop serving (bc_stage_history). Agent a owns 8 tick slots x `cams` planes,
// plane (a*8 + j)*cams + k. The frame of tick t goes to slot s = t mod 4 AND s + 4 (every slot on a reset), so the agent's 4-frame
// window is always the contiguous planes [(s+1)*cams, (s+5)*cams) and conv1 reads it with plain (stride_n, stride_c) =
// (8*cams, 1) planes. One unit = one destination piece of one frame, converted ONCE by the pixel code of the kernels above and
// stored 2 (or 8) times. PLANE = elements per plane; TP: one unit of stage_gray_tp_kernel / stage_aug_tp_kernel, else 4 pixels
// of one row as stage_gray_kernel<4, float> / stage_aug_f32_kernel convert them.
template <bool TP, bool AUG>
__global__ void __launch_bounds__(256) stage_history_kernel(const uint8_t* __restrict__ rgb, int src_h, int src_w,
                                                            const AugRow* __restrict__ table, const uint8_t* __restrict__ reset,
                                                            int reset_all, void* __restrict__ ring, int cams, int slot,
                                                            uint32_t n_units) {
    constexpr uint32_t UPF = TP ? 3u * TP_NQ * TP_NU : (uint32_t)(BC_H * BC_W / 4);     // units per frame
    constexpr int64_t PLANE = TP ? BC_TP_PLANE_ELEMS : BC_H * BC_W;
    const uint32_t stride = gridDim.x * blockDim.x;
    for (uint32_t u = blockIdx.x * blockDim.x + threadIdx.x; u < n_units; u += stride) {      // < 2^31: checked on the host
        const uint32_t row = u / UPF, w = u - row * UPF;             // row = a * cams + k of the frames (and of the table)
        const uint32_t a = row / (uint32_t)cams, k = row - a * (uint32_t)cams;
        const bool all = reset_all || (reset != nullptr && reset[a] != 0);
        int64_t off;                                                  // element offset of this unit inside a plane
        uint32_t pk[6] = {0, 0, 0, 0, 0, 0};
        float4 f;
        uint32_t g = 0;
        if constexpr (TP) {
            const uint32_t t1 = w / TP_NU, q = t1 % TP_NQ, c = t1 / TP_NQ, R = 3u * q + c;
            g = w - t1 * TP_NU;
            off = (int64_t)((c * 2u) * TP_NQ + q) * (TP_NG * 8);
            if (R < BC_H) {
                if constexpr (AUG) {
                    const AugRow t = table[row];
                    float v[12];
                    tp_aug_unit(rgb + (((int64_t)row * src_h + (int)t.cy + (int)R) * (int64_t)src_w + (int)t.cx + 12 * (int)g) * 3, (int)g, t, v);
#pragma unroll
                    for (int i = 0; i < 6; ++i) pk[i] = pack_bf16(v[2 * i], v[2 * i + 1]);
                } else {
                    tp_gray_unit(reinterpret_cast<const uint32_t*>(rgb + ((size_t)row * (BC_H * BC_W) + R * BC_W + 12u * g) * 3), g, pk);
                }
            }
        } else {
            off = (int64_t)w * 4;
            if constexpr (AUG) {
                const AugRow t = table[row];
                const int R = (int)(w / (BC_W / 4)), x4 = (int)(w % (BC_W / 4));
                f = aug4(rgb + (((int64_t)row * src_h + (int)t.cy + R) * (int64_t)src_w + (int)t.cx + 4 * x4) * 3, t);
            } else {
                float v[4];
                gray_group<4>(reinterpret_cast<const uint32_t*>(rgb + ((size_t)row * (BC_H * BC_W) + 4u * w) * 3), v);
                f = make_float4(v[0], v[1], v[2], v[3]);
            }
        }
        bc::pdl_wait();      // the previous tick's conv1 may still read the slot this unit overwrites
        bc::pdl_trigger();
        for (int j = all ? 0 : slot; j < 8; j += all ? 1 : 4) {
            const int64_t plane = ((int64_t)a * 8 + j) * cams + k;   // 64-bit: 4096 agents x 3 cameras x 8 slots of TP planes ~ 8.5e9 elements
            if constexpr (TP)
                tp_store_unit(reinterpret_cast<__nv_bfloat16*>(ring) + plane * PLANE + off, g, pk);
            else
                *reinterpret_cast<float4*>(reinterpret_cast<float*>(ring) + plane * PLANE + off) = f;
        }
    }
}

// ---- EXTENSION: shuffled minibatches from a device-resident frame store (bc_stage_gather). Sample b is the reference's sample
// i = index[b]: frames i .. i+3, side data of frame i+4. Output plane b*4*cams + cams*j + k = camera k of frame i+j (the channel
// order of sliding_window(step=cams), materialised). One unit = one piece of one output plane, in the unit decomposition of
// stage_history_kernel and converted by the same pixel code; every unit is stored once. A sample whose index lies outside
// [0, n_frames - 5] reads nothing and gets zero planes, zero side data and err_flag 5.
template <bool TP, bool AUG>
__global__ void __launch_bounds__(256) stage_gather_kernel(bc_frame_store s, const int64_t* __restrict__ index, int batch,
                                                           const AugRow* __restrict__ table, void* __restrict__ out,
                                                           int64_t* __restrict__ y, int64_t* __restrict__ command,
                                                           float* __restrict__ target, int32_t* __restrict__ err_flag,
                                                           uint32_t n_units) {
    constexpr uint32_t UPF = TP ? 3u * TP_NQ * TP_NU : (uint32_t)(BC_H * BC_W / 4);     // units per plane
    constexpr int64_t PLANE = TP ? BC_TP_PLANE_ELEMS : BC_H * BC_W;
    const uint32_t cams = (uint32_t)s.cams, pps = 4u * cams;                             // planes per sample
    const int64_t last = s.n_frames - 5;
    const uint32_t tid = blockIdx.x * blockDim.x + threadIdx.x, stride = gridDim.x * blockDim.x;
    for (uint32_t u = tid; u < n_units; u += stride) {                // < 2^31: checked on the host
        const uint32_t p = u / UPF, w = u - p * UPF;                  // output plane p
        const uint32_t b = p / pps, r = p - b * pps, j = r / cams, k = r - j * cams;
        const int64_t i = __ldg(index + b);
        const bool ok = i >= 0 && i <= last;
        const int64_t row = (i + j) * cams + k;                       // store row (64-bit: a store is tens of GB)
        int64_t off;
        uint32_t pk[6] = {0, 0, 0, 0, 0, 0};
        float4 f = make_float4(0.f, 0.f, 0.f, 0.f);
        uint32_t g = 0;
        if constexpr (TP) {
            const uint32_t t1 = w / TP_NU, q = t1 % TP_NQ, c = t1 / TP_NQ, R = 3u * q + c;
            g = w - t1 * TP_NU;
            off = (int64_t)((c * 2u) * TP_NQ + q) * (TP_NG * 8);
            if (ok && R < BC_H) {
                if constexpr (AUG) {
                    const AugRow t = table[b * cams + k];
                    float v[12];
                    tp_aug_unit(s.frames + ((row * s.src_h + (int)t.cy + (int)R) * (int64_t)s.src_w + (int)t.cx + 12 * (int)g) * 3, (int)g, t, v);
#pragma unroll
                    for (int m = 0; m < 6; ++m) pk[m] = pack_bf16(v[2 * m], v[2 * m + 1]);
                } else {
                    tp_gray_unit(reinterpret_cast<const uint32_t*>(s.frames + (row * (BC_H * BC_W) + R * BC_W + 12u * g) * 3), g, pk);
                }
            }
        } else {
            off = (int64_t)w * 4;
            if (ok) {
                if constexpr (AUG) {
                    const AugRow t = table[b * cams + k];
                    const int R = (int)(w / (BC_W / 4)), x4 = (int)(w % (BC_W / 4));
                    f = aug4(s.frames + ((row * s.src_h + (int)t.cy + R) * (int64_t)s.src_w + (int)t.cx + 4 * x4) * 3, t);
                } else {
                    float v[4];
                    gray_group<4>(reinterpret_cast<const uint32_t*>(s.frames + (row * (BC_H * BC_W) + 4u * w) * 3), v);
                    f = make_float4(v[0], v[1], v[2], v[3]);
                }
            }
        }
        bc::pdl_wait();      // the previous step's conv1 (forward and weight gradient) may still read the planes this unit overwrites
        bc::pdl_trigger();
        if constexpr (TP)
            tp_store_unit(reinterpret_cast<__nv_bfloat16*>(out) + (int64_t)p * PLANE + off, g, pk);
        else
            *reinterpret_cast<float4*>(reinterpret_cast<float*>(out) + (int64_t)p * PLANE + off) = f;
    }
    // side data of frame i+4, in the same launch: the previous step's head may still read these buffers
    bc::pdl_wait();
    for (uint32_t b = tid; b < (uint32_t)batch; b += stride) {
        const int64_t i = __ldg(index + b);
        const bool ok = i >= 0 && i <= last;
        if (!ok) atomicCAS(err_flag, 0, 5);                        // never masks an error code already set
        if (y && s.labels) y[b] = ok ? __ldg(s.labels + i + 4) : 0;
        if (command && s.commands) command[b] = ok ? __ldg(s.commands + i + 4) : 0;
        if (target && s.targets)
            for (int o = 0; o < s.n_out; ++o) target[(int64_t)b * s.n_out + o] = ok ? __ldg(s.targets + (i + 4) * s.n_out + o) : 0.f;
    }
}

}  // namespace

extern "C" int bc_stage_augment(const uint8_t* rgb, int64_t n_frames, int src_h, int src_w, const float* table, void* out, int out_dtype, void* stream) {
    BC_CHECK_ARG(rgb && table && out && n_frames >= 0, "bc_stage_augment: null pointer");
    BC_CHECK_ARG(src_h >= BC_H && src_w >= BC_W, "bc_stage_augment: source frames %dx%d are smaller than the %dx%d crop", src_h, src_w, BC_H, BC_W);
    BC_CHECK_ARG(out_dtype == BC_F32 || out_dtype == BC_BF16_TP, "bc_stage_augment: output is BC_F32 planes or BC_BF16_TP planes, got %d", out_dtype);
    BC_CHECK_ARG((uintptr_t)out % 16 == 0 && (uintptr_t)table % 16 == 0, "bc_stage_augment: out and table must be 16 B aligned");
    if (n_frames == 0) return BC_OK;
    const int64_t cap = (int64_t)bc::num_sms() * 16;
    if (out_dtype == BC_F32) {
        const int64_t groups = n_frames * BC_H * (BC_W / 4);
        const int blocks = (int)((groups + 255) / 256 < cap ? (groups + 255) / 256 : cap);
        stage_aug_f32_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(rgb, src_h, src_w, (const AugRow*)table, (float*)out, groups);
    } else {
        const int64_t units = n_frames * 3 * TP_NQ * TP_NU;
        const int blocks = (int)((units + 255) / 256 < cap ? (units + 255) / 256 : cap);
        stage_aug_tp_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(rgb, src_h, src_w, (const AugRow*)table, (__nv_bfloat16*)out, units);
    }
    BC_CUDA_LAUNCH_CHECK("stage_aug_kernel");
    return BC_OK;
}

extern "C" int bc_planes_to_tp(const void* planes, int in_dtype, int64_t n_planes, int64_t plane_stride, void* out_tp, void* stream) {
    BC_CHECK_ARG(planes && out_tp && n_planes >= 0, "bc_planes_to_tp: null pointer");
    BC_CHECK_ARG(in_dtype == BC_F32 || in_dtype == BC_BF16, "bc_planes_to_tp: planes are f32 or bf16, got dtype %d", in_dtype);
    const int esz = in_dtype == BC_F32 ? 4 : 2;
    BC_CHECK_ARG((uintptr_t)planes % 16 == 0 && (plane_stride * esz) % 16 == 0 && (uintptr_t)out_tp % 16 == 0, "bc_planes_to_tp: 16 B alignment");
    if (n_planes == 0) return BC_OK;
    const int64_t units = n_planes * 3 * TP_NQ * TP_NG;
    int64_t blocks = (units + 255) / 256;
    const int64_t cap = (int64_t)bc::num_sms() * 16;
    if (blocks > cap) blocks = cap;
    if (in_dtype == BC_F32)
        planes_to_tp_kernel<float><<<(int)blocks, 256, 0, (cudaStream_t)stream>>>((const float*)planes, plane_stride, (__nv_bfloat16*)out_tp, units);
    else
        planes_to_tp_kernel<__nv_bfloat16><<<(int)blocks, 256, 0, (cudaStream_t)stream>>>((const __nv_bfloat16*)planes, plane_stride, (__nv_bfloat16*)out_tp, units);
    BC_CUDA_LAUNCH_CHECK("planes_to_tp_kernel");
    return BC_OK;
}

extern "C" int bc_stage_gray_tp(const uint8_t* rgb, void* tp, void* plain_bf16, int64_t n_frames, void* stream) {
    BC_CHECK_ARG(rgb && tp && n_frames >= 0, "bc_stage_gray_tp: null pointer");
    BC_CHECK_ARG(((uintptr_t)rgb % 4 == 0) && ((uintptr_t)tp % 16 == 0) && ((uintptr_t)plain_bf16 % 8 == 0), "bc_stage_gray_tp: alignment");
    if (n_frames == 0) return BC_OK;
    const int64_t units = n_frames * 3 * TP_NQ * TP_NU;
    BC_CHECK_ARG(units < (int64_t)0x7fffffff - 0x1000000, "bc_stage_gray_tp: %lld frames in one call (the unit index is 32-bit: at most 378,000)", (long long)n_frames);
    const int64_t cap = (int64_t)bc::num_sms() * 16;
    const int blocks = (int)((units + 255) / 256 < cap ? (units + 255) / 256 : cap);
    bc::launch_pdl(stage_gray_tp_kernel, dim3(blocks), dim3(256), 0, (cudaStream_t)stream, rgb, (__nv_bfloat16*)tp, (__nv_bfloat16*)plain_bf16, (uint32_t)units);
    BC_CUDA_LAUNCH_CHECK("stage_gray_tp_kernel");
    return BC_OK;
}

extern "C" int bc_stage_gray(const uint8_t* rgb, void* gray, int64_t n_pixels, int out_dtype, void* stream) {
    BC_CHECK_ARG(rgb && gray, "bc_stage_gray: null pointer");
    BC_CHECK_ARG(n_pixels >= 0 && n_pixels % 8 == 0, "bc_stage_gray: n_pixels=%lld must be a multiple of 8", (long long)n_pixels);
    BC_CHECK_ARG(((uintptr_t)rgb % 4 == 0) && ((uintptr_t)gray % 16 == 0), "bc_stage_gray: rgb must be 4 B and gray 16 B aligned");
    BC_CHECK_ARG(out_dtype == BC_F32 || out_dtype == BC_BF16 || out_dtype == BC_BF16_TP, "bc_stage_gray: bad dtype %d", out_dtype);
    if (n_pixels == 0) return BC_OK;
    cudaStream_t s = (cudaStream_t)stream;
    const int sms = bc::num_sms();
    if (out_dtype == BC_BF16_TP) {
        BC_CHECK_ARG(n_pixels % (BC_H * BC_W) == 0, "bc_stage_gray: the TP layout is defined for whole 256x256 frames");
        const int64_t units = n_pixels / (BC_H * BC_W) * 3 * TP_NQ * TP_NU;
        BC_CHECK_ARG(units < (int64_t)0x7fffffff - 0x1000000, "bc_stage_gray: too many frames in one call for the TP layout (32-bit unit index: at most 378,000)");
        int blocks = (int)((units + 255) / 256 < (int64_t)sms * 16 ? (units + 255) / 256 : (int64_t)sms * 16);
        stage_gray_tp_kernel<<<blocks, 256, 0, s>>>(rgb, (__nv_bfloat16*)gray, nullptr, (uint32_t)units);
    } else if (out_dtype == BC_F32) {
        int64_t groups = n_pixels / 4;
        int blocks = (int)((groups + 255) / 256 < (int64_t)sms * 16 ? (groups + 255) / 256 : (int64_t)sms * 16);
        stage_gray_kernel<4, float><<<blocks, 256, 0, s>>>(rgb, (float*)gray, groups);
    } else {
        int64_t groups = n_pixels / 8;
        int blocks = (int)((groups + 255) / 256 < (int64_t)sms * 16 ? (groups + 255) / 256 : (int64_t)sms * 16);
        stage_gray_kernel<8, __nv_bfloat16><<<blocks, 256, 0, s>>>(rgb, (__nv_bfloat16*)gray, groups);
    }
    BC_CUDA_LAUNCH_CHECK("stage_gray_kernel");
    return BC_OK;
}

extern "C" int bc_stage_history(const uint8_t* rgb, int n_agents, int cams, int src_h, int src_w, const float* table,
                                const uint8_t* reset, int reset_all, void* ring, int slot, int out_dtype, void* stream) {
    BC_CHECK_ARG(rgb && ring, "bc_stage_history: null pointer (rgb, ring)");
    BC_CHECK_ARG(n_agents >= 1, "bc_stage_history: n_agents=%d must be at least 1", n_agents);
    BC_CHECK_ARG(cams == 1 || cams == 3, "bc_stage_history: cams=%d must be 1 or 3 (obs_size 4 or 12)", cams);
    BC_CHECK_ARG(slot >= 0 && slot < 4, "bc_stage_history: slot=%d must lie in [0, 4) (tick mod 4)", slot);
    BC_CHECK_ARG(src_h >= BC_H && src_w >= BC_W, "bc_stage_history: source frames %dx%d are smaller than %dx%d", src_h, src_w, BC_H, BC_W);
    BC_CHECK_ARG(table || (src_h == BC_H && src_w == BC_W), "bc_stage_history: %dx%d sources need a crop table", src_h, src_w);
    BC_CHECK_ARG(out_dtype == BC_F32 || out_dtype == BC_BF16_TP, "bc_stage_history: the ring holds BC_F32 or BC_BF16_TP planes, got %d", out_dtype);
    BC_CHECK_ARG((uintptr_t)ring % 16 == 0 && (uintptr_t)table % 16 == 0, "bc_stage_history: ring and table must be 16 B aligned");
    BC_CHECK_ARG(table || (uintptr_t)rgb % 4 == 0, "bc_stage_history: rgb must be 4 B aligned");
    const bool tp = out_dtype == BC_BF16_TP;
    const int64_t units = (int64_t)n_agents * cams * (tp ? 3 * TP_NQ * TP_NU : BC_H * BC_W / 4);
    BC_CHECK_ARG(units < (int64_t)0x7fffffff - 0x1000000, "bc_stage_history: %d agents x %d cameras in one call (32-bit unit index)", n_agents, cams);
    const int64_t cap = (int64_t)bc::num_sms() * 16;
    const int blocks = (int)((units + 255) / 256 < cap ? (units + 255) / 256 : cap);
    const AugRow* t = (const AugRow*)table;
    cudaStream_t s = (cudaStream_t)stream;
    if (tp && table)
        bc::launch_pdl(stage_history_kernel<true, true>, dim3(blocks), dim3(256), 0, s, rgb, src_h, src_w, t, reset, reset_all, ring, cams, slot, (uint32_t)units);
    else if (tp)
        bc::launch_pdl(stage_history_kernel<true, false>, dim3(blocks), dim3(256), 0, s, rgb, src_h, src_w, t, reset, reset_all, ring, cams, slot, (uint32_t)units);
    else if (table)
        bc::launch_pdl(stage_history_kernel<false, true>, dim3(blocks), dim3(256), 0, s, rgb, src_h, src_w, t, reset, reset_all, ring, cams, slot, (uint32_t)units);
    else
        bc::launch_pdl(stage_history_kernel<false, false>, dim3(blocks), dim3(256), 0, s, rgb, src_h, src_w, t, reset, reset_all, ring, cams, slot, (uint32_t)units);
    BC_CUDA_LAUNCH_CHECK("stage_history_kernel");
    return BC_OK;
}

extern "C" int bc_stage_gather(const bc_frame_store* st, const int64_t* index, int batch, const float* table, void* out,
                               int out_dtype, int64_t* y, int64_t* command, float* target, int32_t* err_flag, void* stream) {
    BC_CHECK_ARG(st && st->frames && index && out && err_flag, "bc_stage_gather: null pointer (store, frames, index, out, err_flag)");
    BC_CHECK_ARG(batch >= 1, "bc_stage_gather: batch=%d must be at least 1", batch);
    BC_CHECK_ARG(st->cams == 1 || st->cams == 3, "bc_stage_gather: cams=%d must be 1 or 3 (obs_size 4 or 12)", st->cams);
    BC_CHECK_ARG(st->n_frames >= 5, "bc_stage_gather: n_frames=%lld: a store holds at least 5 time steps (one window and its label)", (long long)st->n_frames);
    BC_CHECK_ARG(st->src_h >= BC_H && st->src_w >= BC_W, "bc_stage_gather: source frames %dx%d are smaller than %dx%d", st->src_h, st->src_w, BC_H, BC_W);
    BC_CHECK_ARG(table || (st->src_h == BC_H && st->src_w == BC_W), "bc_stage_gather: %dx%d sources need a crop table", st->src_h, st->src_w);
    BC_CHECK_ARG(out_dtype == BC_F32 || out_dtype == BC_BF16_TP, "bc_stage_gather: the output is BC_F32 or BC_BF16_TP planes, got %d", out_dtype);
    BC_CHECK_ARG((uintptr_t)out % 16 == 0 && (uintptr_t)table % 16 == 0, "bc_stage_gather: out and table must be 16 B aligned");
    BC_CHECK_ARG((uintptr_t)index % 8 == 0 && (uintptr_t)st->labels % 8 == 0 && (uintptr_t)st->commands % 8 == 0
                 && (uintptr_t)st->targets % 4 == 0 && (uintptr_t)y % 8 == 0 && (uintptr_t)command % 8 == 0 && (uintptr_t)target % 4 == 0,
                 "bc_stage_gather: index, labels, commands, y, command must be 8 B and targets, target 4 B aligned");
    BC_CHECK_ARG(table || (uintptr_t)st->frames % 4 == 0, "bc_stage_gather: frames must be 4 B aligned");
    BC_CHECK_ARG(!(st->targets && target) || st->n_out >= 1, "bc_stage_gather: n_out=%d must be at least 1 with targets", st->n_out);
    const bool tp = out_dtype == BC_BF16_TP;
    const int64_t units = (int64_t)batch * 4 * st->cams * (tp ? 3 * TP_NQ * TP_NU : BC_H * BC_W / 4);
    BC_CHECK_ARG(units < (int64_t)0x7fffffff - 0x1000000, "bc_stage_gather: batch %d x %d cameras in one call (32-bit unit index)", batch, st->cams);
    const int64_t cap = (int64_t)bc::num_sms() * 16;
    const int blocks = (int)((units + 255) / 256 < cap ? (units + 255) / 256 : cap);
    const AugRow* t = (const AugRow*)table;
    cudaStream_t s = (cudaStream_t)stream;
    if (tp && table)
        bc::launch_pdl(stage_gather_kernel<true, true>, dim3(blocks), dim3(256), 0, s, *st, index, batch, t, out, y, command, target, err_flag, (uint32_t)units);
    else if (tp)
        bc::launch_pdl(stage_gather_kernel<true, false>, dim3(blocks), dim3(256), 0, s, *st, index, batch, t, out, y, command, target, err_flag, (uint32_t)units);
    else if (table)
        bc::launch_pdl(stage_gather_kernel<false, true>, dim3(blocks), dim3(256), 0, s, *st, index, batch, t, out, y, command, target, err_flag, (uint32_t)units);
    else
        bc::launch_pdl(stage_gather_kernel<false, false>, dim3(blocks), dim3(256), 0, s, *st, index, batch, t, out, y, command, target, err_flag, (uint32_t)units);
    BC_CUDA_LAUNCH_CHECK("stage_gather_kernel");
    return BC_OK;
}
