// K13: the tail of the policy forward for closed-loop serving at small batch, ONE launch:
//   conv4x4(32->64)+ReLU+pool2 -> conv3x3(64->128)+ReLU+pool2 -> flatten -> fc 128->64->32->n_actions -> greedy action
// = ConvNet1.cnn_base[6:12] + fc (/root/reference/src/architectures/nets.py:24-33,35-39) and the argmax of
// Imitation.forward's logits the rollout code takes (/root/reference/src/data/stat.py:41). At batch 1..16 the forward is a
// chain of launch latencies (BASELINE configs[4]: 7 dependent launches = 27.5 us at B = 1 with every launch under programmatic
// dependent launch); conv3, conv4, the head and the argmax are 5.9 MFLOP per sample -- this kernel replaces those four
// launches by one.
//
// One thread-block CLUSTER of 8 CTAs per sample, exact f32 FFMA arithmetic on the f32 master weights (both modes):
//   phase A (before griddepcontrol.wait: the parameters are written only by launches that release their dependents after their
//            last write, include/bc_b200.h "Launch ordering contract"): CTA r loads its weight slices into shared memory --
//            conv3 output channels [8r, 8r+8) (16 KB), conv4 output channels [16r, 16r+16) (36 KB), CTA 0 also the head (42 KB);
//   phase B  act2 of the sample (32x12x12 f32, 18 KB) -> shared memory; conv3 for the CTA's 8 channels at the 8x8 conv pixels
//            the floor-mode pool keeps (row / column 8 of the 9x9 output is dropped by MaxPool2d(2), nets.py:26): a thread owns
//            (2 channels, the 2 x 8 conv pixels of one pooled row, 2 of the 32 input channels) = 1,024 FMA on 5 input rows and
//            32 weights held in registers (23 LDS.128 per 512 FMA; the phase is FMA-issue bound at 2 warps per scheduler: a first
//            version with 4x the shared-memory loads took the same 3.0 K cycles); the 16 input-channel pairs meet in shared memory in fixed order, + bias, ReLU, 2x2 max; after a
//            cluster barrier every CTA pulls the other seven CTAs' 128 pooled values through distributed shared memory;
//   phase C  conv4 for the CTA's 16 channels: a thread owns (channel, 4 of the 64 input channels) for all 2x2 conv pixels,
//            16-lane xor tree, + bias, ReLU, max -> the 16 features go to CTA 0's shared memory;
//   phase D  CTA 0: the three Linear layers on all 256 threads (rows split over neighbouring lanes), logits, greedy action
//            (torch.argmax's rule: the first NaN, else the first maximum).
// Two cluster barriers per sample; no global-memory round trip between the layers.
//
// The branched instantiation (bc_policy_tail_branched) serves ConvNet1Branched: the G heads have the single head's shapes and
// padded order [fc.4 | fc.2 | fc.0] (head_branched.cu), so the shared-memory plan and phases B..D are the same. Only CTA 0's
// head load differs: it reads command[b] (before griddepcontrol.wait, like the weights: nothing in this library writes the
// command vector, include/bc_b200.h launch ordering) and loads branch command[b]'s fc.0, fc.2, fc.4 from the branch arena.
// A command outside [0, G) loads branch 0 (the address is clamped before any load), raises flag 4 and leaves a zero output
// row and action 0, as head_branched_kernel does.
#include "bc_common.cuh"
#include "trace.cuh"
#include <cooperative_groups.h>

namespace cg = cooperative_groups;

namespace {

constexpr int CL = 8;                 // CTAs per sample = cluster size (portable maximum)
constexpr int NT = 256;
constexpr int MAXA = BC_MAX_ACTIONS;
constexpr int A3P = 20;               // floats between two channels of the pooled conv3 activation in shared memory (16 used):
                                      // 80 B pitch makes the 16 B patch loads of conv4 conflict-free

// shared-memory plan (floats)
constexpr int W3P = 8 * 32 * 16 / 8 + 4;      // floats between two conv3 output channels in shared memory (512 used): the four
                                              // channel pairs a quarter-warp reads with one LDS.128 fall into disjoint banks
constexpr int PTP = 36;                       // floats between two threads' partial tiles (32 used): conflict-free STS.128
constexpr int O_W3 = 0;                       // [8][W3P]  = [co][ci][ky][kx]
constexpr int W4P = 64 * 9 + 16;              // floats between two conv4 output channels (576 used): the two channels of a warp read disjoint banks
constexpr int O_W4 = O_W3 + 8 * W3P;          // [16][W4P] = [co][ci][ky][kx]
constexpr int O_A2 = O_W4 + 16 * W4P;         // [32][12][12]
constexpr int O_PART = O_A2 + 32 * 144;       // [16 input-channel pairs][16 (pooled row, channel pair)][PTP]
constexpr int O_A3 = O_PART + 16 * 16 * PTP;   // [64][A3P]
constexpr int O_A4 = O_A3 + 64 * A3P;         // [128]
constexpr int O_B3 = O_A4 + 128;              // [8]
constexpr int O_B4 = O_B3 + 8;                // [16]
constexpr int O_HW0 = O_B4 + 16;              // head, CTA 0 only: fc.0 [64][128]
constexpr int O_HW2 = O_HW0 + 64 * 128;       // fc.2 [32][64]
constexpr int O_HW4 = O_HW2 + 32 * 64;        // fc.4 [MAXA][32]
constexpr int O_HB0 = O_HW4 + MAXA * 32;
constexpr int O_HB2 = O_HB0 + 64;
constexpr int O_HB4 = O_HB2 + 32;
constexpr int O_H1 = O_HB4 + MAXA;
constexpr int O_H2 = O_H1 + 64;
constexpr int O_Z = O_H2 + 32;
constexpr int SMEM_FLOATS = O_Z + MAXA;
constexpr int SMEM_BYTES = SMEM_FLOATS * 4;
static_assert(O_A4 % 4 == 0 && O_H1 % 4 == 0 && W3P % 4 == 0 && W4P % 4 == 0 && O_W4 % 4 == 0 && O_A2 % 4 == 0 && O_PART % 4 == 0 && O_A3 % 4 == 0 && O_HW0 % 4 == 0 && O_HW2 % 4 == 0 && O_HW4 % 4 == 0,
              "16 B alignment of the vector-accessed regions");

struct TailArgs {
    const float* act2;                                  // (B,32,12,12) f32: pooled output of conv2 (bc_ctx.act[1])
    const float* w3; const float* b3;                   // cnn_base.6: (64,32,4,4), (64)
    const float* w4; const float* b4;                   // cnn_base.9: (128,64,3,3), (128)
    const float* f0; const float* g0; const float* f2; const float* g2; const float* f4; const float* g4;   // fc.{0,2,4} weight, bias
    float* act3; float* act4; float* hid1; float* hid2; // optional outputs (B,64,4,4) (B,128) (B,64) (B,32)
    float* logits; int64_t* actions;                    // (B,NA), (B)
    int B, NA;
};

struct BranchArgs {                                     // the branched instantiation only
    const int64_t* cmd;                                 // (B,) branch ids
    const float* barena;                                // G x head_len floats, per branch [fc.4 w,b | fc.2 w,b | fc.0 w,b]
    int64_t head_len, w0, b0, w2, b2, w4, b4;           // bc_head_branched_layout
    int G;
    int* err;                                           // flag 4 = command outside [0, G)
};

template <bool kBranched>
__global__ void __launch_bounds__(NT, 1) policy_tail_kernel(const TailArgs a, const BranchArgs br) {
    extern __shared__ __align__(16) float sm[];
    cg::cluster_group cluster = cg::this_cluster();
    const int r = (int)cluster.block_rank();
    const int b = blockIdx.x / CL;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int NA = a.NA;
    bool cmd_ok = true;                  // branched: command[b] in [0, G) (read by CTA 0, which alone writes outputs from it)
    TRACE_T0
    TRACE_DECL
    TRACE(0, 0);

    // every CTA of the cluster has started once this barrier completes (waited on before the first remote store)
    (void)cluster.barrier_arrive();

    // ---- phase A: weight slices (L2 loads: an L1 line of an earlier launch on this SM could be stale) -----------------
    {
        const float4* src3 = reinterpret_cast<const float4*>(a.w3 + (size_t)r * (8 * 32 * 16));
        float4 t3[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) t3[q] = __ldcg(src3 + tid + NT * q);
        const float4* src4 = reinterpret_cast<const float4*>(a.w4 + (size_t)r * (16 * 64 * 9));
        float4 t4[9];
#pragma unroll
        for (int q = 0; q < 9; ++q) t4[q] = __ldcg(src4 + tid + NT * q);
#pragma unroll
        for (int q = 0; q < 4; ++q) {                      // float4 index i = co * 128 + rest -> co * (W3P / 4) + rest
            const int i = tid + NT * q;
            reinterpret_cast<float4*>(sm + O_W3)[(i >> 7) * (W3P / 4) + (i & 127)] = t3[q];
        }
#pragma unroll
        for (int q = 0; q < 9; ++q) {                      // float4 index i = co * 144 + rest -> co * (W4P / 4) + rest
            const int i = tid + NT * q;
            reinterpret_cast<float4*>(sm + O_W4)[(i / 144) * (W4P / 4) + (i % 144)] = t4[q];
        }
        if (tid < 8) sm[O_B3 + tid] = __ldcg(a.b3 + 8 * r + tid);
        if (tid < 16) sm[O_B4 + tid] = __ldcg(a.b4 + 16 * r + tid);
    }
    if (r == 0) {
        const float *f0 = a.f0, *g0 = a.g0, *f2 = a.f2, *g2 = a.g2, *f4 = a.f4, *g4 = a.g4;
        if constexpr (kBranched) {       // the commanded branch: clamped to branch 0 before any load of its weights
            const int64_t cmd = __ldcg(br.cmd + b);
            cmd_ok = cmd >= 0 && cmd < br.G;
            const float* P = br.barena + (cmd_ok ? cmd : 0) * br.head_len;
            f0 = P + br.w0; g0 = P + br.b0; f2 = P + br.w2; g2 = P + br.b2; f4 = P + br.w4; g4 = P + br.b4;
        }
        const float4* w0v = reinterpret_cast<const float4*>(f0);
        float4 t[8];
#pragma unroll
        for (int q = 0; q < 8; ++q) t[q] = __ldcg(w0v + tid + NT * q);
        const float4* w2v = reinterpret_cast<const float4*>(f2);
        const float4 u0 = __ldcg(w2v + tid), u1 = __ldcg(w2v + tid + NT);
        const bool has4 = tid < NA * 8;
        const float4 u4 = has4 ? __ldcg(reinterpret_cast<const float4*>(f4) + tid) : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
        for (int q = 0; q < 8; ++q) reinterpret_cast<float4*>(sm + O_HW0)[tid + NT * q] = t[q];
        reinterpret_cast<float4*>(sm + O_HW2)[tid] = u0;
        reinterpret_cast<float4*>(sm + O_HW2)[tid + NT] = u1;
        if (has4) reinterpret_cast<float4*>(sm + O_HW4)[tid] = u4;
        if (tid < 64) sm[O_HB0 + tid] = __ldcg(g0 + tid);
        if (tid < 32) sm[O_HB2 + tid] = __ldcg(g2 + tid);
        if (tid < NA) sm[O_HB4 + tid] = __ldcg(g4 + tid);
    }
    TRACE(1, 0);
    bc::pdl_wait();                      // act2 is the previous launch's output
    bc::pdl_trigger();
    TRACE(2, 0);

    // ---- phase B: conv3 + ReLU + pool -------------------------------------------------------------------------------------
    {
        const float4* src = reinterpret_cast<const float4*>(a.act2 + (size_t)b * (32 * 144));
        float4 t[5];
#pragma unroll
        for (int q = 0; q < 5; ++q) { const int i = tid + NT * q; t[q] = i < 1152 ? __ldcg(src + i) : make_float4(0.f, 0.f, 0.f, 0.f); }
#pragma unroll
        for (int q = 0; q < 5; ++q) { const int i = tid + NT * q; if (i < 1152) reinterpret_cast<float4*>(sm + O_A2)[i] = t[q]; }
    }
    __syncthreads();
    TRACE(3, 0);
    {
        // lane = channel pair + 4 * pooled row + 16 * (input-channel pair & 1), warp = input-channel pair >> 1: a quarter-warp reads
        // 2 distinct input rows and 4 distinct weight rows per LDS.128, all in disjoint banks; everything else is a broadcast
        const int cp = tid & 3, py = (tid >> 2) & 3, cs = 2 * warp + (lane >> 4);
        float acc[2][2][8];
#pragma unroll
        for (int h = 0; h < 2; ++h)
#pragma unroll
            for (int dy = 0; dy < 2; ++dy)
#pragma unroll
                for (int ox = 0; ox < 8; ++ox) acc[h][dy][ox] = 0.f;
#pragma unroll
        for (int i = 0; i < 2; ++i) {
            const int ci = 2 * cs + i;
            const float4* ap = reinterpret_cast<const float4*>(sm + O_A2 + ci * 144 + (2 * py) * 12);   // input rows 2py .. 2py+4, 12 columns
            float in[5][12];
#pragma unroll
            for (int rr = 0; rr < 5; ++rr) {
#pragma unroll
                for (int j = 0; j < 3; ++j) {
                    const float4 v = ap[rr * 3 + j];
                    in[rr][4 * j] = v.x; in[rr][4 * j + 1] = v.y; in[rr][4 * j + 2] = v.z; in[rr][4 * j + 3] = v.w;
                }
            }
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                const float4* wv = reinterpret_cast<const float4*>(sm + O_W3 + (2 * cp + h) * W3P + ci * 16);
#pragma unroll
                for (int ky = 0; ky < 4; ++ky) {
                    const float4 w = wv[ky];
#pragma unroll
                    for (int dy = 0; dy < 2; ++dy) {
#pragma unroll
                        for (int ox = 0; ox < 8; ++ox) {
                            float t = acc[h][dy][ox];
                            t = fmaf(w.x, in[dy + ky][ox], t); t = fmaf(w.y, in[dy + ky][ox + 1], t);
                            t = fmaf(w.z, in[dy + ky][ox + 2], t); t = fmaf(w.w, in[dy + ky][ox + 3], t);
                            acc[h][dy][ox] = t;
                        }
                    }
                }
            }
        }
        float4* part = reinterpret_cast<float4*>(sm + O_PART + (cs * 16 + (tid & 15)) * PTP);   // [h][dy][ox]
#pragma unroll
        for (int h = 0; h < 2; ++h)
#pragma unroll
            for (int dy = 0; dy < 2; ++dy) {
                part[(h * 2 + dy) * 2] = make_float4(acc[h][dy][0], acc[h][dy][1], acc[h][dy][2], acc[h][dy][3]);
                part[(h * 2 + dy) * 2 + 1] = make_float4(acc[h][dy][4], acc[h][dy][5], acc[h][dy][6], acc[h][dy][7]);
            }
    }
    TRACE(4, 0);
    __syncthreads();
    cluster.barrier_wait();              // all eight CTAs run: their shared memory may be written
    TRACE(5, 0);
    {
        // thread = (pooled column px, conv row dy of the window, channel h of the pair, g = channel pair + 4 * pooled row): the two conv
        // rows of a window meet by one shuffle, the four pooled values of a row by three (one 16 B store)
        const int px = tid & 3, dy = (tid >> 2) & 1, h = (tid >> 3) & 1, g = tid >> 4;
        const int cl = 2 * (g & 3) + h, py = g >> 2;                   // local channel 0..7
        const float* pp = sm + O_PART + g * PTP + h * 16 + dy * 8 + 2 * px;
        float2 s0 = *reinterpret_cast<const float2*>(pp);
#pragma unroll
        for (int k = 1; k < 16; ++k) {                        // input-channel pairs in fixed order
            const float2 t0 = *reinterpret_cast<const float2*>(pp + k * 16 * PTP);
            s0.x += t0.x; s0.y += t0.y;
        }
        float v = fmaxf(s0.x, s0.y);
        v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, 4));
        v = fmaxf(v + sm[O_B3 + cl], 0.f);                    // max_k relu(s_k + bias) = relu(max_k s_k + bias)
        const float v1 = __shfl_xor_sync(0xffffffffu, v, 1), v2 = __shfl_xor_sync(0xffffffffu, v, 2), v3 = __shfl_xor_sync(0xffffffffu, v, 3);
        if (px == 0 && dy == 0)                               // own channels -> own shared memory only
            *reinterpret_cast<float4*>(sm + O_A3 + (8 * r + cl) * A3P + py * 4) = make_float4(v, v1, v2, v3);
    }
    TRACE(15, 0);
    // all-gather of the 64 x 4 x 4 activation by PULL: a cluster barrier with no remote store in flight, then every thread fetches one
    // 16 B row of another CTA's eight channels through distributed shared memory (256 threads x 16 B = the whole activation). The push
    // form (each CTA storing its rows into all eight CTAs ahead of the barrier) cost 940 + 1,500 cycles: the barrier's release waits for
    // every remote store (tools/tail_trace.py).
    cluster.sync();
    {
        const int d = tid >> 5, cl = (tid >> 2) & 7, py = tid & 3;
        if (d != r) {
            const int off = O_A3 + (8 * d + cl) * A3P + py * 4;
            *reinterpret_cast<float4*>(sm + off) = *reinterpret_cast<const float4*>(cluster.map_shared_rank(sm, d) + off);
        }
    }
    __syncthreads();                     // the 64 x 4 x 4 activation is complete in this CTA
    TRACE(6, 0);

    // ---- phase C: conv4 + ReLU + pool -------------------------------------------------------------------------------------
    float feat = 0.f;
    {
        const int s = tid & 15, c = tid >> 4;                 // input channels s, s+16, s+32, s+48 of local output channel c
        float o[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const int ci = s + 16 * i;
            const float4* ip = reinterpret_cast<const float4*>(sm + O_A3 + ci * A3P);
            const float4 r0 = ip[0], r1 = ip[1], r2 = ip[2], r3 = ip[3];
            const float in[4][4] = {{r0.x, r0.y, r0.z, r0.w}, {r1.x, r1.y, r1.z, r1.w}, {r2.x, r2.y, r2.z, r2.w}, {r3.x, r3.y, r3.z, r3.w}};
            const float* wp = sm + O_W4 + c * W4P + ci * 9;
#pragma unroll
            for (int ky = 0; ky < 3; ++ky) {
#pragma unroll
                for (int kx = 0; kx < 3; ++kx) {
                    const float w = wp[ky * 3 + kx];
                    o[0] = fmaf(w, in[ky][kx], o[0]);
                    o[1] = fmaf(w, in[ky][kx + 1], o[1]);
                    o[2] = fmaf(w, in[ky + 1][kx], o[2]);
                    o[3] = fmaf(w, in[ky + 1][kx + 1], o[3]);
                }
            }
        }
#pragma unroll
        for (int off = 8; off > 0; off >>= 1) {               // the 16 input-channel slices of a channel sit in one half-warp
#pragma unroll
            for (int k = 0; k < 4; ++k) o[k] += __shfl_xor_sync(0xffffffffu, o[k], off);
        }
        if (s == 0) {
            feat = fmaxf(fmaxf(fmaxf(o[0], o[1]), fmaxf(o[2], o[3])) + sm[O_B4 + c], 0.f);
            cluster.map_shared_rank(sm + O_A4, 0)[16 * r + c] = feat;
        }
    }
    TRACE(7, 0);
    cluster.sync();                      // the 128 features are complete in CTA 0; nobody touches another CTA's memory afterwards
    TRACE(8, 0);
    // the optional copies of the two activations leave only now: a global store ahead of a cluster barrier makes the barrier's
    // release wait for its acknowledgement from L2 (measured: 2.5 K cycles for the first exchange with the store, see profiles/)
    if (a.act3 && tid < 32) {
        const int cl = tid >> 2, py = tid & 3;
        *reinterpret_cast<float4*>(a.act3 + ((size_t)b * 64 + 8 * r + cl) * 16 + py * 4) = *reinterpret_cast<const float4*>(sm + O_A3 + (8 * r + cl) * A3P + py * 4);
    }
    if (a.act4 && (tid & 15) == 0) a.act4[(size_t)b * 128 + 16 * r + (tid >> 4)] = feat;
    if (r != 0) { TRACE_END; return; }

    // ---- phase D: fc head + greedy action: every Linear layer on all 256 threads (a row is split over 4 / 8 / 8 neighbouring lanes and
    // folded by shuffles; the inner index is rotated per lane so that the 32 lanes of a warp, whose rows are congruent mod 32 floats,
    // read 32 different banks) -- the warp-per-output form of head_kernel took 3.6 K cycles here, on the critical path of one sample
    const float* s_a = sm + O_A4;
    float* s_h1 = sm + O_H1; float* s_h2 = sm + O_H2; float* s_z = sm + O_Z;
    {
        const int j = tid >> 2, q = tid & 3;                  // fc.0: output j, inputs [32q, 32q + 32) as eight 16 B words, rotated by the lane
        const float4* wr = reinterpret_cast<const float4*>(sm + O_HW0 + j * 128 + q * 32);
        const float4* ar = reinterpret_cast<const float4*>(s_a + q * 32);
        float p0 = 0.f, p1 = 0.f, p2 = 0.f, p3 = 0.f;
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const int k = (i + lane) & 7;
            const float4 w = wr[k], x = ar[k];
            p0 = fmaf(w.x, x.x, p0); p1 = fmaf(w.y, x.y, p1); p2 = fmaf(w.z, x.z, p2); p3 = fmaf(w.w, x.w, p3);
        }
        float p = (p0 + p1) + (p2 + p3);
        p += __shfl_xor_sync(0xffffffffu, p, 1);
        p += __shfl_xor_sync(0xffffffffu, p, 2);
        if (q == 0) s_h1[j] = fmaxf(p + sm[O_HB0 + j], 0.f);
    }
    __syncthreads();
    {
        const int j = tid >> 3, e = tid & 7;                  // fc.2: output j, inputs [8e, 8e + 8) as two 16 B words
        const float4* wr = reinterpret_cast<const float4*>(sm + O_HW2 + j * 64 + e * 8);
        const float4* hr = reinterpret_cast<const float4*>(s_h1 + e * 8);
        const int k0 = (e >> 2) & 1;                          // lanes e and e + 4 of a quarter-warp read different banks
        const float4 w0 = wr[k0], x0 = hr[k0], w1 = wr[k0 ^ 1], x1 = hr[k0 ^ 1];
        float p0 = fmaf(w0.x, x0.x, w0.y * x0.y), p1 = fmaf(w0.z, x0.z, w0.w * x0.w);
        p0 = fmaf(w1.x, x1.x, p0); p1 = fmaf(w1.y, x1.y, p1); p0 = fmaf(w1.z, x1.z, p0); p1 = fmaf(w1.w, x1.w, p1);
        float p = p0 + p1;
        p += __shfl_xor_sync(0xffffffffu, p, 1);
        p += __shfl_xor_sync(0xffffffffu, p, 2);
        p += __shfl_xor_sync(0xffffffffu, p, 4);
        if (e == 0) s_h2[j] = fmaxf(p + sm[O_HB2 + j], 0.f);
    }
    __syncthreads();
    {
        const int c = tid >> 3, e = tid & 7;                  // fc.4: output c (< NA), inputs [4e, 4e + 4)
        const int cc = c < NA ? c : NA - 1;                   // rows >= NA do not exist in shared memory
        const float* wr = sm + O_HW4 + cc * 32 + e * 4;
        const float* hr = s_h2 + e * 4;
        float p = 0.f;
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const int k = (i + c) & 3;
            p = fmaf(wr[k], hr[k], p);
        }
        p += __shfl_xor_sync(0xffffffffu, p, 1);
        p += __shfl_xor_sync(0xffffffffu, p, 2);
        p += __shfl_xor_sync(0xffffffffu, p, 4);
        if (e == 0 && c < NA) s_z[c] = p + sm[O_HB4 + c];
    }
    __syncthreads();
    if (a.hid1 && tid < 64) a.hid1[(size_t)b * 64 + tid] = s_h1[tid];
    if (a.hid2 && tid < 32) a.hid2[(size_t)b * 32 + tid] = s_h2[tid];
    if (tid < NA) a.logits[(size_t)b * NA + tid] = cmd_ok ? s_z[tid] : 0.f;
    if (warp == 0 && a.actions) {
        const float z = lane < NA ? s_z[lane] : -INFINITY;
        const float m = bc::warp_max(z);                                         // fmaxf: drops NaN
        // like torch.argmax: the first NaN if there is one (NaN counts as the maximum), else the first maximum
        const unsigned nan = __ballot_sync(0xffffffffu, lane < NA && isnan(z));
        const unsigned hit = nan ? nan : __ballot_sync(0xffffffffu, lane < NA && z == m);
        if (lane == 0) a.actions[b] = hit && cmd_ok ? (int64_t)(__ffs((int)hit) - 1) : 0;
    }
    if (kBranched && !cmd_ok && tid == 0 && br.err) atomicExch(br.err, 4);
    TRACE(9, 0);
    TRACE_END;
}

}  // namespace

BC_TRACE_EXPORT(bc_debug_tail_trace)       // debug builds only: not part of the ABI

// one launcher for both instantiations: `br` NULL = the single head (bc_ctx's fc and logits), else the commanded branch
static int launch_tail(const bc_ctx* c, const bc_branched* h, int64_t* actions, void* stream) {
    const char* who = h ? "bc_policy_tail_branched" : "bc_policy_tail";
    BC_CHECK_ARG(c && c->params && c->act[1], "%s: null buffer (needs params, act[1])", who);
    BC_CHECK_ARG(c->n_actions >= 1 && c->n_actions <= MAXA, "%s: n_actions %d outside 1..%d", who, c->n_actions, MAXA);
    BC_CHECK_ARG(c->batch >= 0 && c->batch <= BC_POLICY_TAIL_MAX_BATCH, "%s: batch %d outside 0..%d (one 8-CTA cluster per sample; "
                 "larger batches belong to the tensor-core kernels: bc_forward_act)", who, c->batch, BC_POLICY_TAIL_MAX_BATCH);
    if (h) {
        BC_CHECK_ARG(h->params && h->command && h->out, "%s: null buffer in bc_branched (needs params, command, out)", who);
        BC_CHECK_ARG(h->n_branches >= 1 && h->n_branches <= 16, "%s: n_branches %d outside 1..16", who, h->n_branches);
        BC_CHECK_ARG(h->n_out >= 1 && h->n_out <= MAXA, "%s: n_out %d outside 1..%d", who, h->n_out, MAXA);
        BC_CHECK_ARG(h->batch == c->batch, "%s: bc_branched.batch %d differs from bc_ctx.batch %d", who, h->batch, c->batch);
        BC_CHECK_ARG((uintptr_t)h->params % 16 == 0, "%s: the branch arena is read as 16 B words", who);
    } else {
        BC_CHECK_ARG(c->logits, "%s: null buffer (needs logits)", who);
    }
    if (c->batch == 0) return BC_OK;
    BC_CHECK_ARG(((uintptr_t)c->params | (uintptr_t)c->act[1]) % 16 == 0 && (!c->act[2] || (uintptr_t)c->act[2] % 16 == 0),
                 "%s: params, act[1] and act[2] are read / written as 16 B words", who);
    void (*kern)(const TailArgs, const BranchArgs) = h ? policy_tail_kernel<true> : policy_tail_kernel<false>;
    static bc::PerDeviceOnce once_[2]; bool& configured = once_[h ? 1 : 0]();
    if (!configured) {
        cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES);
        if (e != cudaSuccess) return bc::fail(BC_ERR_DEVICE, "policy_tail_kernel: smem opt-in %d B failed: %s", SMEM_BYTES, cudaGetErrorString(e));
        configured = true;
    }
    const bc::Arena ar = bc::arena_layout(c->obs_size, c->n_actions);
    TailArgs a{};
    a.act2 = c->act[1];
    a.w3 = c->params + ar.w[2]; a.b3 = c->params + ar.b[2];
    a.w4 = c->params + ar.w[3]; a.b4 = c->params + ar.b[3];
    a.f0 = c->params + ar.w[4]; a.g0 = c->params + ar.b[4];
    a.f2 = c->params + ar.w[5]; a.g2 = c->params + ar.b[5];
    a.f4 = c->params + ar.w[6]; a.g4 = c->params + ar.b[6];
    a.act3 = c->act[2]; a.act4 = c->act[3]; a.hid1 = c->hid1; a.hid2 = c->hid2;
    a.logits = c->logits; a.actions = actions;
    a.B = c->batch; a.NA = c->n_actions;
    BranchArgs br{};
    if (h) {
        int64_t off[6], siz[6];                          // state_dict order: 0.weight 0.bias 2.weight 2.bias 4.weight 4.bias
        br.head_len = bc_head_branched_layout(h->n_out, off, siz);
        br.w0 = off[0]; br.b0 = off[1]; br.w2 = off[2]; br.b2 = off[3]; br.w4 = off[4]; br.b4 = off[5];
        br.cmd = h->command; br.barena = h->params; br.G = h->n_branches; br.err = h->err_flag;
        a.logits = h->out; a.NA = h->n_out;              // fc.0 .. fc.4 come from the branch arena; conv3 / conv4 from the trunk's
        a.f0 = a.g0 = a.f2 = a.g2 = a.f4 = a.g4 = nullptr;
    }
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(c->batch * CL); cfg.blockDim = dim3(NT); cfg.dynamicSmemBytes = SMEM_BYTES; cfg.stream = (cudaStream_t)stream;
    cudaLaunchAttribute at[2];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = CL; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
    at[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[1].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = at; cfg.numAttrs = 2;
    const cudaError_t e = cudaLaunchKernelEx(&cfg, kern, a, br);
    if (e != cudaSuccess) bc::pending_launch_error() = e;
    BC_CUDA_LAUNCH_CHECK("policy_tail_kernel");
    return BC_OK;
}

extern "C" int bc_policy_tail(const bc_ctx* c, int64_t* actions, void* stream) {
    return launch_tail(c, nullptr, actions, stream);
}

extern "C" int bc_policy_tail_branched(const bc_ctx* c, const bc_branched* h, int64_t* actions, void* stream) {
    return launch_tail(c, h, actions, stream);
}
