// K5-K7: the fc head 128 -> 64 -> 32 -> n_actions, CrossEntropy(mean) and their backward,
// one kernel. Replaces ConvNet1.fc (/root/reference/src/architectures/nets.py:31-33,38),
// nn.CrossEntropyLoss() (/root/reference/src/models/imitation.py:43-44) and the autograd
// of both. A CTA keeps all three weight matrices in shared memory (42 KB) and walks its
// samples one by one; per-sample vectors are reduced with warp shuffles, weight gradients
// accumulate in registers (45 per thread) across the CTA's samples and leave as one partial
// per CTA (fixed-order second pass in bc_reduce_partials => deterministic).
#include "bc_common.cuh"

namespace {

constexpr int NT = 256;
constexpr int MAXA = BC_MAX_ACTIONS;

struct HeadArgs {
    const float* act3;   // (B,128)
    const int64_t* y;
    const float* w0; const float* b0; const float* w2; const float* b2; const float* w4; const float* b4;
    float* hid1; float* hid2; float* logits; float* dlogits; float* ghead;
    float* part;         // partial copies of the head gradient segment, [gridDim.x][seg_len]
    float* loss_part;    // [gridDim.x]
    int64_t seg_len;
    int64_t ow0, ob0, ow2, ob2, ow4, ob4;  // offsets inside the segment
    int B, NA, mode;
    float loss_scale;
    int* err;            // device flag: 3 = a label outside [0, n_actions) (nn.CrossEntropyLoss raises there)
    int64_t* actions;    // optional (B): greedy action = first maximum of the logits (serving: no separate argmax launch)
};

__global__ void __launch_bounds__(NT) head_kernel(const HeadArgs a) {
    __shared__ __align__(16) float s_w0[64 * 128];
    __shared__ __align__(16) float s_w2[32 * 64];
    __shared__ __align__(16) float s_w4[MAXA * 32];
    __shared__ float s_b0[64], s_b2[32], s_b4[MAXA];
    __shared__ float s_a[128], s_h1[64], s_h2[32], s_z[MAXA], s_dl[MAXA], s_dh2[32], s_dh1[64];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int NA = a.NA;
    // 42 KB of weights per CTA as 16 B loads, all of a thread's loads in flight at once (arena tensors are padded to 32 floats:
    // 16 B aligned); the scalar version of this prologue was a quarter of the kernel's time. The parameters are written only
    // by kernels that release their dependents after their last write (Adam: abi.cu), so this prologue runs BEFORE the wait,
    // under conv4's forward; L2 loads (ld.cg): an L1 line of an earlier launch on this SM could be stale.
    {
        const float4* w0v = reinterpret_cast<const float4*>(a.w0);
        float4 t[8];
#pragma unroll
        for (int q = 0; q < 8; ++q) t[q] = __ldcg(w0v + tid + NT * q);
        const float4* w2v = reinterpret_cast<const float4*>(a.w2);
        float4 u0 = __ldcg(w2v + tid), u1 = __ldcg(w2v + tid + NT);
        const bool has4 = tid < NA * 8;
        float4 u4 = has4 ? __ldcg(reinterpret_cast<const float4*>(a.w4) + tid) : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
        for (int q = 0; q < 8; ++q) reinterpret_cast<float4*>(s_w0)[tid + NT * q] = t[q];
        reinterpret_cast<float4*>(s_w2)[tid] = u0;
        reinterpret_cast<float4*>(s_w2)[tid + NT] = u1;
        if (has4) reinterpret_cast<float4*>(s_w4)[tid] = u4;
    }
    if (tid < 64) s_b0[tid] = __ldcg(a.b0 + tid);
    if (tid < 32) s_b2[tid] = __ldcg(a.b2 + tid);
    if (tid < NA) s_b4[tid] = __ldcg(a.b4 + tid);
    bc::pdl_trigger();
    bc::pdl_wait();                       // activations, labels and every output from here on

    float acc0[32], acc2[8], acc4[2], accb = 0.f, block_loss = 0.f;
#pragma unroll
    for (int r = 0; r < 32; ++r) acc0[r] = 0.f;
#pragma unroll
    for (int r = 0; r < 8; ++r) acc2[r] = 0.f;
    acc4[0] = acc4[1] = 0.f;
    const bool do_ce = a.mode & 1, do_bwd = a.mode & 2;

    for (int b = blockIdx.x; b < a.B; b += gridDim.x) {
        __syncthreads();  // weights loaded / previous sample's vectors no longer read
        if (tid < 128) s_a[tid] = a.act3[(size_t)b * 128 + tid];
        __syncthreads();
        // fc.0 + ReLU: warp w -> outputs 8w..8w+7
#pragma unroll
        for (int q = 0; q < 8; ++q) {
            const int j = warp * 8 + q;
            float p = 0.f;
#pragma unroll
            for (int i = 0; i < 4; ++i) p = fmaf(s_w0[j * 128 + lane + 32 * i], s_a[lane + 32 * i], p);
            p = bc::warp_sum(p);
            if (lane == 0) s_h1[j] = fmaxf(p + s_b0[j], 0.f);
        }
        __syncthreads();
        // fc.2 + ReLU: warp w -> outputs 4w..4w+3
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const int j = warp * 4 + q;
            float p = fmaf(s_w2[j * 64 + lane], s_h1[lane], s_w2[j * 64 + lane + 32] * s_h1[lane + 32]);
            p = bc::warp_sum(p);
            if (lane == 0) s_h2[j] = fmaxf(p + s_b2[j], 0.f);
        }
        __syncthreads();
        // fc.4: warp w -> outputs w, w+8
        for (int c = warp; c < NA; c += 8) {
            float p = bc::warp_sum(s_w4[c * 32 + lane] * s_h2[lane]);
            if (lane == 0) s_z[c] = p + s_b4[c];
        }
        __syncthreads();
        if (tid < 64) a.hid1[(size_t)b * 64 + tid] = s_h1[tid];
        if (tid < 32) a.hid2[(size_t)b * 32 + tid] = s_h2[tid];
        if (tid < NA) a.logits[(size_t)b * NA + tid] = s_z[tid];
        if (a.actions && warp == 0) {
            const float z = lane < NA ? s_z[lane] : -INFINITY;
            const float m = bc::warp_max(z);                                         // fmaxf: drops NaN
            // like torch.argmax: the first NaN if there is one (NaN counts as the maximum), else the first maximum
            const unsigned nan = __ballot_sync(0xffffffffu, lane < NA && isnan(z));
            const unsigned hit = nan ? nan : __ballot_sync(0xffffffffu, lane < NA && z == m);
            if (lane == 0) a.actions[b] = hit ? (int64_t)(__ffs((int)hit) - 1) : 0;
        }
        if (!do_ce && !do_bwd) continue;
        if (warp == 0) {
            if (do_ce) {
                const float z = lane < NA ? s_z[lane] : -INFINITY;
                const float m = bc::warp_max(z);
                const float e = lane < NA ? expf(z - m) : 0.f;
                const float sum = bc::warp_sum(e);
                int yb = (int)a.y[b];
                if (yb < 0 || yb >= NA) {        // reported through the device flag (checked by the host at epoch end / in tests); the sample contributes class 0
                    if (lane == 0 && a.err) atomicExch(a.err, 3);
                    yb = 0;
                }
                const float zy = __shfl_sync(0xffffffffu, z, yb & 31);
                if (lane == 0) block_loss += (logf(sum) + m - zy);
                const float dl = (e / sum - (lane == yb ? 1.f : 0.f)) * a.loss_scale;
                if (lane < NA) { s_dl[lane] = dl; a.dlogits[(size_t)b * NA + lane] = dl; }
            } else if (lane < NA) {
                s_dl[lane] = a.dlogits[(size_t)b * NA + lane];
            }
        }
        if (!do_bwd) continue;
        __syncthreads();
        // fc.4 grads; dh2 = W4^T dl, masked by ReLU
#pragma unroll
        for (int r = 0; r < 2; ++r) {
            const int e = tid + NT * r;
            if (e < NA * 32) acc4[r] = fmaf(s_dl[e >> 5], s_h2[e & 31], acc4[r]);
        }
        if (tid >= 96 && tid < 96 + NA) accb += s_dl[tid - 96];
        if (tid < 32) {
            float p = 0.f;
            for (int c = 0; c < NA; ++c) p = fmaf(s_dl[c], s_w4[c * 32 + tid], p);
            s_dh2[tid] = s_h2[tid] > 0.f ? p : 0.f;
        }
        __syncthreads();
#pragma unroll
        for (int r = 0; r < 8; ++r) {
            const int e = tid + NT * r;
            acc2[r] = fmaf(s_dh2[e >> 6], s_h1[e & 63], acc2[r]);
        }
        if (tid >= 64 && tid < 96) accb += s_dh2[tid - 64];
        if (tid < 64) {
            float p = 0.f;
#pragma unroll 8
            for (int j = 0; j < 32; ++j) p = fmaf(s_dh2[j], s_w2[j * 64 + tid], p);
            s_dh1[tid] = s_h1[tid] > 0.f ? p : 0.f;
        }
        __syncthreads();
#pragma unroll
        for (int r = 0; r < 32; ++r) {
            const int e = tid + NT * r;
            acc0[r] = fmaf(s_dh1[e >> 7], s_a[e & 127], acc0[r]);
        }
        if (tid < 64) accb += s_dh1[tid];
        if (tid < 128) {
            float p = 0.f;
#pragma unroll 8
            for (int k = 0; k < 64; ++k) p = fmaf(s_dh1[k], s_w0[k * 128 + tid], p);
            a.ghead[(size_t)b * 128 + tid] = p;
        }
    }
    if (do_ce && tid == 0) a.loss_part[blockIdx.x] = block_loss * a.loss_scale;
    if (do_bwd) {
        float* part = a.part + (size_t)blockIdx.x * a.seg_len;
#pragma unroll
        for (int r = 0; r < 32; ++r) part[a.ow0 + tid + NT * r] = acc0[r];
#pragma unroll
        for (int r = 0; r < 8; ++r) part[a.ow2 + tid + NT * r] = acc2[r];
#pragma unroll
        for (int r = 0; r < 2; ++r) if (tid + NT * r < NA * 32) part[a.ow4 + tid + NT * r] = acc4[r];
        if (tid < 64) part[a.ob0 + tid] = accb;
        else if (tid < 96) part[a.ob2 + tid - 64] = accb;
        else if (tid < 96 + NA) part[a.ob4 + tid - 96] = accb;
    }
}

__global__ void argmax_kernel(const float* __restrict__ logits, int64_t* __restrict__ out, int B, int NA) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    const float* z = logits + (size_t)b * NA;
    // like torch.argmax: the first NaN if there is one (NaN counts as the maximum), else the first maximum
    float best = z[0]; int idx = 0;
    for (int c = 1; c < NA && !isnan(best); ++c) if (z[c] > best || isnan(z[c])) { best = z[c]; idx = c; }
    out[b] = idx;
}

__global__ void __launch_bounds__(256) scale_inplace_kernel(float4* __restrict__ v, int64_t n4, const float* __restrict__ scale) {
    bc::pdl_wait();
    bc::pdl_trigger();
    const float s = *scale;
    if (s == 1.0f) return;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += stride) {
        float4 t = v[i];
        t.x *= s; t.y *= s; t.z *= s; t.w *= s;
        v[i] = t;
    }
}

}  // namespace

extern "C" int bc_scale_inplace(float* v, int64_t n, const float* scale_dev, void* stream) {
    BC_CHECK_ARG(v && scale_dev && n >= 0 && n % 4 == 0 && (uintptr_t)v % 16 == 0, "bc_scale_inplace: null / unaligned buffer or n not a multiple of 4");
    if (n == 0) return BC_OK;
    int blocks = (int)((n / 4 + 255) / 256);
    if (blocks > bc::num_sms() * 4) blocks = bc::num_sms() * 4;
    bc::launch_pdl(scale_inplace_kernel, dim3(blocks), dim3(256), 0, (cudaStream_t)stream, (float4*)v, n / 4, scale_dev);
    BC_CUDA_LAUNCH_CHECK("scale_inplace_kernel");
    return BC_OK;
}

int bc_head_launch(const bc_ctx* c, int head_mode, int64_t* actions, void* stream) {
    BC_CHECK_ARG(c && c->params && c->act[3] && c->hid1 && c->hid2 && c->logits, "bc_head: null buffer");
    BC_CHECK_ARG(c->n_actions >= 1 && c->n_actions <= MAXA, "bc_head: n_actions %d outside 1..%d", c->n_actions, MAXA);
    BC_CHECK_ARG(!(head_mode & 1) || (c->y && c->dlogits && c->partials), "bc_head: CE needs y, dlogits, partials");
    BC_CHECK_ARG(!(head_mode & 2) || (c->dlogits && c->ghead && c->partials), "bc_head: backward needs dlogits, ghead, partials");
    if (c->batch == 0 && !(head_mode & 3)) return BC_OK;
    const bc::Arena ar = bc::arena_layout(c->obs_size, c->n_actions);
    const bc::Partials pl = bc::partials_layout(ar);
    HeadArgs a{};
    a.act3 = c->act[3]; a.y = c->y;
    a.w0 = c->params + ar.w[4]; a.b0 = c->params + ar.b[4];
    a.w2 = c->params + ar.w[5]; a.b2 = c->params + ar.b[5];
    a.w4 = c->params + ar.w[6]; a.b4 = c->params + ar.b[6];
    a.hid1 = c->hid1; a.hid2 = c->hid2; a.logits = c->logits; a.dlogits = c->dlogits; a.ghead = c->ghead;
    a.part = c->partials ? c->partials + pl.off[0] : nullptr;
    a.loss_part = c->partials ? c->partials + pl.loss_off : nullptr;
    a.seg_len = ar.seg_len[0];
    a.ow0 = ar.w[4]; a.ob0 = ar.b[4]; a.ow2 = ar.w[5]; a.ob2 = ar.b[5]; a.ow4 = ar.w[6]; a.ob4 = ar.b[6];
    a.B = c->batch; a.NA = c->n_actions; a.mode = head_mode; a.loss_scale = c->loss_scale; a.err = c->err_flag;
    a.actions = actions;
    // the partial layout has a fixed number of copies, so the grid is fixed as well
    bc::launch_pdl(head_kernel, dim3(bc::kHeadBlocks), dim3(NT), 0, (cudaStream_t)stream, a);
    BC_CUDA_LAUNCH_CHECK("head_kernel");
    return BC_OK;
}

extern "C" int bc_head(const bc_ctx* c, int head_mode, void* stream) { return bc_head_launch(c, head_mode, nullptr, stream); }

extern "C" int bc_argmax(const float* logits, int64_t* actions, int batch, int n_actions, void* stream) {
    BC_CHECK_ARG(logits && actions && batch >= 0 && n_actions >= 1, "bc_argmax: bad arguments");
    if (batch == 0) return BC_OK;
    argmax_kernel<<<(batch + 127) / 128, 128, 0, (cudaStream_t)stream>>>(logits, actions, batch, n_actions);
    BC_CUDA_LAUNCH_CHECK("argmax_kernel");
    return BC_OK;
}
