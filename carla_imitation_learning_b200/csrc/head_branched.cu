// EXTENSION (no counterpart in the reference): command-conditioned branched action heads with CE / L1 / MSE loss.
// BASELINE.json's north_star asks for "command-conditioned action heads ... the per-command MLP branches and the L1/MSE
// steer/throttle/brake loss become a grouped GEMM with warp-shuffle reductions"; the reference's ConvNet1 has ONE head
// (/root/reference/src/architectures/nets.py:31-33) and CrossEntropyLoss (/root/reference/src/models/imitation.py:43-44),
// so parity for this file is against oracle/ext_oracle.py ("extension -- no reference parity").
//
// G branches, each the reference's MLP shape 128 -> 64 -> 32 -> n_out. Sample b is evaluated by branch command[b] only
// (the branch-select mask of conditional imitation learning); the other branches get no gradient from it.
// Grouped GEMM: grid = (blocks per branch, G). CTA (i, g) keeps branch g's three weight matrices in shared memory (42 KB)
// and walks the samples commanded to g whose rank within g is congruent to i mod nb, in increasing b. The command vector is
// read in coalesced chunks of kChunk samples; a block-wide ballot/popc prefix gives every sample of the chunk its rank within
// g, and the CTA compacts its own samples into a shared list (no CTA walks the whole batch one dependent load at a time).
// Per-sample vectors are reduced with warp shuffles, weight gradients accumulate in registers across the CTA's samples and
// leave as one partial per CTA; a second pass adds the partials of a branch in a fixed order (deterministic, no atomics).
// The branch weights are fetched as 16 B L2 loads BEFORE griddepcontrol.wait, under the previous kernel's tail, like the
// single head (head.cu): the branch arena is written only by torch ops and by bc_adam_tick_step, which releases its
// dependents after its last write (include/bc_b200.h, launch ordering). A command outside [0, G) raises flag 4; that
// sample's out row (and dout row with the loss, gfeat row with the backward) is written as zeros.
// Serving (bc_forward_branched_act, tail = 0): with `actions` set (mode 0 only), warp 0 also takes each sample's greedy
// action from its outputs, by the ballot code of the single-head tail (policy_tail.cu); an out-of-range command gets 0.
#include "bc_common.cuh"

namespace {

constexpr int NT = 256;
constexpr int MAXA = BC_MAX_ACTIONS;
constexpr int kBranchCtas = 128;      // CTAs over all branches (nb = kBranchCtas / G per branch)
constexpr int kMaxBranches = 16;
constexpr int kChunk = 1024;          // commands scanned per round: NT threads x kPer samples
constexpr int kPer = kChunk / NT;
constexpr int kListMax = kChunk / (kBranchCtas / kMaxBranches);   // most samples one CTA can own in a chunk (nb >= 8)
static_assert(kChunk % NT == 0 && kBranchCtas % kMaxBranches == 0, "chunking");

struct HeadLayout { int64_t w4, b4, w2, b2, w0, b0, len; };
__host__ __device__ inline int64_t pad32i(int64_t n) { return (n + 31) / 32 * 32; }
__host__ inline HeadLayout head_layout(int na) {      // the order of the arena's head segment (bc_common.cuh): fc.4, fc.2, fc.0; weight then bias
    HeadLayout l{};
    int64_t off = 0;
    l.w4 = off; off += pad32i((int64_t)na * 32); l.b4 = off; off += pad32i(na);
    l.w2 = off; off += pad32i(32 * 64);          l.b2 = off; off += pad32i(32);
    l.w0 = off; off += pad32i(64 * 128);         l.b0 = off; off += pad32i(64);
    l.len = off;
    return l;
}

struct BrArgs {
    const float* feat; const int64_t* cmd; const int64_t* y; const float* tgt; const float* params;
    float* out; float* dout; float* gfeat; float* part; float* loss_part;
    int64_t* actions;                         // (B,) greedy actions over out, or NULL (mode 0 only)
    HeadLayout L;
    int B, NA, G, nb, mode, kind;
    float loss_scale;
    int* err;
};

__global__ void __launch_bounds__(NT) head_branched_kernel(const BrArgs a) {
    __shared__ __align__(16) float s_w0[64 * 128];
    __shared__ __align__(16) float s_w2[32 * 64];
    __shared__ __align__(16) float s_w4[MAXA * 32];
    __shared__ float s_b0[64], s_b2[32], s_b4[MAXA];
    __shared__ float s_a[128], s_h1[64], s_h2[32], s_z[MAXA], s_dl[MAXA], s_dh2[32], s_dh1[64];
    __shared__ int s_wcnt[kPer][NT / 32];     // per scan round: matches of branch g in each warp
    __shared__ int s_list[kListMax];          // this CTA's samples of the current chunk, increasing b
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int NA = a.NA, g = blockIdx.y, nb = a.nb, bx = blockIdx.x;
    {
        // branch g's weights: 16 B L2 loads (ld.cg: an L1 line of an earlier launch on this SM could be stale), all in
        // flight at once; segment offsets are 32-float padded, so every tensor is 16 B aligned
        const float* P = a.params + (size_t)g * a.L.len;
        const float4* w0v = reinterpret_cast<const float4*>(P + a.L.w0);
        float4 t[8];
#pragma unroll
        for (int q = 0; q < 8; ++q) t[q] = __ldcg(w0v + tid + NT * q);
        const float4* w2v = reinterpret_cast<const float4*>(P + a.L.w2);
        float4 u0 = __ldcg(w2v + tid), u1 = __ldcg(w2v + tid + NT);
        const bool has4 = tid < NA * 8;
        float4 u4 = has4 ? __ldcg(reinterpret_cast<const float4*>(P + a.L.w4) + tid) : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
        for (int q = 0; q < 8; ++q) reinterpret_cast<float4*>(s_w0)[tid + NT * q] = t[q];
        reinterpret_cast<float4*>(s_w2)[tid] = u0;
        reinterpret_cast<float4*>(s_w2)[tid + NT] = u1;
        if (has4) reinterpret_cast<float4*>(s_w4)[tid] = u4;
        if (tid < 64) s_b0[tid] = __ldcg(P + a.L.b0 + tid);
        if (tid < 32) s_b2[tid] = __ldcg(P + a.L.b2 + tid);
        if (tid < NA) s_b4[tid] = __ldcg(P + a.L.b4 + tid);
    }
    bc::pdl_wait();                           // features, commands, labels, targets and every output from here on
    bc::pdl_trigger();

    float acc0[32], acc2[8], acc4[2], accb = 0.f, block_loss = 0.f;
#pragma unroll
    for (int r = 0; r < 32; ++r) acc0[r] = 0.f;
#pragma unroll
    for (int r = 0; r < 8; ++r) acc2[r] = 0.f;
    acc4[0] = acc4[1] = 0.f;
    const bool do_loss = a.mode & 1, do_bwd = a.mode & 2;
    const bool reporter = bx == 0 && g == 0;  // the CTA that raises flag 4 and zeroes the rows of out-of-range commands
    // samples of branch g with rank r < s that this CTA owns (r = bx, bx + nb, ...)
    auto owned_below = [&](int s) { return s > bx ? (s - bx + nb - 1) / nb : 0; };

    int seen = 0;                                   // samples of this branch in earlier chunks (same count in every CTA of the branch)
    for (int c0 = 0; c0 < a.B; c0 += kChunk) {
        // ---- scan: sample c0 + NT*k + tid in round k (coalesced), rank within g by ballot/popc prefix
        int64_t cmd[kPer];
#pragma unroll
        for (int k = 0; k < kPer; ++k) {
            const int b = c0 + NT * k + tid;
            cmd[k] = b < a.B ? a.cmd[b] : (int64_t)g + 1;     // past the batch: matches no branch, never reported
        }
        unsigned bal[kPer];
#pragma unroll
        for (int k = 0; k < kPer; ++k) {
            const int b = c0 + NT * k + tid;
            bal[k] = __ballot_sync(0xffffffffu, cmd[k] == g);
            if (b < a.B && (cmd[k] < 0 || cmd[k] >= a.G) && reporter) {   // reported; the sample leaves zero rows behind
                if (a.err) atomicExch(a.err, 4);
                for (int j = 0; j < NA; ++j) a.out[(size_t)b * NA + j] = 0.f;
                if (a.actions) a.actions[b] = 0;
                if (do_loss) for (int j = 0; j < NA; ++j) a.dout[(size_t)b * NA + j] = 0.f;
                if (do_bwd) for (int j = 0; j < 128; ++j) a.gfeat[(size_t)b * 128 + j] = 0.f;
            }
            if (lane == 0) s_wcnt[k][warp] = __popc(bal[k]);
        }
        __syncthreads();                            // s_wcnt complete; the previous chunk's list is no longer read
        const int first = owned_below(seen);
        int run = seen;
#pragma unroll
        for (int k = 0; k < kPer; ++k) {
            int before = 0, total = 0;
#pragma unroll
            for (int w = 0; w < NT / 32; ++w) {
                const int n = s_wcnt[k][w];
                before += w < warp ? n : 0;
                total += n;
            }
            if (cmd[k] == g) {
                const int r = run + before + __popc(bal[k] & ((1u << lane) - 1u));
                if (r % nb == bx) s_list[r / nb - first] = c0 + NT * k + tid;
            }
            run += total;
        }
        const int n_mine = owned_below(run) - first;
        seen = run;
        __syncthreads();                            // s_list complete
        for (int li = 0; li < n_mine; ++li) {
            const int b = s_list[li];
            __syncthreads();  // weights loaded / previous sample's vectors no longer read
            if (tid < 128) s_a[tid] = a.feat[(size_t)b * 128 + tid];
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
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const int j = warp * 4 + q;
                float p = fmaf(s_w2[j * 64 + lane], s_h1[lane], s_w2[j * 64 + lane + 32] * s_h1[lane + 32]);
                p = bc::warp_sum(p);
                if (lane == 0) s_h2[j] = fmaxf(p + s_b2[j], 0.f);
            }
            __syncthreads();
            for (int c = warp; c < NA; c += 8) {
                float p = bc::warp_sum(s_w4[c * 32 + lane] * s_h2[lane]);
                if (lane == 0) s_z[c] = p + s_b4[c];
            }
            __syncthreads();
            if (tid < NA) a.out[(size_t)b * NA + tid] = s_z[tid];
            if (warp == 0 && a.actions) {
                const float z = lane < NA ? s_z[lane] : -INFINITY;
                const float m = bc::warp_max(z);                                 // fmaxf: drops NaN
                // like torch.argmax: the first NaN if there is one (NaN counts as the maximum), else the first maximum
                const unsigned nan = __ballot_sync(0xffffffffu, lane < NA && isnan(z));
                const unsigned hit = nan ? nan : __ballot_sync(0xffffffffu, lane < NA && z == m);
                if (lane == 0) a.actions[b] = hit ? (int64_t)(__ffs((int)hit) - 1) : 0;
            }
            if (!do_loss && !do_bwd) continue;
            if (warp == 0) {
                if (do_loss) {
                    float dl = 0.f;
                    if (a.kind == 0) {                   // CrossEntropy over the branch's n_out classes
                        const float z = lane < NA ? s_z[lane] : -INFINITY;
                        const float m = bc::warp_max(z);
                        const float e = lane < NA ? expf(z - m) : 0.f;
                        const float sum = bc::warp_sum(e);
                        int yb = (int)a.y[b];
                        if (yb < 0 || yb >= NA) { if (lane == 0 && a.err) atomicExch(a.err, 3); yb = 0; }
                        const float zy = __shfl_sync(0xffffffffu, z, yb & 31);
                        if (lane == 0) block_loss += (logf(sum) + m - zy);
                        dl = (e / sum - (lane == yb ? 1.f : 0.f)) * a.loss_scale;
                    } else {                             // L1 / MSE on the regression targets (steer, throttle, brake)
                        const float d = lane < NA ? s_z[lane] - a.tgt[(size_t)b * NA + lane] : 0.f;
                        const float l = a.kind == 1 ? fabsf(d) : d * d;
                        const float tot = bc::warp_sum(l);
                        if (lane == 0) block_loss += tot;
                        dl = (a.kind == 1 ? (d > 0.f ? 1.f : (d < 0.f ? -1.f : 0.f)) : 2.f * d) * a.loss_scale;
                    }
                    if (lane < NA) { s_dl[lane] = dl; a.dout[(size_t)b * NA + lane] = dl; }
                } else if (lane < NA) {
                    s_dl[lane] = a.dout[(size_t)b * NA + lane];
                }
            }
            if (!do_bwd) continue;
            __syncthreads();
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
                a.gfeat[(size_t)b * 128 + tid] = p;
            }
        }
    }
    const int slot = g * a.nb + blockIdx.x;
    if (do_loss && tid == 0) a.loss_part[slot] = block_loss * a.loss_scale;
    if (do_bwd) {
        float* part = a.part + (size_t)slot * a.L.len;
#pragma unroll
        for (int r = 0; r < 32; ++r) part[a.L.w0 + tid + NT * r] = acc0[r];
#pragma unroll
        for (int r = 0; r < 8; ++r) part[a.L.w2 + tid + NT * r] = acc2[r];
#pragma unroll
        for (int r = 0; r < 2; ++r) if (tid + NT * r < NA * 32) part[a.L.w4 + tid + NT * r] = acc4[r];
        if (tid < 64) part[a.L.b0 + tid] = accb;
        else if (tid < 96) part[a.L.b2 + tid - 64] = accb;
        else if (tid < 96 + NA) part[a.L.b4 + tid - 96] = accb;
    }
}

// grads[g][i] = sum over the branch's nb partial copies, in slot order; loss = sum of all loss partials.
// grads_epoch != NULL (data-parallel peer exchange): grads is double-buffered, the half ((*grads_epoch + 1) & 1) is written
__global__ void __launch_bounds__(256) branched_reduce_kernel(const float* __restrict__ part, const float* __restrict__ loss_part,
                                                               float* __restrict__ grads, float* __restrict__ loss,
                                                               int64_t len, int G, int nb, int with_grads, int with_loss,
                                                               const uint32_t* __restrict__ grads_epoch, int64_t grads_stride) {
    bc::pdl_wait();
    bc::pdl_trigger();
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (with_grads && i < len * G) {
        const int g = (int)(i / len);
        const int64_t e = i - (int64_t)g * len;
        float s = 0.f;
        for (int k = 0; k < nb; ++k) s += part[((size_t)g * nb + k) * len + e];
        const int64_t par = grads_epoch ? (int64_t)((*grads_epoch + 1u) & 1u) * grads_stride : 0;
        grads[par + i] = s;
    }
    if (with_loss && blockIdx.x == 0 && threadIdx.x < 32) {
        float v = 0.f;
        for (int k = threadIdx.x; k < G * nb; k += 32) v += loss_part[k];
        v = bc::warp_sum(v);
        if (threadIdx.x == 0) loss[0] = v;
    }
}

}  // namespace

extern "C" int64_t bc_head_branched_layout(int n_out, int64_t offsets[6], int64_t sizes[6]) {
    const HeadLayout l = head_layout(n_out);
    // state_dict order of one branch: 0.weight 0.bias 2.weight 2.bias 4.weight 4.bias
    offsets[0] = l.w0; sizes[0] = 64 * 128; offsets[1] = l.b0; sizes[1] = 64;
    offsets[2] = l.w2; sizes[2] = 32 * 64;  offsets[3] = l.b2; sizes[3] = 32;
    offsets[4] = l.w4; sizes[4] = (int64_t)n_out * 32; offsets[5] = l.b4; sizes[5] = n_out;
    return l.len;
}

static int branch_ctas(int G) { int nb = kBranchCtas / (G < 1 ? 1 : G); return nb < 1 ? 1 : nb; }

extern "C" size_t bc_head_branched_partials_floats(int n_branches, int n_out) {
    const HeadLayout l = head_layout(n_out);
    const int nb = branch_ctas(n_branches);
    return (size_t)n_branches * nb * l.len + 32 * (((size_t)n_branches * nb + 31) / 32);
}

// bc_head_branched, and the serving head of bc_forward_branched_act (mode 0, `actions` may be set, no partials needed)
static int head_branched_launch(const bc_branched* h, int mode, int64_t* actions, void* stream) {
    BC_CHECK_ARG(h && h->feat && h->command && h->params && h->out && (h->partials || !(mode & 3)), "bc_head_branched: null buffer");
    BC_CHECK_ARG(!actions || mode == 0, "bc_head_branched: greedy actions are taken in mode 0 (outputs only)");
    BC_CHECK_ARG(h->n_branches >= 1 && h->n_branches <= 16, "bc_head_branched: n_branches %d outside 1..16", h->n_branches);
    BC_CHECK_ARG(h->n_out >= 1 && h->n_out <= MAXA, "bc_head_branched: n_out %d outside 1..%d", h->n_out, MAXA);
    BC_CHECK_ARG(h->loss_kind >= 0 && h->loss_kind <= 2, "bc_head_branched: loss_kind %d (0 CE, 1 L1, 2 MSE)", h->loss_kind);
    BC_CHECK_ARG(!(mode & 1) || (h->dout && h->loss && (h->loss_kind == 0 ? (const void*)h->labels : (const void*)h->targets)),
                 "bc_head_branched: the loss needs dout, loss and labels (CE) or targets (L1/MSE)");
    BC_CHECK_ARG(!(mode & 2) || (h->dout && h->gfeat && h->grads), "bc_head_branched: backward needs dout, gfeat, grads");
    if (h->batch == 0 && !(mode & 3)) return BC_OK;
    BrArgs a{};
    a.feat = h->feat; a.cmd = h->command; a.y = h->labels; a.tgt = h->targets; a.params = h->params;
    a.out = h->out; a.dout = h->dout; a.gfeat = h->gfeat; a.actions = actions;
    a.L = head_layout(h->n_out);
    a.B = h->batch; a.NA = h->n_out; a.G = h->n_branches; a.nb = branch_ctas(h->n_branches); a.mode = mode; a.kind = h->loss_kind;
    a.loss_scale = h->loss_scale; a.err = h->err_flag;
    a.part = h->partials;
    a.loss_part = h->partials ? h->partials + (size_t)a.G * a.nb * a.L.len : nullptr;
    bc::launch_pdl(head_branched_kernel, dim3(a.nb, a.G), dim3(NT), 0, (cudaStream_t)stream, a);
    BC_CUDA_LAUNCH_CHECK("head_branched_kernel");
    if (mode & 3) {
        const int64_t n = a.L.len * a.G;
        bc::launch_pdl(branched_reduce_kernel, dim3((unsigned)((n + 255) / 256)), dim3(256), 0, (cudaStream_t)stream,
                       (const float*)a.part, (const float*)a.loss_part, h->grads, h->loss, a.L.len, a.G, a.nb, (mode & 2) ? 1 : 0, (mode & 1) ? 1 : 0,
                       h->grads_epoch, h->grads_stride);
        BC_CUDA_LAUNCH_CHECK("branched_reduce_kernel");
    }
    return BC_OK;
}

extern "C" int bc_head_branched(const bc_branched* h, int mode, void* stream) {
    BC_CHECK_ARG(h && h->partials, "bc_head_branched: null buffer");
    return head_branched_launch(h, mode, nullptr, stream);
}

extern "C" int bc_forward_branched_act(const bc_ctx* c, const bc_branched* h, int64_t* actions, int tail, void* stream) {
    BC_CHECK_ARG(c && h, "bc_forward_branched_act: null ctx / branched heads");
    BC_CHECK_ARG(h->batch == c->batch, "bc_forward_branched_act: bc_branched.batch %d differs from bc_ctx.batch %d", h->batch, c->batch);
    BC_CHECK_ARG(!tail || (c->batch >= 0 && c->batch <= BC_POLICY_TAIL_MAX_BATCH),
                 "bc_forward_branched_act: tail = 1 serves batches up to %d (got %d)", BC_POLICY_TAIL_MAX_BATCH, c->batch);
    BC_CHECK_ARG(h->params && (uintptr_t)h->params % 16 == 0, "bc_forward_branched_act: the branch arena must be 16 B aligned");
    BC_CHECK_ARG(c->act[3] || tail, "bc_forward_branched_act: tail = 0 needs act[3] (the heads' features)");
    for (int l = 0; l < (tail ? 2 : 4); ++l) {
        int rc = bc_conv_relu_pool_fwd(c, l, stream);
        if (rc) return rc;
    }
    if (tail) return bc_policy_tail_branched(c, h, actions, stream);
    bc_branched hh = *h;                      // the heads read the trunk's pooled conv4 output
    hh.feat = c->act[3];
    return head_branched_launch(&hh, 0, actions, stream);
}
