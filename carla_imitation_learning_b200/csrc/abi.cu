// C-ABI glue: error state, device check, arena layout, forward/backward drivers, fused Adam.
#include "bc_common.cuh"
#include "pack.cuh"
#include <math.h>
#include <type_traits>

namespace bc {

static thread_local char g_err[512] = "";
char* err_buf() { return g_err; }
int fail(int code, const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return code;
}

cudaError_t& pending_launch_error() {
    static thread_local cudaError_t e = cudaSuccess;
    return e;
}

int num_sms() {
    static int cached[64] = {0};
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return 148;
    if (cached[dev] == 0) {
        int n = 0;
        if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) n = 148;
        cached[dev] = n;
    }
    return cached[dev];
}

}  // namespace bc

namespace {

// ---- K10: fused multi-tensor Adam over the flat arena ---------------------------------------
// state (doubles, like the Python scalars torch.optim.Adam works with):
//   [0] lr [1] beta1 [2] beta2 [3] eps [4] step [5] grad_scale [6] step_size (out) [7] bc2_sqrt (out)
// beta1 ** step and beta2 ** step for the integer-valued step count, by binary exponentiation with the two chains
// interleaved: ~2 log2(step) dependent f64 multiplies (a few hundred cycles) where two calls of the general pow() cost
// 1.3 us at the head of a 10 us kernel (profiles/README.md). The products differ from the correctly rounded power by
// < 1e-14 relative; the bias corrections they enter are rounded to f32 before use.
__device__ __forceinline__ void beta_powers(double b1, double b2, double step, double& p1, double& p2) {
    if (!(step >= 1.0 && step < 9.0e15) || step != floor(step)) { p1 = pow(b1, step); p2 = pow(b2, step); return; }
    unsigned long long n = (unsigned long long)step;
    double r1 = 1.0, r2 = 1.0;
    while (true) {
        if (n & 1ull) { r1 *= b1; r2 *= b2; }
        n >>= 1;
        if (!n) break;
        b1 *= b1; b2 *= b2;
    }
    p1 = r1; p2 = r2;
}

__global__ void adam_tick_kernel(double* st) {
    bc::pdl_wait();
    bc::pdl_trigger();
    // torch/optim/adam.py (single-tensor path): bias_correction1 = 1 - beta1 ** step;
    // step_size = lr / bias_correction1; bias_correction2_sqrt = sqrt(1 - beta2 ** step) -- all in f64.
    const double step = st[4] + 1.0;
    double p1, p2;
    beta_powers(st[1], st[2], step, p1, p2);
    st[4] = step;
    st[6] = st[0] / (1.0 - p1);
    st[7] = sqrt(1.0 - p2);
}

// tick folded into the update: every CTA derives the step's scalars from st[4] + 1 itself (same f64 formulas as
// adam_tick_kernel), the last CTA to finish publishes them and the new step count. st has 9 doubles here: [8] is the
// CTA counter (as u32). Saves one launch per step.
__device__ __forceinline__ void adam_scalars(const double* st, double* s_sc) {
    // L2 loads: the step count was published by another SM's CTA of the previous optimiser launch
    const double step = __ldcg(st + 4) + 1.0;
    s_sc[0] = step;
    double p1, p2;
    beta_powers(__ldcg(st + 1), __ldcg(st + 2), step, p1, p2);
    s_sc[1] = __ldcg(st + 0) / (1.0 - p1);
    s_sc[2] = sqrt(1.0 - p2);
}
__device__ __forceinline__ void adam_publish(double* st, const double* s_sc) {   // called by thread 0 of every CTA after its work
    __threadfence();
    unsigned int* ctr = reinterpret_cast<unsigned int*>(st + 8);
    if (atomicAdd(ctr, 1u) == gridDim.x - 1) {
        st[4] = s_sc[0]; st[6] = s_sc[1]; st[7] = s_sc[2];
        *ctr = 0u;
    }
}

struct AdamK { float w1, b2, w2, eps, gs, neg_step, bc2s; };
__device__ __forceinline__ AdamK adam_consts(const double* st, double step_size, double bc2_sqrt) {
    // the f64 scalars are rounded to f32 exactly where ATen rounds its Scalar arguments
    return AdamK{(float)(1.0 - st[1]), (float)st[2], (float)(1.0 - st[2]), (float)st[3], (float)st[5], (float)(-step_size), (float)bc2_sqrt};
}
__device__ __forceinline__ void adam4(float4& pp, float4 gg, float4& mm, float4& vv, const AdamK& k) {
    float* P = &pp.x; float* G = &gg.x; float* M = &mm.x; float* V = &vv.x;
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        const float gk = G[q] * k.gs;                              // grad_scale folds the DDP 1/world mean
        M[q] = __fmaf_rn(k.w1, gk - M[q], M[q]);                   // exp_avg.lerp_(grad, 1 - beta1), weight < 0.5 branch
        V[q] = __fmaf_rn(k.w2 * gk, gk, V[q] * k.b2);              // exp_avg_sq.mul_(beta2).addcmul_(g, g, value=1 - beta2)
        const float denom = __fadd_rn(__fdiv_rn(__fsqrt_rn(V[q]), k.bc2s), k.eps);   // (sqrt(v) / bc2_sqrt).add_(eps)
        P[q] = __fmaf_rn(k.neg_step, __fdiv_rn(M[q], denom), P[q]);                  // addcdiv_(m, denom, value=-step_size)
    }
}

// tick + update (+ refresh of the bf16 MMA operand images of the weights just updated, pm.base != nullptr: bf16 mode --
// the step then needs no separate pack launch)
__global__ void __launch_bounds__(256) adam_tick_step_kernel(float4* __restrict__ p, const float4* __restrict__ g,
                                                             float4* __restrict__ m, float4* __restrict__ v,
                                                             double* __restrict__ st, int64_t n4, const ctc::PackMap pm) {
    __shared__ double s_sc[3];
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    // Parameters, moments and the step scalars were last written by the PREVIOUS optimiser launch (or by ordinary launches
    // before it), and a launch that writes them releases its dependents only after its last write: they are fetched here,
    // before the dependency wait, under the gradient reduction that precedes this kernel. Only the gradients wait.
    // (L2 loads: no L1 line of an earlier launch on this SM can be served.)
    const float4 z4 = make_float4(0.f, 0.f, 0.f, 0.f);
    float4 pp = z4, mm = z4, vv = z4, gg = z4;
    if (i < n4) { pp = __ldcg(p + i); mm = __ldcg(m + i); vv = __ldcg(v + i); }
    if (threadIdx.x == 0) adam_scalars(st, s_sc);
    bc::pdl_wait();
    if (i < n4) gg = g[i];
    __syncthreads();
    const AdamK k = adam_consts(st, s_sc[1], s_sc[2]);
    while (i < n4) {
        adam4(pp, gg, mm, vv, k);
        p[i] = pp; m[i] = mm; v[i] = vv;
        ctc::pack_updated4(pm, 4 * i, &pp.x);
        i += stride;
        if (i < n4) { pp = __ldcg(p + i); mm = __ldcg(m + i); vv = __ldcg(v + i); gg = g[i]; }
    }
    __syncthreads();
    if (threadIdx.x == 0) adam_publish(st, s_sc);
    // writer of the parameters / operand images: dependents are released only after the last write (the conv and head kernels
    // fetch their weights BEFORE their own griddepcontrol.wait)
    __threadfence();
    bc::pdl_trigger();
}

__global__ void __launch_bounds__(256) adam_kernel(float4* __restrict__ p, const float4* __restrict__ g,
                                                   float4* __restrict__ m, float4* __restrict__ v,
                                                   const double* __restrict__ st, int64_t n4) {
    bc::pdl_wait();
    const AdamK k = adam_consts(st, st[6], st[7]);
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += stride) {
        float4 pp = p[i], mm = m[i], vv = v[i];
        adam4(pp, g[i], mm, vv, k);
        p[i] = pp; m[i] = mm; v[i] = vv;
    }
    // writer of the parameters / operand images: dependents are released only after the last write (the conv and head kernels
    // fetch their weights BEFORE their own griddepcontrol.wait)
    __threadfence();
    bc::pdl_trigger();
}

// ---- K11 + K10 fused: the data-parallel gradient exchange inside the Adam step, over NVLink peer memory -------------
// Every rank's gradients live in a symmetric allocation that all ranks map (torch symmetric memory, i.e. cudaIpc /
// fabric handles: plumbing): TWO arenas per rank, step e writes and exchanges arena (e & 1). One kernel per rank and
// bucket ([fc..conv2] = bucket 0, conv1 = bucket 1; SURVEY 8e):
//   A  announce "bucket b of my gradients of epoch e is complete" in every peer's signal pad, wait for every peer's;
//   B  read that bucket of all `world` arenas straight from peer memory, add them in RANK ORDER (so every rank computes
//      bitwise the same sum and the replicas never drift), scale by grad_scale = 1/world, apply Adam to the local replica
//      (and refresh the bf16 operand images of the weights just updated);
//   C  (publishing launch only) the last CTA publishes the epoch and the Adam step scalars.
// There is no "done reading" handshake: a rank overwrites arena (e & 1) again at step e + 2, and by then it has seen every
// peer's announcement of epoch e + 1, which a peer makes only after its own exchange kernels of epoch e have finished.
// Bucket 0 is launched on a side stream as soon as [fc..conv2] are reduced and runs UNDER conv1's wgrad (the longest
// backward kernel); only the 12.6 KB conv1 bucket stays on the critical path. No separate all-reduce launch, no host
// involvement, CUDA-graph capturable. Waits are bounded by wall-clock time; a failed wait leaves the parameters untouched.
__device__ __forceinline__ void st_release_sys(uint32_t* p, uint32_t v) {
    asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ uint32_t ld_acquire_sys(const uint32_t* p) {
    uint32_t v;
    asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ float4 ld_relaxed_sys_f4(const float4* p) {
    float4 v;
    asm volatile("ld.relaxed.sys.global.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ uint64_t globaltimer_ns() {
    uint64_t t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}
__device__ bool wait_epoch(const uint32_t* flag, uint32_t epoch, int* err) {
    const uint64_t t0 = globaltimer_ns();
    while ((int32_t)(ld_acquire_sys(flag) - epoch) < 0) {
        if (globaltimer_ns() - t0 > 20000000000ull) {       // 20 s: a peer died or the ranks disagree on the step count
            if (err) atomicExch(err, 2);
            return false;
        }
        __nanosleep(100);
    }
    return true;
}

constexpr int kSigReady = 256;                               // u32 word offset inside a rank's signal pad: [bucket][64 ranks]

struct ExchangeArgs {
    float4* p; const float4* const* peer_grads; uint32_t* const* peer_signals; float4* m; float4* v; double* st;
    uint32_t* sync;             // [0] completed epochs, [1] CTA counter of the publishing launch
    int64_t lo4, hi4, arena4;   // float4 range of this bucket; float4 length of one arena (parity stride)
    int rank, world, bucket, publish;
    int* err;
    ctc::PackMap pm;
};
// Two arenas in one exchange (bc_adam_step_exchange_arenas): each half of the gradient buffer is [arena 0 | arena 1];
// float4 i < split4 belongs to arena 0 (p, m, v, st above; the operand images follow it), the rest to arena 1.
struct ExchangeArgs2 : ExchangeArgs {
    float4* p2; float4* m2; float4* v2; double* st2;
    int64_t split4;
};
template <int NSEG> using ExchangeArgsN = std::conditional_t<NSEG == 1, ExchangeArgs, ExchangeArgs2>;

template <int NSEG>
__global__ void __launch_bounds__(128) adam_exchange_kernel(const ExchangeArgsN<NSEG> a) {
    __shared__ int s_last;
    __shared__ double s_sc[3 * NSEG];
    bc::pdl_wait();                                         // no early release of the dependents: this kernel writes the parameters (see adam_tick_step_kernel)
    if (threadIdx.x == 0) {                                 // the tick is folded in (published by the last CTA of the publishing launch)
        adam_scalars(a.st, s_sc);
        if constexpr (NSEG == 2) adam_scalars(a.st2, s_sc + 3);
    }
    const uint32_t epoch = a.sync[0] + 1;
    const int64_t par = (int64_t)(epoch & 1u) * a.arena4;
    uint32_t* my_sig = a.peer_signals[a.rank];
    // ---- A
    int ok = *reinterpret_cast<volatile int*>(a.err) == 0;  // an earlier failed wait: do nothing any more
    if (ok && blockIdx.x == 0 && threadIdx.x < a.world) {
        __threadfence_system();
        st_release_sys(a.peer_signals[threadIdx.x] + kSigReady + a.bucket * 64 + a.rank, epoch);
    }
    if (ok && threadIdx.x < a.world) ok = wait_epoch(my_sig + kSigReady + a.bucket * 64 + threadIdx.x, epoch, a.err);
    ok = __syncthreads_and(ok);
    if (!ok) return;                                        // parameters, moments, step count and epoch stay as they were
    // ---- B
    const AdamK k = adam_consts(a.st, s_sc[1], s_sc[2]);
    AdamK k2 = k;
    if constexpr (NSEG == 2) k2 = adam_consts(a.st2, s_sc[4], s_sc[5]);
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = a.lo4 + (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < a.hi4; i += stride) {
        float4 *p = a.p, *m = a.m, *v = a.v;
        int64_t j = i;
        bool first = true;
        if constexpr (NSEG == 2) {
            if (i >= a.split4) { p = a.p2; m = a.m2; v = a.v2; j = i - a.split4; first = false; }
        }
        float4 pp = p[j], mm = m[j], vv = v[j];                     // local state first: in flight under the NVLink round trips
        float4 gg = ld_relaxed_sys_f4(a.peer_grads[0] + par + i);
        for (int r = 1; r < a.world; ++r) {
            const float4 o = ld_relaxed_sys_f4(a.peer_grads[r] + par + i);
            gg.x = __fadd_rn(gg.x, o.x); gg.y = __fadd_rn(gg.y, o.y); gg.z = __fadd_rn(gg.z, o.z); gg.w = __fadd_rn(gg.w, o.w);
        }
        adam4(pp, gg, mm, vv, first ? k : k2);
        p[j] = pp; m[j] = mm; v[j] = vv;
        if (first) ctc::pack_updated4(a.pm, 4 * i, &pp.x);          // the operand images belong to arena 0 only
    }
    // ---- C
    if (!a.publish) return;
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence();
        s_last = atomicAdd(a.sync + 1, 1u) == gridDim.x - 1;
    }
    __syncthreads();
    if (s_last && threadIdx.x == 0) {
        if constexpr (NSEG == 2) { a.st2[4] = s_sc[3]; a.st2[6] = s_sc[4]; a.st2[7] = s_sc[5]; }
        a.sync[1] = 0; a.sync[0] = epoch; a.st[4] = s_sc[0]; a.st[6] = s_sc[1]; a.st[7] = s_sc[2];
    }
    // early returns above release the dependents implicitly when the grid completes
}

}  // namespace

extern "C" {

const char* bc_last_error_string(void) { return bc::err_buf(); }
int bc_abi_version(void) { return 2; }

int bc_device_check(void) {
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return bc::fail(BC_ERR_DEVICE, "no CUDA device: %s (there is no CPU fallback)", cudaGetErrorString(e));
    int major = 0, minor = 0;
    cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev);
    cudaDeviceGetAttribute(&minor, cudaDevAttrComputeCapabilityMinor, dev);
    if (major != 10) return bc::fail(BC_ERR_DEVICE, "device %d is sm_%d%d; this library is built for sm_100a only", dev, major, minor);
    return BC_OK;
}

int64_t bc_arena_layout(int obs_size, int n_actions, int64_t offsets[14], int64_t sizes[14]) {
    const bc::Arena a = bc::arena_layout(obs_size, n_actions);
    for (int l = 0; l < 7; ++l) {
        offsets[2 * l] = a.w[l]; sizes[2 * l] = a.nw[l];
        offsets[2 * l + 1] = a.b[l]; sizes[2 * l + 1] = a.nb[l];
    }
    return a.total;
}

size_t bc_partials_floats(int obs_size, int n_actions) {
    return (size_t)bc::partials_layout(bc::arena_layout(obs_size, n_actions)).total;
}

int bc_forward(const bc_ctx* c, void* stream) {
    for (int l = 0; l < 4; ++l) {
        int rc = bc_conv_relu_pool_fwd(c, l, stream);
        if (rc) return rc;
    }
    return bc_head(c, 0, stream);
}

int bc_forward_act(const bc_ctx* c, int64_t* actions, int tail, void* stream) {
    BC_CHECK_ARG(c && actions, "bc_forward_act: null ctx / actions");
    for (int l = 0; l < (tail ? 2 : 4); ++l) {
        int rc = bc_conv_relu_pool_fwd(c, l, stream);
        if (rc) return rc;
    }
    return tail ? bc_policy_tail(c, actions, stream) : bc_head_launch(c, 0, actions, stream);
}

int bc_backward(const bc_ctx* c, int with_loss, void* stream) {
    BC_CHECK_ARG(c, "bc_backward: null ctx");
    // head: (CE from labels when with_loss, else the caller's dlogits) + MLP backward -> ghead
    int rc = bc_head(c, with_loss ? 3 : 2, stream);
    if (rc) return rc;
    for (int l = 3; l >= 1; --l) {
        rc = bc_conv_bwd_wgrad(c, l, stream);
        if (!rc) rc = bc_conv_bwd_dgrad(c, l, stream);
        if (rc) return rc;
    }
    if ((rc = bc_conv_bwd_wgrad(c, 0, stream))) return rc;
    return bc_reduce_partials(c, with_loss, stream);
}

int bc_adam_tick(double* state, void* stream) {
    BC_CHECK_ARG(state, "bc_adam_tick: null state");
    bc::launch_pdl(adam_tick_kernel, dim3(1), dim3(1), 0, (cudaStream_t)stream, state);
    BC_CUDA_LAUNCH_CHECK("adam_tick_kernel");
    return BC_OK;
}

int bc_adam_step(float* params, const float* grads, float* exp_avg, float* exp_avg_sq, const double* state,
                 int64_t n, void* stream) {
    BC_CHECK_ARG(params && grads && exp_avg && exp_avg_sq && state, "bc_adam_step: null pointer");
    BC_CHECK_ARG(n >= 0 && n % 4 == 0, "bc_adam_step: n=%lld must be a multiple of 4 (the arena is padded)", (long long)n);
    BC_CHECK_ARG(((uintptr_t)params | (uintptr_t)grads | (uintptr_t)exp_avg | (uintptr_t)exp_avg_sq) % 16 == 0, "bc_adam_step: 16 B alignment");
    if (n == 0) return BC_OK;
    const int64_t n4 = n / 4;
    int blocks = (int)((n4 + 255) / 256);
    const int cap = bc::num_sms() * 8;
    if (blocks > cap) blocks = cap;
    bc::launch_pdl(adam_kernel, dim3(blocks), dim3(256), 0, (cudaStream_t)stream, (float4*)params, (const float4*)grads, (float4*)exp_avg,
                   (float4*)exp_avg_sq, state, n4);
    BC_CUDA_LAUNCH_CHECK("adam_kernel");
    return BC_OK;
}

static int pack_map_for(ctc::PackMap* pm, void* w_packed, int obs_size, int n_actions, int64_t n, const char* who) {
    *pm = ctc::PackMap{nullptr, 0, 0, 0, 0, 0};
    if (!w_packed) return BC_OK;
    if (obs_size != 4 && obs_size != 12) return bc::fail(BC_ERR_ARG, "%s: the bf16 operand images exist for obs_size 4 and 12 (got %d)", who, obs_size);
    const bc::Arena a = bc::arena_layout(obs_size, n_actions);
    if (a.total != n) return bc::fail(BC_ERR_ARG, "%s: n=%lld is not the arena of (obs %d, actions %d) = %lld floats", who, (long long)n, obs_size, n_actions, (long long)a.total);
    if ((uintptr_t)w_packed % 16 != 0) return bc::fail(BC_ERR_ARG, "%s: w_packed must be 16 B aligned", who);
    *pm = ctc::pack_map(a, w_packed, obs_size);
    return BC_OK;
}

int bc_adam_tick_step(float* params, const float* grads, float* exp_avg, float* exp_avg_sq, double* state9, int64_t n,
                      void* w_packed, int obs_size, int n_actions, void* stream) {
    BC_CHECK_ARG(params && grads && exp_avg && exp_avg_sq && state9, "bc_adam_tick_step: null pointer");
    BC_CHECK_ARG(n >= 0 && n % 4 == 0, "bc_adam_tick_step: n=%lld must be a multiple of 4 (the arena is padded)", (long long)n);
    BC_CHECK_ARG(((uintptr_t)params | (uintptr_t)grads | (uintptr_t)exp_avg | (uintptr_t)exp_avg_sq) % 16 == 0, "bc_adam_tick_step: 16 B alignment");
    ctc::PackMap pm;
    if (int rc = pack_map_for(&pm, w_packed, obs_size, n_actions, n, "bc_adam_tick_step")) return rc;
    const int64_t n4 = n / 4;
    int blocks = (int)((n4 + 255) / 256);
    const int cap = bc::num_sms() * 8;
    if (blocks > cap) blocks = cap;
    if (blocks < 1) blocks = 1;                               // n == 0 still ticks
    bc::launch_pdl(adam_tick_step_kernel, dim3(blocks), dim3(256), 0, (cudaStream_t)stream, (float4*)params, (const float4*)grads,
                   (float4*)exp_avg, (float4*)exp_avg_sq, state9, n4, pm);
    BC_CUDA_LAUNCH_CHECK("adam_tick_step_kernel");
    return BC_OK;
}

int bc_adam_step_exchange(float* params, float* exp_avg, float* exp_avg_sq, double* state9, int64_t n, const bc_peer* peer,
                          int64_t lo, int64_t hi, int bucket, int publish, void* w_packed, int obs_size, int n_actions, void* stream) {
    BC_CHECK_ARG(params && exp_avg && exp_avg_sq && state9 && peer, "bc_adam_step_exchange: null pointer");
    BC_CHECK_ARG(peer->peer_grads_dev && peer->peer_signals_dev && peer->sync_state && peer->err_flag, "bc_adam_step_exchange: null pointer in bc_peer");
    BC_CHECK_ARG(n > 0 && n % 4 == 0, "bc_adam_step_exchange: n=%lld must be a positive multiple of 4", (long long)n);
    BC_CHECK_ARG(0 <= lo && lo < hi && hi <= n && lo % 4 == 0 && hi % 4 == 0, "bc_adam_step_exchange: bucket [%lld,%lld) outside the arena or not a multiple of 4", (long long)lo, (long long)hi);
    BC_CHECK_ARG(bucket == 0 || bucket == 1, "bc_adam_step_exchange: bucket %d (0 = [fc..conv2], 1 = conv1 or the whole arena)", bucket);
    BC_CHECK_ARG(peer->world >= 1 && peer->world <= 64 && peer->rank >= 0 && peer->rank < peer->world, "bc_adam_step_exchange: rank %d of %d", peer->rank, peer->world);
    ExchangeArgs a{};
    if (int rc = pack_map_for(&a.pm, w_packed, obs_size, n_actions, n, "bc_adam_step_exchange")) return rc;
    a.p = (float4*)params; a.peer_grads = (const float4* const*)peer->peer_grads_dev; a.peer_signals = (uint32_t* const*)peer->peer_signals_dev;
    a.m = (float4*)exp_avg; a.v = (float4*)exp_avg_sq; a.st = state9; a.sync = peer->sync_state;
    a.lo4 = lo / 4; a.hi4 = hi / 4; a.arena4 = n / 4;
    a.rank = peer->rank; a.world = peer->world; a.bucket = bucket; a.publish = publish; a.err = peer->err_flag;
    int blocks = (int)((a.hi4 - a.lo4 + 127) / 128);           // one float4 per thread: a single NVLink round trip per thread
    const int cap = 2 * bc::num_sms();                         // every CTA spins on the flags: all of them must be resident
    if (blocks > cap) blocks = cap;
    bc::launch_pdl(adam_exchange_kernel<1>, dim3(blocks), dim3(128), 0, (cudaStream_t)stream, a);
    BC_CUDA_LAUNCH_CHECK("adam_exchange_kernel");
    return BC_OK;
}

int bc_adam_step_exchange_arenas(float* params, float* exp_avg, float* exp_avg_sq, double* state9,
                                 float* params_b, float* exp_avg_b, float* exp_avg_sq_b, double* state9_b,
                                 int64_t n, int64_t split, const bc_peer* peer, void* w_packed, int obs_size, int n_actions,
                                 void* stream) {
    BC_CHECK_ARG(params && exp_avg && exp_avg_sq && state9 && params_b && exp_avg_b && exp_avg_sq_b && state9_b && peer,
                 "bc_adam_step_exchange_arenas: null pointer");
    BC_CHECK_ARG(peer->peer_grads_dev && peer->peer_signals_dev && peer->sync_state && peer->err_flag, "bc_adam_step_exchange_arenas: null pointer in bc_peer");
    BC_CHECK_ARG(n > 0 && n % 4 == 0, "bc_adam_step_exchange_arenas: n=%lld must be a positive multiple of 4", (long long)n);
    BC_CHECK_ARG(0 < split && split < n && split % 4 == 0, "bc_adam_step_exchange_arenas: split %lld outside (0, %lld) or not a multiple of 4", (long long)split, (long long)n);
    BC_CHECK_ARG(peer->world >= 1 && peer->world <= 64 && peer->rank >= 0 && peer->rank < peer->world, "bc_adam_step_exchange_arenas: rank %d of %d", peer->rank, peer->world);
    BC_CHECK_ARG(((uintptr_t)params | (uintptr_t)exp_avg | (uintptr_t)exp_avg_sq | (uintptr_t)params_b | (uintptr_t)exp_avg_b |
                  (uintptr_t)exp_avg_sq_b) % 16 == 0, "bc_adam_step_exchange_arenas: 16 B alignment");
    ExchangeArgs2 a{};
    if (int rc = pack_map_for(&a.pm, w_packed, obs_size, n_actions, split, "bc_adam_step_exchange_arenas")) return rc;
    a.p = (float4*)params; a.peer_grads = (const float4* const*)peer->peer_grads_dev; a.peer_signals = (uint32_t* const*)peer->peer_signals_dev;
    a.m = (float4*)exp_avg; a.v = (float4*)exp_avg_sq; a.st = state9; a.sync = peer->sync_state;
    a.p2 = (float4*)params_b; a.m2 = (float4*)exp_avg_b; a.v2 = (float4*)exp_avg_sq_b; a.st2 = state9_b; a.split4 = split / 4;
    a.lo4 = 0; a.hi4 = n / 4; a.arena4 = n / 4;
    a.rank = peer->rank; a.world = peer->world; a.bucket = 1; a.publish = 1; a.err = peer->err_flag;
    int blocks = (int)((a.hi4 + 127) / 128);                   // one float4 per thread, as above
    const int cap = 2 * bc::num_sms();                         // every CTA spins on the flags: all of them must be resident
    if (blocks > cap) blocks = cap;
    bc::launch_pdl(adam_exchange_kernel<2>, dim3(blocks), dim3(128), 0, (cudaStream_t)stream, a);
    BC_CUDA_LAUNCH_CHECK("adam_exchange_kernel");
    return BC_OK;
}

// ---- the backward pass with the weight-gradient kernels of conv4..conv2 on a side stream -----------------------------
// main:  head -> dgrad4 -> dgrad3 -> dgrad2 -> conv1 wgrad ------------------------> [join] reduce
// side:          wgrad4 (after head) -> wgrad3 (after dgrad4) -> wgrad2 (after dgrad3) --^
// wgrad(l) and dgrad(l) both depend only on the gradient of layer l's output, so the dgrad chain (the critical path to
// conv1's wgrad) no longer waits for the weight gradients. ev[0..3]: caller-owned events (fork x3, join). Capturable.
static int record_wait(void* ev, void* on, void* waiter) {
    cudaError_t e = cudaEventRecord((cudaEvent_t)ev, (cudaStream_t)on);
    if (e == cudaSuccess) e = cudaStreamWaitEvent((cudaStream_t)waiter, (cudaEvent_t)ev, 0);
    if (e != cudaSuccess) return bc::fail(BC_ERR_DEVICE, "bc_backward_overlap: event fork/join failed: %s", cudaGetErrorString(e));
    return BC_OK;
}

int bc_backward_overlap(const bc_ctx* c, int with_loss, void* stream, void* side_stream, void* const* ev, int flags) {
    BC_CHECK_ARG(c && side_stream && ev && ev[0] && ev[1] && ev[2] && ev[3], "bc_backward_overlap: null ctx / side stream / events");
    BC_CHECK_ARG(side_stream != stream, "bc_backward_overlap: the side stream must differ from the main stream");
    const bool dp_split = flags & 1, wgrad_main = flags & 2;
    int rc = bc_head(c, with_loss ? 3 : 2, stream);
    if (rc) return rc;
    for (int l = 3; l >= 1; --l) {
        if (wgrad_main) {
            if ((rc = bc_conv_bwd_wgrad(c, l, stream))) return rc;
        } else {
            if ((rc = record_wait(ev[3 - l], stream, side_stream))) return rc;     // the gradient of layer l's output is complete
            if ((rc = bc_conv_bwd_wgrad(c, l, side_stream))) return rc;
        }
        if ((rc = bc_conv_bwd_dgrad(c, l, stream))) return rc;
    }
    if (dp_split) {
        // data-parallel overlap: [fc..conv2] are reduced on the side stream as soon as conv2's wgrad is done; the caller
        // launches the bucket-0 exchange there, then joins (ev[3]) and reduces conv1 on the main stream
        if (wgrad_main && (rc = record_wait(ev[0], stream, side_stream))) return rc;   // everything up to conv2's dgrad (and wgrad) is enqueued
        if ((rc = bc_reduce_partials_range(c, 0, 4, with_loss, side_stream))) return rc;
        return bc_conv_bwd_wgrad(c, 0, stream);
    }
    if ((rc = bc_conv_bwd_wgrad(c, 0, stream))) return rc;
    if (!wgrad_main && (rc = record_wait(ev[3], side_stream, stream))) return rc;
    return bc_reduce_partials(c, with_loss, stream);
}

}  // extern "C"
