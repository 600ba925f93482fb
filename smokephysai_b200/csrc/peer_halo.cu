// peer_halo.cu -- the slab halo exchange (SURVEY.md s8e) as direct peer stores over NVLink, and the phase-kernel step that whole
// grids (abi.cu's run_steps) and row slabs (smk_slab_step) share.
//
// Why.  A row slab of an 8192 x 8192 grid on eight GPUs runs ~250 us of kernels per step; the ncclSend / ncclRecv group of
// nccl_halo.cu costs ~85 us of stream time per exchange for ~10 us of data (NCCL's proxy and FIFO protocol are built for
// big messages), and issuing the step's ten launches from Python costs more host time than the kernels take.  Here:
//
//   * every rank owns a MAILBOX (device memory, exported once with CUDA IPC and mapped by its two neighbours): per neighbour two
//     slots (exchange number & 1) of four field regions (u, v, density, p ghost rows), and one arrival counter per neighbour;
//   * k_halo_push copies this rank's boundary rows straight into the neighbours' mailboxes with 16-byte peer stores; the last CTA to
//     finish fences at system scope and bumps the neighbours' counters with st.release.sys;
//   * k_halo_unpack spins (ld.acquire.sys, one thread per CTA) until both counters show this exchange, then copies the mailbox
//     slots into the slab's ghost rows.  Two small kernels, ~6 MB each way at eight slabs, no host round trip, no proxy thread.
//
// Two slots are enough without any "slot free" handshake: a rank can only be in exchange n after it completed exchange n - 1, which
// needed its neighbour's push n - 1, which that neighbour issued (stream order) after its own unpack n - 2 -- the last reader of the
// slot exchange n overwrites.  Counters only grow, so nothing is ever reset between steps or after setup_grid().
//
// Both kernels read the exchange number from device memory (seq[0]), not from a launch argument: a captured CUDA graph of the step
// replays correctly.  smk_slab_step issues the exchange, then phase_step: forces/diffusion/divergence + the Jacobi launches +
// gradient subtract + the three advections, from one C call; the results are those of the phase entry points called one by one
// (same launchers).
#include <cuda.h>
#include <cstring>
#include "common.cuh"

namespace smk {

struct HxCopy { const float4* src; float4* dst; long long n4; int parity_on_dst; };
struct HxArgs {
    HxCopy c[8];
    int n;
    long long parity_stride4;           // float4 between the two slots of a mailbox region
    unsigned* flag[2];                  // push: the neighbours' counters to bump; unpack: this rank's counters to wait for
    unsigned* seq;                      // seq[0]: exchanges completed by this rank, seq[1]: CTA tickets of the running kernel
    unsigned long long timeout_ns;      // wall-clock budget of the wait in unpack
};

__device__ __forceinline__ unsigned hx_ld_acquire_sys(const unsigned* p)
{
    unsigned v;
    asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void hx_st_release_sys(unsigned* p, unsigned v)
{
    asm volatile("st.release.sys.global.u32 [%0], %1;" :: "l"(p), "r"(v) : "memory");
}

// blockIdx.y = copy, blockIdx.x strides over it.  PUSH: local rows -> the neighbour's mailbox slot, then publish.
// !PUSH: wait for the neighbours' publications, mailbox slot -> local ghost rows, then count the exchange as done.
template <bool PUSH>
__global__ void __launch_bounds__(256)
k_halo_xfer(const HxArgs a)
{
    pdl_prologue();
    __shared__ unsigned s_seq;
    if (threadIdx.x == 0) {
        const unsigned seq = *reinterpret_cast<volatile const unsigned*>(a.seq);
        if (!PUSH) {
            unsigned long long t0 = 0;
            for (int k = 0; k < 2; ++k)
                if (a.flag[k])
                    while ((int)(hx_ld_acquire_sys(a.flag[k]) - (seq + 1u)) < 0) {      // wrap-safe "counter < seq + 1"
                        __nanosleep(200);
                        unsigned long long now;
                        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(now));
                        if (t0 == 0) t0 = now;
                        // the neighbour never pushed (it died, or the ranks disagree on the exchange sequence): fail the launch
                        // after timeout_ns of wall-clock time instead of hanging the GPU
                        if (now - t0 > a.timeout_ns) __trap();
                    }
        }
        s_seq = seq;
    }
    __syncthreads();
    const long long poff = (long long)(s_seq & 1u) * a.parity_stride4;
    const HxCopy c = a.c[blockIdx.y];
    const float4* __restrict__ src = c.src + (c.parity_on_dst ? 0 : poff);
    float4* __restrict__ dst = c.dst + (c.parity_on_dst ? poff : 0);
    // four independent 16-byte loads in flight per thread (a copy is ~50 k of them at eight slabs of 8192 columns: latency, not
    // bandwidth, is what a short copy pays).  The mailbox is written by another GPU: it is never read through this SM's L1.
    const long long stride = (long long)gridDim.x * 256;
    long long k = (long long)blockIdx.x * 256 + threadIdx.x;
    for (; k + 3 * stride < c.n4; k += 4 * stride) {
        const float4 v0 = __ldcg(src + k), v1 = __ldcg(src + k + stride), v2 = __ldcg(src + k + 2 * stride), v3 = __ldcg(src + k + 3 * stride);
        dst[k] = v0; dst[k + stride] = v1; dst[k + 2 * stride] = v2; dst[k + 3 * stride] = v3;
    }
    for (; k < c.n4; k += stride) dst[k] = __ldcg(src + k);
    // last CTA out: publish (push) / count the exchange (unpack)
    if (PUSH) __threadfence_system();
    __syncthreads();
    if (threadIdx.x == 0) {
        const unsigned total = gridDim.x * gridDim.y;
        const unsigned ticket = atomicAdd(a.seq + 1, 1u);
        if (ticket == total - 1) {
            __threadfence();                                // every other CTA's stores and fences happen-before this point
            a.seq[1] = 0;
            if (PUSH) {
                __threadfence_system();
                for (int k = 0; k < 2; ++k)
                    if (a.flag[k]) hx_st_release_sys(a.flag[k], s_seq + 1u);
            } else {
                a.seq[0] = s_seq + 1u;
            }
        }
    }
}

static int build_args(const smk_peer_comm_t* c, float* const* base, bool push, HxArgs* out, const char* who)
{
    if (!c || !base) return fail(SMK_EINVAL, "%s: NULL", who);
    if (!c->seq || (c->parity_stride & 3) || (c->field_stride & 3) || c->parity_stride < 4 * c->field_stride)
        return fail(SMK_EINVAL, "%s: bad mailbox strides (field %lld, parity %lld) or seq NULL", who, (long long)c->field_stride, (long long)c->parity_stride);
    HxArgs a;
    memset(&a, 0, sizeof a);
    a.parity_stride4 = c->parity_stride / 4;
    a.seq = c->seq;
    a.timeout_ns = 20ull * 1000000000ull;                    // 20 s: ranks may start seconds apart; a dead neighbour fails the launch
    for (int l = 0; l < 2; ++l) {
        const smk_peer_link_t& k = c->link[l];
        if (!k.remote_mailbox) continue;                     // no neighbour on this side
        if (!k.local_mailbox || !k.remote_flag || !k.local_flag) return fail(SMK_EINVAL, "%s: link %d is half wired", who, l);
        a.flag[l] = push ? k.remote_flag : k.local_flag;
        for (int f = 0; f < 4; ++f) {
            if (!base[f]) continue;
            const int64_t n = push ? k.send_count[f] : k.recv_count[f], off = push ? k.send_off[f] : k.recv_off[f];
            if (n == 0) continue;
            if (n < 0 || (n & 3) || (off & 3) || off < 0 || n > c->field_stride || !aligned16(base[f]))
                return fail(SMK_EINVAL, "%s: link %d field %d: offset %lld / count %lld not a multiple of 4, negative, or larger than a mailbox region",
                            who, l, f, (long long)off, (long long)n);
            HxCopy& cp = a.c[a.n++];
            float* box = (push ? k.remote_mailbox : k.local_mailbox) + (int64_t)f * c->field_stride;
            cp.src = reinterpret_cast<const float4*>(push ? base[f] + off : box);
            cp.dst = reinterpret_cast<float4*>(push ? box : base[f] + off);
            cp.n4 = n / 4;
            cp.parity_on_dst = push ? 1 : 0;
        }
    }
    *out = a;
    return SMK_OK;
}

static int peer_xfer(const smk_peer_comm_t* c, float* const* base, bool push, cudaStream_t s)
{
    HxArgs a;
    const int rc = build_args(c, base, push, &a, push ? "smk_peer_push" : "smk_peer_unpack");
    if (rc != SMK_OK) return rc;
    if (a.n == 0) return SMK_OK;                             // no neighbour at all (world of one)
    long long most = 0;
    for (int k = 0; k < a.n; ++k) most = most > a.c[k].n4 ? most : a.c[k].n4;
    int per = (int)((most + 256 * 4 - 1) / (256 * 4));       // four 16-byte elements per thread
    per = per < 1 ? 1 : (per > 32 ? 32 : per);               // at most 8 x 32 = 256 CTAs of 256 threads: all co-resident (2 per SM)
    ProfScope prof_(push ? SMK_PH_HALO : SMK_PH_HALO_UNPACK, s);      // the unpack's time includes the wait for the slower neighbour
    if (push) launch_chain(k_halo_xfer<true>, dim3(per, a.n), dim3(256), 0, s, a);
    else      launch_chain(k_halo_xfer<false>, dim3(per, a.n), dim3(256), 0, s, a);
    return check_launch(push ? "k_halo_push" : "k_halo_unpack");
}

// The push a step issues for the NEXT step (SMK_SLAB_PUSH_TAIL) runs on a stream of its own, next to the rest of the density
// advection: forked from the caller's stream after the boundary bands (ev_fork), joined at the head of the next step (ev_join,
// which also keeps the push's reads of p ahead of that step's Jacobi launches).  One set per device; highest stream priority, so
// the push's CTAs are placed as soon as CTAs of the advection retire.
struct SideStream { cudaStream_t s; cudaEvent_t ev_fork, ev_join; bool ok, pending; };
static SideStream* side_stream()
{
    static SideStream side[64] = {};
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return nullptr;
    SideStream& x = side[dev];
    if (!x.ok) {
        int lo = 0, hi = 0;
        if (cudaDeviceGetStreamPriorityRange(&lo, &hi) != cudaSuccess) { lo = hi = 0; }
        if (cudaStreamCreateWithPriority(&x.s, cudaStreamNonBlocking, hi) != cudaSuccess ||
            cudaEventCreateWithFlags(&x.ev_fork, cudaEventDisableTiming) != cudaSuccess ||
            cudaEventCreateWithFlags(&x.ev_join, cudaEventDisableTiming) != cudaSuccess) {
            (void)cudaGetLastError();
            return nullptr;
        }
        x.ok = true;
    }
    return &x;
}

typedef CUresult (*hx_range_fn)(CUdeviceptr*, size_t*, CUdeviceptr);
static hx_range_fn hx_range()
{
    static hx_range_fn fn = nullptr;
    if (!fn) {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q = cudaDriverEntryPointSymbolNotFound;
        if (cudaGetDriverEntryPoint("cuMemGetAddressRange", &p, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess)
            fn = (hx_range_fn)p;
    }
    return fn;
}

}  // namespace smk

using namespace smk;

#define SMK_TRY_(x) do { const int rc_ = (x); if (rc_ != SMK_OK) return rc_; } while (0)

// The density advection of a step, writing the frame (may be NULL) as it goes, or -- slabs, no frame -- with the NEXT step's
// halo push issued from the middle of it (push_comm != NULL): the tile rows that hold the rows this rank sends to its neighbours
// are advected first (two short launches), then k_halo_push copies the boundary rows of the new u, v, density and of p into the
// neighbours' mailboxes, then the rest of the field is advected -- the NVLink transfer, the counters' flight and the neighbours'
// skew hide behind that last launch and the neighbour's own, instead of heading the next step.  new_base: the live u, v,
// density, p once this step is complete.
static int advect_density(const smk_grid_t* g, const float* d_in, float* d_out, const float* u, const float* v, const smk_params_t* prm,
                          void* frame, int64_t frame_stride, const float* fmul, int frame_format,
                          const smk_slab_check_t* chk_d, cudaStream_t s, const smk_peer_comm_t* push_comm, float* const* new_base)
{
    if (!push_comm)
        return launch_advect(g, d_in, d_out, g->h, g->w, g->pitch_c, g->stride_c, u, v, prm->dt, prm->decay, frame, frame_stride, fmul,
                             chk_d, s, 0, nullptr, nullptr, nullptr, frame_format);
    AdvectPart rest = {0, 0, {0, 0}, {0, 0}};
    int nb = 0;
    if (advect_is_tiled(g, g->h, g->w)) {
        const int TR = advect_tile_rows(), nty = (g->h + TR - 1) / TR;
        int lo[2], hi[2];
        for (int l = 0; l < 2; ++l) {
            const smk_peer_link_t& k = push_comm->link[l];
            if (!k.remote_mailbox || k.send_count[2] <= 0) continue;
            const int64_t r0 = k.send_off[2] / g->pitch_c, r1 = (k.send_off[2] + k.send_count[2] + g->pitch_c - 1) / g->pitch_c;
            int a = (int)(r0 / TR), b = (int)((r1 + TR - 1) / TR);
            a = a < 0 ? 0 : a; b = b > nty ? nty : b;
            if (a >= b) continue;
            lo[nb] = a; hi[nb] = b; ++nb;
        }
        if (nb == 2 && lo[1] < lo[0]) { int t = lo[0]; lo[0] = lo[1]; lo[1] = t; t = hi[0]; hi[0] = hi[1]; hi[1] = t; }
        if (nb == 2 && lo[1] < hi[0]) { hi[0] = hi[0] > hi[1] ? hi[0] : hi[1]; nb = 1; }          // overlapping bands: one
        for (int k = 0; k < nb; ++k) {
            const AdvectPart band = {lo[k], hi[k] - lo[k], {0, 0}, {0, 0}};
            SMK_TRY_(launch_advect(g, d_in, d_out, g->h, g->w, g->pitch_c, g->stride_c, u, v, prm->dt, prm->decay, nullptr, 0, nullptr,
                                   chk_d, s, 0, nullptr, nullptr, &band));
            rest.skip_lo[k] = lo[k]; rest.skip_n[k] = hi[k] - lo[k];
        }
    }
    if (nb == 0) {
        // small field (direct kernel) or nothing to send: advect everything, then push
        SMK_TRY_(launch_advect(g, d_in, d_out, g->h, g->w, g->pitch_c, g->stride_c, u, v, prm->dt, prm->decay, nullptr, 0, nullptr, chk_d, s));
        return peer_xfer(push_comm, new_base, true, s);
    }
    // the push on the side stream (after the bands), the rest of the advection on the caller's; SMK_PUSH_STREAM=0: one stream
    SideStream* side = env().push_stream == 0 ? nullptr : side_stream();
    if (side && cudaEventRecord(side->ev_fork, s) == cudaSuccess && cudaStreamWaitEvent(side->s, side->ev_fork, 0) == cudaSuccess) {
        SMK_TRY_(peer_xfer(push_comm, new_base, true, side->s));
        if (cudaEventRecord(side->ev_join, side->s) != cudaSuccess) return fail(SMK_EINVAL, "smk_slab_step: cudaEventRecord failed: %s", cudaGetErrorString(cudaGetLastError()));
        side->pending = true;
    } else {
        (void)cudaGetLastError();
        SMK_TRY_(peer_xfer(push_comm, new_base, true, s));
    }
    return launch_advect(g, d_in, d_out, g->h, g->w, g->pitch_c, g->stride_c, u, v, prm->dt, prm->decay, nullptr, 0, nullptr, chk_d, s,
                         0, nullptr, nullptr, &rest);
}

// The tail of a step on a grid or slab whose live u, v, density are the outputs of forces + diffusion and whose live p holds the
// K sweeps: gradient subtract (navier_stokes.py:148-149), sequential advection of u, v, density (:166-168), decay (:171), the
// frame copy (:173).  The live copies of u and density flip; so does v's, except on big fields, where the gradient subtract runs
// inside the u advection (k_advect_tiled<.., 1>, stencil.cu), the projected v passes through the spare copy and the live v ends
// where it was.
static int project_advect(const smk_grid_t* g, smk_state_t* st, const smk_params_t* prm, void* frame, int64_t frame_stride,
                          const float* fmul, int frame_format,
                          const smk_slab_check_t* chk_u, const smk_slab_check_t* chk_v, const smk_slab_check_t* chk_d,
                          const smk_peer_comm_t* push_comm, cudaStream_t s)
{
    const int cu = st->cur_u, cv = st->cur_v, cd = st->cur_d;
    float *u1 = st->u[cu], *u0 = st->u[cu ^ 1], *v1 = st->v[cv], *v0 = st->v[cv ^ 1], *d1 = st->d[cd], *d0 = st->d[cd ^ 1];
    float* pl = st->p[st->cur_p];
    if (advect_can_fuse_project(g)) {
        // u advection with the gradient subtract inside; it leaves the projected v in the spare copy v0, so the v advection runs
        // v0 -> v1 and the live v stays in the copy it was in
        SMK_TRY_(launch_advect(g, u1, u0, g->h + 1, g->w, g->pitch_u, g->stride_u, u1, v1, prm->dt, 1.0f, nullptr, 0, nullptr, chk_u, s, 1, pl, v0));
        SMK_TRY_(launch_advect(g, v0, v1, g->h, g->w + 1, g->pitch_v, g->stride_v, u0, v0, prm->dt, 1.0f, nullptr, 0, nullptr, chk_v, s));
        float* nb_[4] = {u0, v1, d0, pl};
        SMK_TRY_(advect_density(g, d1, d0, u0, v1, prm, frame, frame_stride, fmul, frame_format, chk_d, s, push_comm, nb_));
        st->cur_u = cu ^ 1; st->cur_d = cd ^ 1;
        return SMK_OK;
    }
    SMK_TRY_(launch_project(g, pl, u1, v1, prm->dt, s));
    SMK_TRY_(launch_advect(g, u1, u0, g->h + 1, g->w, g->pitch_u, g->stride_u, u1, v1, prm->dt, 1.0f, nullptr, 0, nullptr, chk_u, s));
    SMK_TRY_(launch_advect(g, v1, v0, g->h, g->w + 1, g->pitch_v, g->stride_v, u0, v1, prm->dt, 1.0f, nullptr, 0, nullptr, chk_v, s));
    float* nb_[4] = {u0, v0, d0, pl};
    SMK_TRY_(advect_density(g, d1, d0, u0, v0, prm, frame, frame_stride, fmul, frame_format, chk_d, s, push_comm, nb_));
    st->cur_u = cu ^ 1; st->cur_v = cv ^ 1; st->cur_d = cd ^ 1;
    return SMK_OK;
}

int smk::phase_step(const smk_grid_t* g, smk_state_t* st, const smk_params_t* prm, const smk_source_t* csrc, const int32_t* coff,
                    void* frame, int64_t frame_stride, const float* fmul, int frame_format,
                    const smk_slab_check_t* chk_u, const smk_slab_check_t* chk_v, const smk_slab_check_t* chk_d,
                    const smk_peer_comm_t* push_comm, cudaStream_t s)
{
    if (csrc) SMK_TRY_(launch_splat(g, st->d[st->cur_d], csrc, coff, s));     // add_smoke_source, then the step (bit-equal by construction)
    const int cu = st->cur_u, cv = st->cur_v, cd = st->cur_d;
    // 1-2. buoyancy + diffusion + divergence                                   navier_stokes.py:154-160, :136
    SMK_TRY_(launch_forces_diffuse_div(g, st->u[cu], st->v[cv], st->d[cd], st->u[cu ^ 1], st->v[cv ^ 1], st->d[cd ^ 1], st->div,
                                       prm->dt, prm->c_uv, prm->c_d, s));
    st->cur_u = cu ^ 1; st->cur_v = cv ^ 1; st->cur_d = cd ^ 1;
    // 3. Jacobi sweeps                                                         :139-145
    int flip = 0;
    SMK_TRY_(launch_jacobi(g, st->div, st->p[st->cur_p], st->p[st->cur_p ^ 1], prm->jacobi_iters, prm->sweeps_per_launch, &flip, s));
    st->cur_p ^= flip;
    // 4-5. gradient subtract + the three advections + decay + frame            :148-149, :166-173
    return project_advect(g, st, prm, frame, frame_stride, fmul, frame_format, chk_u, chk_v, chk_d, push_comm, s);
}

#define SMK_TRY(x) do { const int rc_ = (x); if (rc_ != SMK_OK) return rc_; } while (0)

extern "C" {

int smk_ipc_export(const void* ptr, void* handle64_host, int64_t* offset_host)
{
    if (!ptr || !handle64_host || !offset_host) return fail(SMK_EINVAL, "smk_ipc_export: NULL");
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "cudaIpcMemHandle_t is 64 bytes");
    hx_range_fn range = hx_range();
    if (!range) return fail(SMK_EUNSUPPORTED, "smk_ipc_export: cuMemGetAddressRange not available");
    CUdeviceptr base = 0; size_t size = 0;
    const CUresult r = range(&base, &size, (CUdeviceptr)(uintptr_t)ptr);
    if (r != CUDA_SUCCESS) return fail(SMK_EINVAL, "smk_ipc_export: not a device allocation (CUresult %d)", (int)r);
    cudaIpcMemHandle_t h;
    const cudaError_t e = cudaIpcGetMemHandle(&h, reinterpret_cast<void*>((uintptr_t)base));
    if (e != cudaSuccess) {
        (void)cudaGetLastError();
        return fail((int)e, "smk_ipc_export: cudaIpcGetMemHandle: %s (an expandable-segments allocator cannot be shared this way)", cudaGetErrorString(e));
    }
    memcpy(handle64_host, &h, sizeof h);
    *offset_host = (int64_t)((uintptr_t)ptr - (uintptr_t)base);
    return SMK_OK;
}

int smk_ipc_open(const void* handle64_host, int64_t offset, void** ptr_out_host)
{
    if (!handle64_host || !ptr_out_host || offset < 0) return fail(SMK_EINVAL, "smk_ipc_open: bad arguments");
    cudaIpcMemHandle_t h;
    memcpy(&h, handle64_host, sizeof h);
    void* base = nullptr;
    const cudaError_t e = cudaIpcOpenMemHandle(&base, h, cudaIpcMemLazyEnablePeerAccess);
    if (e != cudaSuccess) {
        (void)cudaGetLastError();
        return fail((int)e, "smk_ipc_open: cudaIpcOpenMemHandle: %s", cudaGetErrorString(e));
    }
    *ptr_out_host = static_cast<char*>(base) + offset;
    return SMK_OK;
}

int smk_ipc_close(void* ptr, int64_t offset)
{
    if (!ptr) return SMK_OK;
    const cudaError_t e = cudaIpcCloseMemHandle(static_cast<char*>(ptr) - offset);
    if (e != cudaSuccess) {
        (void)cudaGetLastError();
        return fail((int)e, "smk_ipc_close: %s", cudaGetErrorString(e));
    }
    return SMK_OK;
}

int smk_peer_push(const smk_peer_comm_t* c, float* const* field_base_host, void* stream)
{
    return peer_xfer(c, field_base_host, true, (cudaStream_t)stream);
}

int smk_peer_unpack(const smk_peer_comm_t* c, float* const* field_base_host, void* stream)
{
    return peer_xfer(c, field_base_host, false, (cudaStream_t)stream);
}

int smk_slab_step(const smk_grid_t* g, smk_state_t* st, const smk_params_t* prm, const smk_peer_comm_t* comm, int32_t flags,
                  const smk_slab_check_t* chk_u, const smk_slab_check_t* chk_v, const smk_slab_check_t* chk_d, void* stream)
{
    SMK_TRY(check_grid(g, "smk_slab_step"));
    if (!st || !prm) return fail(SMK_EINVAL, "smk_slab_step: state/params NULL");
    if (g->batch != 1) return fail(SMK_EUNSUPPORTED, "smk_slab_step: batch must be 1");
    const void* ps[] = {st->u[0], st->u[1], st->v[0], st->v[1], st->d[0], st->d[1], st->p[0], st->p[1], st->div};
    for (const void* p : ps)
        if (!p || !aligned16(p)) return fail(SMK_EINVAL, "smk_slab_step: a state pointer is NULL or not 16-byte aligned");
    if ((st->cur_u | st->cur_v | st->cur_d | st->cur_p) & ~1) return fail(SMK_EINVAL, "smk_slab_step: cur_* must be 0 or 1");
    if (prm->jacobi_iters < 0 || !(prm->dt != 0.0f)) return fail(SMK_EINVAL, "smk_slab_step: bad jacobi_iters / dt");
    for (const smk_slab_check_t* c : {chk_u, chk_v, chk_d})
        if (c && (!c->overflow_flag || c->need_lo > c->need_hi || c->valid_lo > c->valid_hi)) return fail(SMK_EINVAL, "smk_slab_step: bad check ranges");
    cudaStream_t s = (cudaStream_t)stream;
    // 0. ghost rows of the live u, v, density, p from both neighbours (one exchange per step: the caller's halo is >= K + 4 rows)
    //    SMK_SLAB_PUSH_HEAD: this rank's rows are pushed here; without it the previous step already pushed them from its tail
    if (flags & ~(SMK_SLAB_PUSH_HEAD | SMK_SLAB_PUSH_TAIL)) return fail(SMK_EINVAL, "smk_slab_step: unknown flags 0x%x", (unsigned)flags);
    if (comm) {
        // join the push the previous step left on the side stream (if any)
        SideStream* side = side_stream();
        if (side && side->pending) {
            side->pending = false;
            if (cudaStreamWaitEvent(s, side->ev_join, 0) != cudaSuccess) return fail(SMK_EINVAL, "smk_slab_step: cudaStreamWaitEvent failed: %s", cudaGetErrorString(cudaGetLastError()));
        }
        float* base[4] = {st->u[st->cur_u], st->v[st->cur_v], st->d[st->cur_d], st->p[st->cur_p]};
        if (flags & SMK_SLAB_PUSH_HEAD) SMK_TRY(peer_xfer(comm, base, true, s));
        SMK_TRY(peer_xfer(comm, base, false, s));
    }
    // SMK_SLAB_PUSH_TAIL: the ghost rows of the NEXT step leave from the middle of the density advection
    return phase_step(g, st, prm, nullptr, nullptr, nullptr, 0, nullptr, SMK_FRAME_F32, chk_u, chk_v, chk_d,
                      (comm && (flags & SMK_SLAB_PUSH_TAIL)) ? comm : nullptr, s);
}

int smk_project_advect(const smk_grid_t* g, smk_state_t* st, const smk_params_t* prm,
                       const smk_slab_check_t* chk_u, const smk_slab_check_t* chk_v, const smk_slab_check_t* chk_d, void* stream)
{
    SMK_TRY(check_grid(g, "smk_project_advect"));
    if (!st || !prm) return fail(SMK_EINVAL, "smk_project_advect: state/params NULL");
    if (g->batch != 1) return fail(SMK_EUNSUPPORTED, "smk_project_advect: batch must be 1");
    const void* ps[] = {st->u[0], st->u[1], st->v[0], st->v[1], st->d[0], st->d[1], st->p[0], st->p[1]};
    for (const void* p : ps)
        if (!p || !aligned16(p)) return fail(SMK_EINVAL, "smk_project_advect: a state pointer is NULL or not 16-byte aligned");
    if ((st->cur_u | st->cur_v | st->cur_d | st->cur_p) & ~1) return fail(SMK_EINVAL, "smk_project_advect: cur_* must be 0 or 1");
    for (const smk_slab_check_t* c : {chk_u, chk_v, chk_d})
        if (c && (!c->overflow_flag || c->need_lo > c->need_hi || c->valid_lo > c->valid_hi)) return fail(SMK_EINVAL, "smk_project_advect: bad check ranges");
    return project_advect(g, st, prm, nullptr, 0, nullptr, SMK_FRAME_F32, chk_u, chk_v, chk_d, nullptr, (cudaStream_t)stream);
}

}  // extern "C"
