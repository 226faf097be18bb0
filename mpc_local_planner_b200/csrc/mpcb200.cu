// mpcb200.cu -- sm_100a kernels + C-ABI host side of the batched receding-horizon OCP solver (include/mpcb200.h).
//
// Execution model.  ONE CTA OWNS ONE INSTANCE FOR ITS WHOLE SOLVE: solve_fused_kernel is a persistent kernel whose CTAs take
// instances from a queue (atomic counter), keep the instance's resident prefix (mpc_layout.h: iterate, slacks, multipliers,
// KKT stage records, KKT stage matrices, obstacles -- 50-70 KB) in shared memory, and run initial guess, association and the
// interior-point iterations (eval -> KKT -> line search, mpc_device.cuh) back to back until the instance converges or gives
// up; then the results are written and the CTA takes the next instance.  No launch chain, no HBM round trip of records or
// gains between the phases, and no instance waits for the slowest one of its batch.  Thread mapping inside the CTA: the
// stage-parallel phases (eval, line search) put one lane on one horizon stage (ceil(N/32) warps); the KKT phase is the
// warp-cooperative Riccati sweep of mpc_riccati_warp.h on warp 0 (lanes = entries of the stage matrix, one barrier per stage).
//
// The same device functions are exposed phase by phase (mpcb200_run_phase / mpcb200_time_phase, and the "phased" solve mode)
// through phase_kernel (stages the prefix, runs one phase, writes it back) and kkt_warp_kernel (one warp per instance:
// bulk-async copy of the stage records into shared memory, sweep, Newton step back to HBM) -- the kernel the HBM roofline of
// the KKT factorisation is measured on (SURVEY 8d).
//
// This file is the ONLY implementation of the hot path: there is no CPU fallback.  Every entry point fails with
// MPCB200_E_NODEVICE / MPCB200_E_CUDA when no CUDA device is usable.
#include <cuda_runtime.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <string>
#include <vector>

#include "mpc_device.cuh"
#include "mpc_costmap.cuh"

#define WARPS_PER_CTA 4
#define MAX_IMG_SMEM (227 * 1024 - 2048)  // dynamic shared memory a CTA may request
#define IMG_HEAD 16                        // bytes in front of the resident prefix in dynamic shared memory (mbarrier)

// device-side counters of a handle (unsigned long long each)
#define CNT_KKT_INST 0     // (instance, iteration) pairs the KKT phase factorised
#define CNT_KKT_SWEEPS 1   // backward sweeps incl. inertia-correction refactorisations
#define CNT_CYC 2          // +phase: SM cycles CTAs spent in each phase of the fused kernel (thread 0's clock64)
#define CNT_CYC_TOTAL 7    // SM cycles CTAs spent on instances in the fused kernel
#define CNT_INST 8         // instances solved by the fused kernel
#define CNT_GATE 9         // SM cycles CTAs waited at the phase gates (MPCB200_OPT_SM_PHASE_SYNC)
#define CNT_WORDS 16

// ---- kernel: inputs of a batch into the instance blocks (phased path; the fused kernel scatters into shared memory itself) ----
__global__ void scatter_inputs_kernel(WsLayout L, double* ws, int B, InputPtrs in)
{
    const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (warp >= B) return;
    double* W = ws + (int64_t)warp * L.stride;
    const bool ok = scatter_one(L, W, in, warp, lane, W + L.oXINIT);
    if (lane == 0) ASC(MPCB200_SC_VALID) = ok ? 1.0 : 0.0;
}

// stage [0, words) of an instance block in shared memory (one bulk-async copy) / write [0, words) back
__device__ __forceinline__ void stage_in(double* W, const double* Gp, int words, uint32_t bar, uint32_t parity, int tid)
{
    if (tid == 0)
    {
        fence_async();
        mbar_expect_tx(bar, (uint32_t)words * 8u);
        bulk_g2s(smem_addr(W), Gp, (uint32_t)words * 8u, bar);
    }
    mbar_wait(bar, parity);
}
__device__ __forceinline__ void stage_out(double* Gp, const double* W, int words, int tid)
{
    __syncthreads();
    if (tid == 0)
    {
        fence_async();   // the CTA's ordinary stores to shared memory before the async-proxy read
        bulk_s2g(Gp, smem_addr(W), (uint32_t)words * 8u);
        bulk_commit_wait();
    }
    __syncthreads();
}

// an instance whose inputs are not finite: reported, never iterated, starts cold next time
__device__ __forceinline__ void mark_invalid(const WsLayout& L, double* W)
{
    ASC(MPCB200_SC_STATUS) = (double)MPCB200_STATUS_INVALID_INPUT;
    ASC(MPCB200_SC_COLD) = 1.0; ASC(MPCB200_SC_ITER) = 0.0; ASC(MPCB200_SC_ERR0) = 0.0; ASC(MPCB200_SC_DT) = 0.0;
}

// ---- kernel: ONE PHASE of the solve for every instance of a batch (kernel-level API and the phased solve mode) ----
template <bool LINES>
__global__ void __launch_bounds__(MAX_GROUP_WARPS * 32, 3) phase_kernel(const __grid_constant__ Cfg c, const __grid_constant__ WsLayout L, double* ws, int B, int phase,
                                                                       double uprev_dt, int force_cold, int first_outer, int* n_active, int img_words, InputPtrs in)
{
    extern __shared__ __align__(128) unsigned char dyn_smem[];
    __shared__ CtaShared sh;
    const int inst = blockIdx.x, tid = threadIdx.x, lane = tid & 31, wid = tid >> 5, nt = blockDim.x;
    double* Gp = ws + (int64_t)inst * L.stride;
    if (Gp[L.oSCAL + MPCB200_SC_VALID] == 0.0)
    {
        if (tid == 0 && phase == MPCB200_PHASE_INIT) mark_invalid(L, Gp);
        return;
    }
    if (phase >= MPCB200_PHASE_EVAL && Gp[L.oSCAL + MPCB200_SC_STATUS] >= 0.0) return;  // finished instance: exact no-op (uniform over the CTA)
    double* W = reinterpret_cast<double*>(dyn_smem + IMG_HEAD);
    const uint32_t bar = smem_addr(dyn_smem);
    if (tid == 0) { mbar_init(bar, 1); asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
    __syncthreads();
    stage_in(W, Gp, img_words, bar, 0, tid);
    switch (phase)
    {
        case MPCB200_PHASE_INIT: if (wid == 0) dev_init(c, L, W, obstacle_source(L, W, in, inst), Gp + L.oXINIT, force_cold, lane); break;
        case MPCB200_PHASE_ASSOCIATE:
            if (wid == 0)
            {
                const bool long_list = in.obst_count && in.obst_max > L.M;
                dev_associate(c, L, W, uprev_dt, first_outer, lane, obstacle_source(L, W, in, inst), long_list, Gp + L.oOGIDX);
            }
            break;
        case MPCB200_PHASE_EVAL:
        {
            const int fin = dev_eval<LINES>(c, L, W, uprev_dt, sh, tid, nt);
            if (!fin && n_active && tid == 0) atomicAdd(n_active, 1);
            break;
        }
        case MPCB200_PHASE_LINESEARCH: dev_linesearch<LINES>(c, L, W, uprev_dt, sh, tid, nt); break;
        default: break;
    }
    // everything but the inputs -- except after the association over a long list, which fills the resident obstacles
    const bool wrote_obstacles = phase == MPCB200_PHASE_ASSOCIATE && in.obst_count && in.obst_max > L.M;
    stage_out(Gp, W, wrote_obstacles ? img_words : L.oOTYPE, tid);
}

// ---- kernel: PHASE_KKT -- one warp per instance: records HBM -> shared memory (one bulk-async copy), warp-cooperative
//      Riccati sweep (mpc_riccati_warp.h), Newton step -> HBM.  Algorithmic traffic: the records in, 8 words per stage out. ----
template <bool EXT>
__global__ void __launch_bounds__(32) kkt_warp_kernel(const __grid_constant__ Cfg c, const __grid_constant__ WsLayout L, double* ws, int B, unsigned long long* counters)
{
    extern __shared__ __align__(128) unsigned char dyn_smem[];
    const int inst = blockIdx.x, lane = threadIdx.x;
    const int N = L.N;
    double* Gp = ws + (int64_t)inst * L.stride;
    if (Gp[L.oSCAL + MPCB200_SC_VALID] == 0.0 || Gp[L.oSCAL + MPCB200_SC_STATUS] >= 0.0) return;
    const int rec_words = (N * RSTR + 1) & ~1;
    double* recs = reinterpret_cast<double*>(dyn_smem + IMG_HEAD);
    double* mms = recs + rec_words;
    double* stp = mms + rw_scratch_words<EXT>(N);
    const uint32_t bar = smem_addr(dyn_smem);
    if (lane == 0)
    {
        mbar_init(bar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        mbar_expect_tx(bar, (uint32_t)rec_words * 8u);
        bulk_g2s(smem_addr(recs), Gp + L.oKKT, (uint32_t)rec_words * 8u, bar);
    }
    CudaWarp<EXT> ex;
    ex.lane = lane;
    kkt_warp_setup<EXT>(ex, c.variable_dt);   // beside the copy
    const double htt = Gp[L.oSCAL + MPCB200_SC_HTT], gt = Gp[L.oSCAL + MPCB200_SC_GT], dlast = Gp[L.oSCAL + MPCB200_SC_DELTA_LAST];
    __syncwarp();
    mbar_wait(bar, 0);
    double ddt = 0.0, delta = 0.0;
    int nreg = 0;
    const int ok = kkt_warp_solve<EXT>(ex, c, N, recs, mms, stp, htt, gt, dlast, &ddt, &delta, &nreg);
    __syncwarp();
    if (ok)
        for (int i = lane; i < 8 * N; i += 32) Gp[L.oSTEP + i] = stp[i];
    if (lane == 0)
    {
        kkt_store_outcome(Gp + L.oSCAL, ok, ddt, delta, nreg);
        if (counters) { atomicAdd(counters + CNT_KKT_INST, 1ull); atomicAdd(counters + CNT_KKT_SWEEPS, (unsigned long long)(nreg + (ok ? 1 : 0))); }
    }
}
template <bool EXT>
static size_t kkt_smem_bytes(int N) { return IMG_HEAD + (size_t)(((N * RSTR + 1) & ~1) + rw_scratch_words<EXT>(N) + 8 * N) * 8; }

// ---- kernel: THE SOLVE.  Persistent CTAs take instances from a queue and own them until they terminate. ----
struct FusedArgs
{
    double* ws;              // instance blocks (batch mode: instance i <-> block i, warm state in / out); unused in queue mode
    InputPtrs in;
    OutputPtrs out;
    int total;               // instances in the queue
    int queue_mode;          // 1: a queue of cold instances without blocks (mpcb200_solve_stream)
    int force_cold;
    double uprev_dt;
    int img_words;           // resident prefix
    int* queue;              // next instance
    const int* order;        // queue position -> instance (nullptr: identity)
    unsigned long long* counters;
    unsigned long long* sm_sync;   // [SMs] phase alignment words (nullptr: off)
    int sm_gates;                  // 3: gates before eval, KKT and line search; 2: before KKT and line search only
};
// ---- phase alignment of the CTAs that share an SM ---------------------------------------------------------------------------
// The solve kernel's iteration is ~128 KB of straight fp64 code, four times the SM's instruction cache (32 KB): CTAs that sit on
// the same SM in different phases evict each other's code and every warp streams its instructions from the GPC-level cache
// (ncu: 40 % of the instruction-cache requests miss, `no_instruction` is the first stall reason).  The co-resident CTAs therefore
// enter each phase of the iteration together: one word per SM in global memory -- generation | arrived | members -- is a barrier
// with changing membership (a CTA is a member while it iterates, not while it sets up or writes back an instance).
// The generation counts barriers; generation mod 3 is the phase the barrier opens (eval, KKT, line search): a CTA that arrives
// out of step keeps arriving (and idles) until the generation matches its phase.  Timing only -- no data crosses CTAs.
#define SMS_POLL_NS 128   // pause between two polls of the barrier word (the polling thread shares its scheduler with working warps)
__device__ __forceinline__ unsigned sm_index() { unsigned r; asm volatile("mov.u32 %0, %%smid;" : "=r"(r)); return r; }
#define SMS_MEMBERS(w_) ((unsigned)((w_) & 0xFFFFull))
#define SMS_ARRIVED(w_) ((unsigned)(((w_) >> 16) & 0xFFFFull))
#define SMS_GEN(w_) ((unsigned)((w_) >> 32))
#define SMS_PACK(g_, a_, m_) (((unsigned long long)(g_) << 32) | ((unsigned long long)(a_) << 16) | (unsigned long long)(m_))
__device__ __forceinline__ void sms_join(unsigned long long* st) { atomicAdd(st, 1ull); }
__device__ __forceinline__ void sms_leave(unsigned long long* st)
{
    unsigned long long old = *(volatile unsigned long long*)st, assumed;
    do
    {
        assumed = old;
        unsigned m = SMS_MEMBERS(assumed) - 1u, ar = SMS_ARRIVED(assumed), g = SMS_GEN(assumed);
        if (ar > 0u && ar >= m) { ar = 0u; ++g; }   // the others were waiting for this CTA only
        old = atomicCAS(st, assumed, SMS_PACK(g, ar, m));
    } while (old != assumed);
}
__device__ __forceinline__ void sms_arrive(unsigned long long* st, unsigned phase, unsigned nph)
{
    for (;;)
    {
        unsigned long long old = *(volatile unsigned long long*)st, assumed;
        unsigned g;
        bool released;
        do
        {
            assumed = old;
            unsigned m = SMS_MEMBERS(assumed), ar = SMS_ARRIVED(assumed) + 1u;
            g = SMS_GEN(assumed);
            released = ar >= m;
            old = atomicCAS(st, assumed, released ? SMS_PACK(g + 1u, 0u, m) : SMS_PACK(g, ar, m));
        } while (old != assumed);
        if (!released)
            while (SMS_GEN(*(volatile unsigned long long*)st) == g) __nanosleep(SMS_POLL_NS);
        if (g % nph == phase) return;
    }
}

// ---- kernel: queue order of a batch = longest first by the iteration counts of the PREVIOUS solve of the same slots ----
// A batch costs its slowest instance: an instance that needs 100 iterations and is taken from the queue when the first slots free
// up (2-3 ms into the step) ends 2-3 ms later than if it had been among the first.  Nothing predicts the iteration count of a cold
// instance from its geometry (correlations < 0.2 on the BASELINE instances), but a robot that was hard in the last cycle tends to be
// hard in this one, so the history is the hint.  Counting sort (descending, stable) by min(iters, 1023) in one CTA.
__global__ void __launch_bounds__(1024) order_by_history_kernel(const int* __restrict__ prev_iters, int B, int* __restrict__ order)
{
    __shared__ int hist[1024];
    __shared__ int warp_tot[32];
    const int t = threadIdx.x, lane = t & 31, wid = t >> 5;
    hist[t] = 0;
    __syncthreads();
    for (int i = t; i < B; i += 1024) { int k = prev_iters[i]; k = k < 0 ? 0 : (k > 1023 ? 1023 : k); atomicAdd(&hist[1023 - k], 1); }
    __syncthreads();
    // exclusive scan of hist (bucket 0 = the longest)
    const int v = hist[t];
    int incl = v;
    for (int o = 1; o < 32; o <<= 1) { const int u = __shfl_up_sync(FULLMASK, incl, o); if (lane >= o) incl += u; }
    if (lane == 31) warp_tot[wid] = incl;
    __syncthreads();
    int woff = 0;
    for (int w = 0; w < wid; ++w) woff += warp_tot[w];
    __syncthreads();
    hist[t] = woff + incl - v;   // first position of bucket t
    __syncthreads();
    // stable placement: the thread that owns a bucket walks the instances in index order (buckets are few and short in practice;
    // the walk is B loads per non-empty bucket owner -- done by the warps in parallel over the buckets)
    if (v > 0)
    {
        int pos = hist[t];
        const int key = 1023 - t;
        for (int i = 0; i < B; ++i)
        {
            int k = prev_iters[i]; k = k < 0 ? 0 : (k > 1023 ? 1023 : k);
            if (k == key) order[pos++] = i;
        }
    }
}

template <bool LINES, bool EXT>
__global__ void __launch_bounds__(MAX_GROUP_WARPS * 32, 3) solve_fused_kernel(const __grid_constant__ Cfg c, const __grid_constant__ WsLayout L, const __grid_constant__ FusedArgs a)
{
    extern __shared__ __align__(128) unsigned char dyn_smem[];
    __shared__ CtaShared sh;
    __shared__ int s_inst, s_valid;
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5, nt = blockDim.x;
    const int N = L.N;
    double* W = reinterpret_cast<double*>(dyn_smem + IMG_HEAD);
    const uint32_t bar = smem_addr(dyn_smem);
    if (tid == 0) { mbar_init(bar, 1); asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
    CudaWarp<EXT> ex;
    ex.lane = lane;
    if (wid == 0) kkt_warp_setup<EXT>(ex, c.variable_dt);
    __syncthreads();
    uint32_t parity = 0;
    unsigned long long cyc[MPCB200_NUM_PHASES] = {0, 0, 0, 0, 0}, cyc_total = 0, n_kkt = 0, n_sweeps = 0, n_inst = 0;
    const unsigned nph = (unsigned)a.sm_gates;
    unsigned long long gate_cyc = 0;   // waiting at the phase gates (included in the phase that follows the gate)
    unsigned long long* sms = a.sm_sync ? a.sm_sync + sm_index() : nullptr;
    const int outer = c.outer_iterations > 0 ? c.outer_iterations : 1;
// Phase clocks: EVERY thread keeps them (thread 0's are reported).  Not `if (tid == 0)`: a thread-0-only block directly in front of
// warp-collective code (shuffles, votes) made the compiler split the paths of thread 0 and of lanes 1..31 through the KKT phase in
// one build variant -- lanes 1..31 ran their shuffles on the converged fast path, thread 0 waited in the collective slow path for
// ever (found with cuda-gdb, profiles/r2_phase_alignment.txt).  Branch-free bookkeeping leaves nothing to split.
#define TICK(p_) do { const long long t_ = clock64(); cyc[p_] += (unsigned long long)(t_ - t_mark); t_mark = t_; } while (0)
    for (;;)
    {
        if (tid == 0) { const int q = atomicAdd(a.queue, 1); s_inst = (q < a.total && a.order) ? a.order[q] : q; }
        __syncthreads();
        const int inst = s_inst;
        if (inst >= a.total) break;
        long long t_mark = clock64();
        const long long t_begin = t_mark;
        double* Gp = a.queue_mode ? nullptr : a.ws + (int64_t)inst * L.stride;
        // ---- state: warm trajectory and scalars of the block, or a fresh cold slot ----
        if (!a.queue_mode) { stage_in(W, Gp, L.oNU, bar, parity, tid); parity ^= 1u; }
        else if (tid < MPCB200_SCAL_WORDS) W[L.oSCAL + tid] = tid == MPCB200_SC_COLD ? 1.0 : (tid == MPCB200_SC_STATUS ? -1.0 : 0.0);
        __syncthreads();
        // ---- inputs ----
        if (wid == 0)
        {
            const bool ok = scatter_one(L, W, a.in, inst, lane, nullptr);
            if (lane == 0) { s_valid = ok; ASC(MPCB200_SC_VALID) = ok ? 1.0 : 0.0; if (!ok) mark_invalid(L, W); }
        }
        __syncthreads();
        if (s_valid)
        {
            const bool long_list = a.in.obst_count && a.in.obst_max > L.M;
            const ObstSrc os = obstacle_source(L, W, a.in, inst);
            double* gidx = W + L.oMM;   // scratch of the KKT / line-search phases, free while the association runs
            if (wid == 0) dev_init(c, L, W, os, a.in.x_init ? a.in.x_init + (int64_t)inst * 3 * N : nullptr, a.force_cold, lane);
            __syncthreads();
            TICK(MPCB200_PHASE_INIT);
            for (int oi = 0; oi < outer; ++oi)
            {
                if (wid == 0)
                {
                    dev_associate(c, L, W, a.uprev_dt, oi == 0, lane, os, long_list, gidx);
                    if (long_list && Gp)
                        for (int i = lane; i < L.M; i += 32) Gp[L.oOGIDX + i] = gidx[i];
                }
                __syncthreads();
                TICK(MPCB200_PHASE_ASSOCIATE);
                if (sms) { if (tid == 0) sms_join(sms); __syncthreads(); }
#define PHASE_GATE(p_) do { if (sms) { if (tid == 0) { const long long g0_ = clock64(); sms_arrive(sms, p_, nph); gate_cyc += (unsigned long long)(clock64() - g0_); } __syncthreads(); } } while (0)
                for (;;)
                {
                    if (nph == 3u) PHASE_GATE(0u);
                    const int fin = dev_eval<LINES>(c, L, W, a.uprev_dt, sh, tid, nt);
                    TICK(MPCB200_PHASE_EVAL);
                    if (fin) break;
                    PHASE_GATE(nph - 2u);
                    if (wid == 0) dev_kkt<EXT>(c, L, W, ex, &n_sweeps);
                    __syncthreads();
                    TICK(MPCB200_PHASE_KKT);
                    ++n_kkt;
                    if (ASC(MPCB200_SC_STATUS) >= 0.0) break;   // inertia correction failed: given up
                    PHASE_GATE(nph - 1u);
                    dev_linesearch<LINES>(c, L, W, a.uprev_dt, sh, tid, nt);
                    TICK(MPCB200_PHASE_LINESEARCH);
                    if (ASC(MPCB200_SC_STATUS) >= 0.0) break;   // jammed: given up
                }
#undef PHASE_GATE
                if (sms) { if (tid == 0) sms_leave(sms); __syncthreads(); }
            }
            // a failed solve leaves nothing to warm-start from
            if (tid == 0 && ASC(MPCB200_SC_STATUS) == (double)MPCB200_STATUS_NUMERICAL_ERROR) ASC(MPCB200_SC_COLD) = 1.0;
        }
        __syncthreads();
        gather_one(L, W, a.out, inst, tid, nt);
        if (!a.queue_mode) stage_out(Gp, W, L.oSTATE_END, tid);   // state (and what the kernel-level API reads back)
        else __syncthreads();
        cyc_total += (unsigned long long)(clock64() - t_begin); ++n_inst;
    }
#undef TICK
    if (tid == 0 && a.counters)
    {
        for (int p = 0; p < MPCB200_NUM_PHASES; ++p) atomicAdd(a.counters + CNT_CYC + p, cyc[p]);
        atomicAdd(a.counters + CNT_GATE, gate_cyc);
        atomicAdd(a.counters + CNT_CYC_TOTAL, cyc_total);
        atomicAdd(a.counters + CNT_KKT_INST, n_kkt);
        atomicAdd(a.counters + CNT_KKT_SWEEPS, n_sweeps);
        atomicAdd(a.counters + CNT_INST, n_inst);
    }
}

// ---- kernel: gather results into compact arrays (phased path) ----------------------------------------------------------------
__global__ void gather_outputs_kernel(WsLayout L, double* ws, int B, OutputPtrs o)
{
    const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (warp >= B) return;
    double* W = ws + (int64_t)warp * L.stride;
    if (lane == 0 && ASC(MPCB200_SC_STATUS) == (double)MPCB200_STATUS_NUMERICAL_ERROR) ASC(MPCB200_SC_COLD) = 1.0;
    __syncwarp();
    gather_one(L, W, o, warp, lane, 32);
}

__global__ void reset_kernel(WsLayout L, double* ws, int B, const unsigned char* which)
{
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    if (which && !which[b]) return;
    double* W = ws + (int64_t)b * L.stride;
    ASC(MPCB200_SC_COLD) = 1.0;
    ASC(MPCB200_SC_STATUS) = -1.0;
}

// ---- horizon change (grid adaptation): pack the warm trajectories, switch the layout, resample into the new one ----
// record per instance: SCAL words, X (3 x n_old), U (2 x n_old)
__global__ void resample_pack_kernel(WsLayout L, const double* ws, double* rec, int rec_words, int B)
{
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    const double* W = ws + (int64_t)b * L.stride;
    double* r = rec + (size_t)b * rec_words;
    const int N = L.N;
    for (int i = 0; i < MPCB200_SCAL_WORDS; ++i) r[i] = W[L.oSCAL + i];
    for (int i = 0; i < 3 * N; ++i) r[MPCB200_SCAL_WORDS + i] = W[L.oX + i];
    for (int i = 0; i < 2 * N; ++i) r[MPCB200_SCAL_WORDS + 3 * N + i] = W[L.oU + i];
}
__global__ void resample_unpack_kernel(WsLayout L, double* ws, const double* rec, int rec_words, int n_old, int B)
{
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    double* W = ws + (int64_t)b * L.stride;
    const double* r = rec + (size_t)b * rec_words;
    for (int i = 0; i < MPCB200_SCAL_WORDS; ++i) W[L.oSCAL + i] = r[i];
    if (ASC(MPCB200_SC_COLD) != 0.0) return;  // empty grid: the next step initialises it at the new horizon
    ASC(MPCB200_SC_DT) = resample_serial(n_old, r + MPCB200_SCAL_WORDS, r + MPCB200_SCAL_WORDS + 3 * n_old, r[MPCB200_SC_DT], L.N, W + L.oX, W + L.oU);
}


__global__ void flush_kernel(double* buf, size_t n)
{
    size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
    for (; i < n; i += (size_t)gridDim.x * blockDim.x) buf[i] = buf[i] * 0.999 + 1.0;
}

// =================================================================================================================
// host side
// =================================================================================================================
// a CUDA resource that is released with its owner: device or pinned memory, an event, a stream
template <class T, auto Release>
struct Owned
{
    T v{};
    Owned() = default;
    Owned(const Owned&) = delete;
    Owned& operator=(const Owned&) = delete;
    ~Owned() { reset(); }
    void reset() { if (v) Release(v); v = T{}; }
    T* put() { reset(); return &v; }   // out-parameter of the call that creates the resource
    operator T() const { return v; }
};
template <class T> using Dev = Owned<T*, cudaFree>;
template <class T> static cudaError_t alloc(Dev<T>& buf, size_t count) { return cudaMalloc(buf.put(), count * sizeof(T)); }
using Event = Owned<cudaEvent_t, cudaEventDestroy>;

// compact inputs and outputs of `rows` instances on the device ([row][...] as in mpcb200.h), and what the last upload put there
struct Job
{
    size_t rows = 0;   // instances the arrays hold
    int m = 0;         // obstacles per instance the obstacle arrays hold
    Dev<double> x0, xf, uprev, obst, vp, xinit;   // xinit: the resident batch only
    Dev<int> obst_count, obst_type, vp_count;
    Dev<unsigned char> reinit;                    // the resident batch only
    Dev<double> useq, xseq, dt, kkt, upacked;
    Dev<int> status, iters;
    // the last upload
    int B = 0;
    double uprev_dt = 0.0;
    int has_uprev = 0, has_xinit = 0, has_reinit = 0;
    int obst_max = 0, vp_max = 0;   // list lengths per instance (0: no list)
    int has_lines = 0;  // line obstacles, moving obstacles or midpoint differences: the kernels are launched with those (rarely used) paths compiled in

    InputPtrs inputs() const
    {
        return InputPtrs{x0, xf, has_uprev ? uprev.v : nullptr, obst_max ? obst_count.v : nullptr, obst_type, obst, obst_max,
                         vp_max ? vp_count.v : nullptr, vp, vp_max, has_xinit ? xinit.v : nullptr, has_reinit ? reinit.v : nullptr};
    }
    OutputPtrs outputs() const { return OutputPtrs{useq, xseq, dt, status, kkt, iters, upacked}; }
};

struct mpcb200_handle
{
    Cfg cfg;
    WsLayout L;
    int max_batch = 0, device = 0;
    int n_cap = 0;              // horizon the buffers were sized for at create (mpcb200_resample moves cfg.n within [3, n_cap])
    int num_sms = 0, clock_khz = 0;
    int solve_mode = 0;         // MPCB200_OPT_SOLVE_MODE: 0 fused persistent kernel (default), 1 one kernel per phase
    unsigned timing_mask = 1u << MPCB200_PHASE_KKT;   // phased mode: phases bracketed by CUDA events inside solve (bit = phase id)
    int order_by_history = 1;   // MPCB200_OPT_ORDER_BY_HISTORY: batch queue longest-first by the previous solve's iteration counts
    int sm_phase_sync = -1;     // MPCB200_OPT_SM_PHASE_SYNC: co-resident CTAs of the solve kernel enter the phases together
    int max_ctas_per_sm = 0;    // MPCB200_OPT_CTAS_PER_SM: cap on the resident CTAs per SM of the solve kernel (0 = what fits)
    int fused_grid = 0;         // CTAs of the last fused launch
    int hist_B = 0;             // batch size of the last batch solve whose iteration counts are in batch.iters (0: none)
    Owned<cudaStream_t, cudaStreamDestroy> own_stream;   // the stream the handle created
    cudaStream_t stream = nullptr;                       // the stream in use
    Dev<double> ws;             // instance blocks [max_batch][L.stride]
    Job batch;                  // the resident batch: its inputs and the results of its last solve
    Job queue;                  // the last queue job (mpcb200_solve_stream), grown on demand
    Dev<int> d_nactive, d_queue, d_prev_iters, d_order;
    Dev<unsigned long long> d_counters, d_smsync;
    Dev<double> d_flush;
    size_t flush_n = (size_t)40 * 1024 * 1024;   // 320 MB > 126 MB L2
    // scratch grown on demand: mpcb200_resample; the costmap kernels; mpcb200_check_feasible (maps, trajectories, footprint, flags)
    Dev<double> d_resample; size_t resample_cap = 0;
    Dev<char> d_cm; size_t cm_cap = 0;
    Dev<char> d_fz; size_t fz_cap = 0;
    double costmap_ms = 0.0;    // device ms of the last costmap call
    Owned<int*, cudaFreeHost> h_nactive;   // two poll slots
    Event poll_ev[2], t0, t1, c0, c1;      // t: around a solve, c: around the costmap kernels
    mpcb200_stats stats{};
    std::vector<cudaEvent_t> ev;  // pool of event pairs
    std::vector<int> ev_phase;
    size_t ev_used = 0;
    std::string err;
    // the members release their resources after this body, on the handle's device
    ~mpcb200_handle() { cudaSetDevice(device); for (cudaEvent_t e : ev) cudaEventDestroy(e); }
};

static std::string g_create_err = "";

static int set_err(mpcb200_handle* h, int code, const std::string& msg)
{
    if (h) h->err = msg; else g_create_err = msg;
    return code;
}
#define CK(call)                                                                                                   \
    do {                                                                                                           \
        cudaError_t e_ = (call);                                                                                   \
        if (e_ != cudaSuccess)                                                                                     \
            return set_err(h, MPCB200_E_CUDA, std::string(#call) + ": " + cudaGetErrorString(e_));                 \
    } while (0)

extern "C" void mpcb200_default_config(mpcb200_config* c)
{
    memset(c, 0, sizeof(*c));
    c->robot_type = MPCB200_ROBOT_UNICYCLE;
    c->wheelbase = 0.5; c->length_rear = 1.0; c->length_front = 1.0;
    c->u_lb[0] = -0.2; c->u_lb[1] = -0.3; c->u_ub[0] = 0.4; c->u_ub[1] = 0.3;
    c->du_lb[0] = c->du_lb[1] = -MPCB200_INF; c->du_ub[0] = c->du_ub[1] = MPCB200_INF;
    c->n = 20; c->dt_ref = 0.3; c->variable_dt = 1; c->dt_lb = 0.0; c->dt_ub = 10.0;
    c->xf_fixed[0] = c->xf_fixed[1] = c->xf_fixed[2] = 1;
    c->collocation = MPCB200_COLLOC_FORWARD; c->warm_start = 1;
    c->objective = MPCB200_OBJ_MINIMUM_TIME;
    c->vp_position_weight = 1.0; c->vp_orientation_weight = 0.0;
    c->min_obstacle_dist = 0.5; c->force_inclusion_dist = 0.5; c->cutoff_dist = 2.0;
    c->footprint_type = MPCB200_FOOTPRINT_POINT;
    c->k_max_obstacles_per_stage = 5;
    c->max_iter = 100; c->tol = 1e-6; c->mu_init = 0.0; c->outer_iterations = 1; c->quadratic_integral_form = 0;
    c->initial_guess_bumps = 4;
    c->enable_dynamic_obstacles = 0;
    c->terminal_ball = 0; c->terminal_ball_gamma = 5.0;
    for (int i = 0; i < 9; ++i) c->terminal_ball_S[i] = (i % 4 == 0) ? 1.0 : 0.0;
    c->cost_integration = MPCB200_COST_LEFT_SUM;
    c->hybrid_cost_minimum_time = 0;
}


// doubles of the resident prefix with the largest obstacle list the handle accepts
static size_t max_resident_bytes(const WsLayout& L) { return IMG_HEAD + (size_t)resident_words(L, L.M) * 8; }

static int validate_config(const mpcb200_config* c, std::string& why)
{
    if (c->n < 3 || c->n > 512) { why = "n must be in [3, 512]"; return MPCB200_E_INVALID; }
    if (c->robot_type < 0 || c->robot_type > 3) { why = "unknown robot_type"; return MPCB200_E_INVALID; }
    if (c->collocation != MPCB200_COLLOC_FORWARD && c->collocation != MPCB200_COLLOC_MIDPOINT)
    { why = "collocation: forward_differences and midpoint_differences are implemented, crank_nicolson is not"; return MPCB200_E_UNSUPPORTED; }
    if (c->objective < 0 || c->objective > 2) { why = "unknown objective"; return MPCB200_E_INVALID; }
    if (c->cost_integration != MPCB200_COST_LEFT_SUM && c->cost_integration != MPCB200_COST_TRAPEZOIDAL)
    { why = "unknown cost_integration"; return MPCB200_E_INVALID; }
    if (c->footprint_type < 0 || c->footprint_type > 4) { why = "unknown footprint_type"; return MPCB200_E_INVALID; }
    if (c->footprint_type == MPCB200_FOOTPRINT_POLYGON && (c->n_poly < 1 || c->n_poly > MPCB200_MAX_POLY))
    { why = "polygon footprint needs 1..16 vertices"; return MPCB200_E_INVALID; }
    if (c->k_max_obstacles_per_stage < 0 || c->k_max_obstacles_per_stage > 16) { why = "k_max_obstacles_per_stage must be in [0,16]"; return MPCB200_E_INVALID; }
    if (!(c->dt_ref > 0)) { why = "dt_ref must be > 0"; return MPCB200_E_INVALID; }
    if (c->variable_dt && !(c->dt_ub > c->dt_lb)) { why = "dt_ub must exceed dt_lb"; return MPCB200_E_INVALID; }
    if (has_mintime(*c) && !c->variable_dt) { why = "minimum_time objectives need variable_dt"; return MPCB200_E_INVALID; }
    if (!(c->tol > 0) || c->max_iter < 1) { why = "tol > 0 and max_iter >= 1 required"; return MPCB200_E_INVALID; }
    for (int i = 0; i < 2; ++i)
        if (!(c->u_ub[i] > c->u_lb[i])) { why = "u_ub must exceed u_lb"; return MPCB200_E_INVALID; }
    // one CTA keeps the instance's resident prefix in shared memory: that bounds the horizon (about (56 + 6 RS + 4 K) N words)
    WsLayout L;
    make_layout(c, MAX_OBST, MAX_VP, L);
    if (max_resident_bytes(L) > MAX_IMG_SMEM)
    {
        why = "horizon too long for this row budget: the instance does not fit in shared memory (n = " + std::to_string(c->n) + " needs " +
              std::to_string(max_resident_bytes(L)) + " bytes of " + std::to_string((size_t)MAX_IMG_SMEM) + ")";
        return MPCB200_E_UNSUPPORTED;
    }
    return 0;
}

template <class K>
static cudaError_t allow_smem(K kernel) { return cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, MAX_IMG_SMEM); }

// grows a job to `rows` instances with room for `m` obstacles per instance; never shrinks, and what a grown array held is gone
static int reserve(mpcb200_handle* h, Job& j, size_t rows, int m)
{
    if (rows <= j.rows && m <= j.m) return 0;
    CK(cudaStreamSynchronize(h->stream));   // work in flight may still use the old arrays
    if (rows > j.rows)
    {
        const size_t R = rows, N = (size_t)h->n_cap;   // sized for the largest horizon the handle can be resampled to
        j.rows = 0;
        CK(alloc(j.x0, R * 3)); CK(alloc(j.xf, R * 3)); CK(alloc(j.uprev, R * 2)); CK(alloc(j.obst_count, R));
        CK(alloc(j.vp, R * MAX_VP * 3)); CK(alloc(j.vp_count, R));
        CK(alloc(j.useq, R * N * 2)); CK(alloc(j.xseq, R * N * 3)); CK(alloc(j.dt, R)); CK(alloc(j.kkt, R));
        CK(alloc(j.upacked, R * (N - 1) * 2)); CK(alloc(j.status, R)); CK(alloc(j.iters, R));
        j.rows = rows;
    }
    const size_t M = (size_t)(m > j.m ? m : j.m);
    j.m = 0;
    CK(alloc(j.obst, j.rows * M * MPCB200_OBST_STRIDE)); CK(alloc(j.obst_type, j.rows * M));
    j.m = (int)M;
    return 0;
}

// obstacles per instance a job needs for `obst` (longer lists than the ABI accepts are refused by the upload)
static int obstacle_room(const mpcb200_obstacles* obst)
{
    const int m = (obst && obst->count) ? obst->max_per_instance : 0;
    return m > MAX_OBST && m <= MAX_OBST_LIST ? m : MAX_OBST;
}

// scratch that grows on demand; what it held is gone
template <class T> static int grow(mpcb200_handle* h, Dev<T>& buf, size_t& cap, size_t bytes)
{
    if (bytes <= cap) return 0;
    CK(cudaStreamSynchronize(h->stream));   // work in flight may still use the old buffer
    cap = 0;
    CK(cudaMalloc(buf.put(), bytes));
    cap = bytes;
    return 0;
}

// everything on the device a handle needs from the start
static int init_device(mpcb200_handle* h)
{
    CK(cudaSetDevice(h->device));
    CK(cudaStreamCreateWithFlags(h->own_stream.put(), cudaStreamNonBlocking));
    h->stream = h->own_stream;
    const size_t B = (size_t)h->max_batch;
    int rc = reserve(h, h->batch, B, MAX_OBST);
    if (rc) return rc;
    CK(alloc(h->batch.xinit, B * h->n_cap * 3)); CK(alloc(h->batch.reinit, B));
    CK(alloc(h->ws, B * h->L.stride));
    CK(cudaMemsetAsync(h->ws, 0, B * h->L.stride * sizeof(double), h->stream));
    CK(cudaDeviceGetAttribute(&h->num_sms, cudaDevAttrMultiProcessorCount, h->device));
    CK(cudaDeviceGetAttribute(&h->clock_khz, cudaDevAttrClockRate, h->device));
    CK(alloc(h->d_nactive, 2)); CK(alloc(h->d_queue, 1)); CK(alloc(h->d_smsync, 1024)); CK(alloc(h->d_prev_iters, B)); CK(alloc(h->d_order, B));
    CK(alloc(h->d_counters, CNT_WORDS)); CK(cudaMemsetAsync(h->d_counters, 0, CNT_WORDS * 8, h->stream));
    CK(allow_smem(phase_kernel<false>)); CK(allow_smem(phase_kernel<true>));
    CK(allow_smem(kkt_warp_kernel<false>)); CK(allow_smem(kkt_warp_kernel<true>));
    CK(allow_smem(solve_fused_kernel<false, false>)); CK(allow_smem(solve_fused_kernel<false, true>));
    CK(allow_smem(solve_fused_kernel<true, false>)); CK(allow_smem(solve_fused_kernel<true, true>));
    CK(cudaMallocHost(h->h_nactive.put(), 8));
    CK(cudaEventCreateWithFlags(h->poll_ev[0].put(), cudaEventDisableTiming)); CK(cudaEventCreateWithFlags(h->poll_ev[1].put(), cudaEventDisableTiming));
    CK(cudaEventCreate(h->t0.put())); CK(cudaEventCreate(h->t1.put())); CK(cudaEventCreate(h->c0.put())); CK(cudaEventCreate(h->c1.put()));
    CK(alloc(h->d_flush, h->flush_n));
    CK(cudaMemsetAsync(h->d_flush, 0, h->flush_n * 8, h->stream));
    // all instances start cold
    reset_kernel<<<(h->max_batch + 127) / 128, 128, 0, h->stream>>>(h->L, h->ws, h->max_batch, nullptr);
    CK(cudaGetLastError());
    CK(cudaStreamSynchronize(h->stream));
    return 0;
}

extern "C" int mpcb200_create(const mpcb200_config* cfg, int max_batch, int device, mpcb200_handle** out)
{
    if (!cfg || !out || max_batch < 1) return set_err(nullptr, MPCB200_E_INVALID, "bad arguments");
    std::string why;
    int rc = validate_config(cfg, why);
    if (rc) return set_err(nullptr, rc, why);
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0)
        return set_err(nullptr, MPCB200_E_NODEVICE, std::string("no CUDA device (") + cudaGetErrorString(e) + "): this solver has no CPU fallback");
    if (device < 0 || device >= ndev) return set_err(nullptr, MPCB200_E_INVALID, "device index out of range");
    mpcb200_handle* h = new mpcb200_handle();
    h->cfg = *cfg; h->max_batch = max_batch; h->device = device; h->n_cap = cfg->n;
    make_layout(cfg, MAX_OBST, MAX_VP, h->L);
    if ((rc = init_device(h)))
    {
        why = h->err;
        delete h;
        return set_err(nullptr, rc, why);
    }
    *out = h;
    return MPCB200_OK;
}

extern "C" void mpcb200_destroy(mpcb200_handle* h)
{
    if (!h) return;
    cudaSetDevice(h->device);
    cudaStreamSynchronize(h->stream);
    delete h;
}

extern "C" const char* mpcb200_last_error(const mpcb200_handle* h) { return h ? h->err.c_str() : g_create_err.c_str(); }

static inline int grid_for(int B, int wpc) { return (B + wpc - 1) / wpc; }

// event-pair pool: device time per phase launch (CUDA events on the solver stream)
static int ev_begin(mpcb200_handle* h, int phase)
{
    if (h->ev_used + 2 > h->ev.size())
    {
        for (int i = 0; i < 256; ++i) { cudaEvent_t e; if (cudaEventCreate(&e) != cudaSuccess) return -1; h->ev.push_back(e); }
        h->ev_phase.resize(h->ev.size() / 2);
    }
    h->ev_phase[h->ev_used / 2] = phase;
    cudaEventRecord(h->ev[h->ev_used], h->stream);
    return 0;
}
static void ev_end(mpcb200_handle* h)
{
    cudaEventRecord(h->ev[h->ev_used + 1], h->stream);
    h->ev_used += 2;
}
static void ev_collect(mpcb200_handle* h)
{
    for (size_t i = 0; i + 1 < h->ev_used; i += 2)
    {
        float ms = 0.f;
        if (cudaEventElapsedTime(&ms, h->ev[i], h->ev[i + 1]) == cudaSuccess)
        {
            const int p = h->ev_phase[i / 2];
            h->stats.ms[p] += ms; h->stats.launches[p] += 1;
        }
    }
    h->ev_used = 0;
}

// threads of the CTA that owns an instance
static int group_threads(const mpcb200_handle* h)
{
    const int gw = (h->cfg.n + 31) / 32;
    return 32 * (gw < MAX_GROUP_WARPS ? gw : MAX_GROUP_WARPS);   // a lane per stage
}
static int image_words(const mpcb200_handle* h, const Job& j) { return resident_words(h->L, j.obst_max < h->L.M ? j.obst_max : h->L.M); }

static int launch_phase(mpcb200_handle* h, int phase, int B, int force_cold, int first_outer, int* n_active, bool timed)
{
    const Job& j = h->batch;
    const int img_words = image_words(h, j);
    const size_t img_smem = IMG_HEAD + (size_t)img_words * 8;
    if (img_smem > MAX_IMG_SMEM) return set_err(h, MPCB200_E_UNSUPPORTED, "the instance does not fit in shared memory");
    if (timed && ev_begin(h, phase)) return set_err(h, MPCB200_E_CUDA, "cudaEventCreate failed");
    if (phase == MPCB200_PHASE_KKT)
    {
        if (kkt_is_ext(h->cfg)) kkt_warp_kernel<true><<<B, 32, kkt_smem_bytes<true>(h->cfg.n), h->stream>>>(h->cfg, h->L, h->ws, B, h->d_counters);
        else kkt_warp_kernel<false><<<B, 32, kkt_smem_bytes<false>(h->cfg.n), h->stream>>>(h->cfg, h->L, h->ws, B, h->d_counters);
    }
    else if (phase >= 0 && phase < MPCB200_NUM_PHASES)
    {
        const auto kernel = j.has_lines ? phase_kernel<true> : phase_kernel<false>;
        kernel<<<B, group_threads(h), img_smem, h->stream>>>(h->cfg, h->L, h->ws, B, phase, j.uprev_dt, force_cold, first_outer, n_active, img_words, j.inputs());
    }
    else return set_err(h, MPCB200_E_INVALID, "unknown phase");
    if (timed) ev_end(h);
    h->stats.launches_total += 1;
    CK(cudaGetLastError());
    return 0;
}

static int check_batch(mpcb200_handle* h, int B)
{
    if (!h) return MPCB200_E_INVALID;
    if (B < 1 || B > h->max_batch) return set_err(h, MPCB200_E_INVALID, "batch size out of range");
    return 0;
}

// which kernel variants a job needs: line obstacles among the obstacles in use (padding slots are never read)
static bool has_line_obstacles(size_t B, const mpcb200_obstacles* obst)
{
    const size_t M = (size_t)obst->max_per_instance;
    for (size_t b = 0; b < B; ++b)
    {
        const int cnt = obst->count[b] < (int)M ? obst->count[b] : (int)M;
        for (int i = 0; i < cnt; ++i)
            if (obst->type[b * M + i] == MPCB200_OBST_LINE) return true;
    }
    return false;
}

// host -> device copies of the inputs of `B` instances into a job (grown to hold them), and their description
static int upload(mpcb200_handle* h, Job& j, size_t B, const double* x0, const double* xf, const double* u_prev, double u_prev_dt,
                  const mpcb200_obstacles* obst, const mpcb200_viapoints* vp, const double* x_init, const unsigned char* reinit)
{
    if (!x0 || !xf) return set_err(h, MPCB200_E_INVALID, "x0 and xf are required");
    int rc = reserve(h, j, B, obstacle_room(obst));
    if (rc) return rc;
    const size_t N = (size_t)h->cfg.n;
    CK(cudaMemcpyAsync(j.x0, x0, B * 3 * 8, cudaMemcpyHostToDevice, h->stream));
    CK(cudaMemcpyAsync(j.xf, xf, B * 3 * 8, cudaMemcpyHostToDevice, h->stream));
    h->stats.h2d_bytes += (long long)(B * 6 * 8);
    j.has_uprev = u_prev != nullptr;
    if (u_prev) { CK(cudaMemcpyAsync(j.uprev, u_prev, B * 2 * 8, cudaMemcpyHostToDevice, h->stream)); h->stats.h2d_bytes += (long long)(B * 16); }
    j.uprev_dt = u_prev_dt;
    j.obst_max = 0; j.has_lines = is_midpoint(h->cfg);
    if (obst && obst->count && obst->max_per_instance > 0)
    {
        if (obst->max_per_instance > MAX_OBST_LIST) return set_err(h, MPCB200_E_UNSUPPORTED, "more than 2048 obstacles per instance");
        if (!obst->type || !obst->params) return set_err(h, MPCB200_E_INVALID, "obstacle types and parameters are required");
        const size_t M = (size_t)obst->max_per_instance;
        j.has_lines = has_line_obstacles(B, obst) || h->cfg.enable_dynamic_obstacles || is_midpoint(h->cfg);
        CK(cudaMemcpyAsync(j.obst_count, obst->count, B * 4, cudaMemcpyHostToDevice, h->stream));
        CK(cudaMemcpyAsync(j.obst_type, obst->type, B * M * 4, cudaMemcpyHostToDevice, h->stream));
        CK(cudaMemcpyAsync(j.obst, obst->params, B * M * MPCB200_OBST_STRIDE * 8, cudaMemcpyHostToDevice, h->stream));
        h->stats.h2d_bytes += (long long)(B * 4 + B * M * 4 + B * M * MPCB200_OBST_STRIDE * 8);
        j.obst_max = (int)M;
    }
    j.vp_max = 0;
    if (vp && vp->count && vp->max_per_instance > 0)
    {
        if (vp->max_per_instance > MAX_VP) return set_err(h, MPCB200_E_UNSUPPORTED, "more than 8 via-points per instance");
        const size_t V = (size_t)vp->max_per_instance;
        CK(cudaMemcpyAsync(j.vp_count, vp->count, B * 4, cudaMemcpyHostToDevice, h->stream));
        CK(cudaMemcpyAsync(j.vp, vp->poses, B * V * 3 * 8, cudaMemcpyHostToDevice, h->stream));
        h->stats.h2d_bytes += (long long)(B * 4 + B * V * 24);
        j.vp_max = (int)V;
    }
    j.has_xinit = x_init != nullptr;
    if (x_init) { CK(cudaMemcpyAsync(j.xinit, x_init, B * N * 3 * 8, cudaMemcpyHostToDevice, h->stream)); h->stats.h2d_bytes += (long long)(B * N * 24); }
    j.has_reinit = reinit != nullptr;
    if (reinit) { CK(cudaMemcpyAsync(j.reinit, reinit, B, cudaMemcpyHostToDevice, h->stream)); h->stats.h2d_bytes += (long long)B; }
    j.B = (int)B;
    return 0;
}

// the resident batch's inputs into the instance blocks: the kernel-level API (phase kernels) works on the blocks
static int scatter_batch(mpcb200_handle* h)
{
    const int B = h->batch.B;
    scatter_inputs_kernel<<<grid_for(B, WARPS_PER_CTA), WARPS_PER_CTA * 32, 0, h->stream>>>(h->L, h->ws, B, h->batch.inputs());
    h->stats.launches_total += 1;
    CK(cudaGetLastError());
    return 0;
}

// ---- the solve: one launch of the persistent kernel over the instances of a job ----
static int launch_fused(mpcb200_handle* h, const Job& j, int force_cold)
{
    const bool queue_mode = &j == &h->queue;   // cold instances without blocks (mpcb200_solve_stream)
    const int total = j.B;
    FusedArgs a;
    a.ws = h->ws; a.in = j.inputs(); a.out = j.outputs(); a.total = total; a.queue_mode = queue_mode; a.force_cold = force_cold; a.uprev_dt = j.uprev_dt;
    a.img_words = image_words(h, j); a.queue = h->d_queue; a.counters = h->d_counters;
    a.sm_sync = nullptr; a.sm_gates = h->sm_phase_sync == 2 ? 2 : 3;
    a.order = nullptr;
    if (!queue_mode && h->order_by_history && h->hist_B == total && total > h->num_sms)
    {
        // (the iteration counts are rewritten by this solve: order from a copy)
        CK(cudaMemcpyAsync(h->d_prev_iters, j.iters, (size_t)total * 4, cudaMemcpyDeviceToDevice, h->stream));
        order_by_history_kernel<<<1, 1024, 0, h->stream>>>(h->d_prev_iters, total, h->d_order);
        h->stats.launches_total += 1;
        a.order = h->d_order;
    }
    if (!queue_mode) h->hist_B = total;
    const size_t smem = IMG_HEAD + (size_t)a.img_words * 8;
    if (smem > MAX_IMG_SMEM) return set_err(h, MPCB200_E_UNSUPPORTED, "the instance does not fit in shared memory");
    const int threads = group_threads(h);
    const bool ext = kkt_is_ext(h->cfg);
    const auto kernel = j.has_lines ? (ext ? solve_fused_kernel<true, true> : solve_fused_kernel<true, false>)
                                    : (ext ? solve_fused_kernel<false, true> : solve_fused_kernel<false, false>);
    int per_sm = 0;
    CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, threads, smem));
    if (per_sm < 1) return set_err(h, MPCB200_E_UNSUPPORTED, "the solve kernel does not fit on an SM with this configuration");
    if (h->max_ctas_per_sm > 0 && per_sm > h->max_ctas_per_sm) per_sm = h->max_ctas_per_sm;
    const int grid = total < per_sm * h->num_sms ? total : per_sm * h->num_sms;
    h->fused_grid = grid;
    // phase alignment pays when several CTAs share an SM (auto: from three; measured, profiles/r2_phase_alignment.txt)
    if (h->sm_phase_sync > 0 || (h->sm_phase_sync < 0 && per_sm >= 3 && grid > h->num_sms))
    {
        a.sm_sync = h->d_smsync;
        CK(cudaMemsetAsync(h->d_smsync, 0, 1024 * 8, h->stream));
    }
    CK(cudaMemsetAsync(h->d_queue, 0, 4, h->stream));
    kernel<<<grid, threads, smem, h->stream>>>(h->cfg, h->L, a);
    h->stats.launches_total += 1;
    CK(cudaGetLastError());
    return 0;
}

// the phased form of the same solve (MPCB200_OPT_SOLVE_MODE 1): one kernel per phase, the host queues the iterations
static int solve_phased(mpcb200_handle* h, int B, int force_cold)
{
    const unsigned tm = h->timing_mask;
    auto timed = [&](int phase) { return ((tm >> phase) & 1u) != 0; };
    int rc = launch_phase(h, MPCB200_PHASE_INIT, B, force_cold, 0, nullptr, timed(MPCB200_PHASE_INIT));
    if (rc) return rc;
    const int outer = h->cfg.outer_iterations > 0 ? h->cfg.outer_iterations : 1;
    for (int oi = 0; oi < outer; ++oi)
    {
        if ((rc = launch_phase(h, MPCB200_PHASE_ASSOCIATE, B, 0, oi == 0, nullptr, timed(MPCB200_PHASE_ASSOCIATE)))) return rc;
        // The number of unfinished instances is polled every POLL iterations, one poll behind: the host keeps queueing
        // iterations while the count of the previous poll travels back (a finished instance makes every kernel a no-op).
        const int POLL = 4;
        int pending = -1;  // slot of the poll in flight
        bool done = false;
        for (int it = 0; it <= h->cfg.max_iter && !done; ++it)
        {
            const bool poll = (it % POLL == POLL - 1) || it == h->cfg.max_iter;
            const int slot = (it / POLL) & 1;
            if (poll) CK(cudaMemsetAsync(h->d_nactive + slot, 0, 4, h->stream));
            if ((rc = launch_phase(h, MPCB200_PHASE_EVAL, B, 0, 0, poll ? h->d_nactive + slot : nullptr, timed(MPCB200_PHASE_EVAL)))) return rc;
            if (poll)
            {
                CK(cudaMemcpyAsync(h->h_nactive + slot, h->d_nactive + slot, 4, cudaMemcpyDeviceToHost, h->stream));
                CK(cudaEventRecord(h->poll_ev[slot], h->stream));
                if (pending >= 0)
                {
                    CK(cudaEventSynchronize(h->poll_ev[pending]));
                    if (h->h_nactive[pending] == 0) done = true;
                }
                pending = slot;
            }
            if (it == h->cfg.max_iter || done) break;
            if ((rc = launch_phase(h, MPCB200_PHASE_KKT, B, 0, 0, nullptr, timed(MPCB200_PHASE_KKT)))) return rc;
            if ((rc = launch_phase(h, MPCB200_PHASE_LINESEARCH, B, 0, 0, nullptr, timed(MPCB200_PHASE_LINESEARCH)))) return rc;
        }
    }
    gather_outputs_kernel<<<grid_for(B, WARPS_PER_CTA), WARPS_PER_CTA * 32, 0, h->stream>>>(h->L, h->ws, B, h->batch.outputs());
    h->stats.launches_total += 1;
    CK(cudaGetLastError());
    return 0;
}

// fold the cycle counters of the fused kernel into the per-phase statistics: average time a CTA spent in each phase
static int collect_fused_counters(mpcb200_handle* h)
{
    unsigned long long cnt[CNT_WORDS];
    CK(cudaMemcpy(cnt, h->d_counters, sizeof(cnt), cudaMemcpyDeviceToHost));
    const double per_cta = h->fused_grid > 0 ? 1.0 / ((double)h->fused_grid * (double)h->clock_khz) : 0.0;  // cycles -> ms per CTA
    for (int p = 0; p < MPCB200_NUM_PHASES; ++p) h->stats.ms[p] += (double)cnt[CNT_CYC + p] * per_cta;
    h->stats.gate_ms += (double)cnt[CNT_GATE] * per_cta;
    h->stats.kkt_instances += (long long)cnt[CNT_KKT_INST];
    h->stats.kkt_sweeps += (long long)cnt[CNT_KKT_SWEEPS];
    h->stats.launches[MPCB200_PHASE_KKT] += (long long)cnt[CNT_KKT_INST];
    CK(cudaMemsetAsync(h->d_counters, 0, sizeof(cnt), h->stream));
    return 0;
}

// the solve of a job (the resident batch: fused or phased; a queue: fused), timed with events, then the device counters
static int solve_device(mpcb200_handle* h, const Job& j, int force_cold, double* solve_time_s)
{
    CK(cudaEventRecord(h->t0, h->stream));
    const int rc = (&j == &h->batch && h->solve_mode == 1) ? solve_phased(h, j.B, force_cold) : launch_fused(h, j, force_cold);
    if (rc) return rc;
    CK(cudaEventRecord(h->t1, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    float ms = 0.f;
    CK(cudaEventElapsedTime(&ms, h->t0, h->t1));
    if (solve_time_s) *solve_time_s = ms * 1e-3;
    ev_collect(h);
    return collect_fused_counters(h);
}

// device -> host copies of the results of a job's last solve
static int fetch(mpcb200_handle* h, const Job& j, double* u_seq, double* x_seq, double* dt_out, int* status, double* kkt_err, int* iters)
{
    const size_t B = (size_t)j.B, N = (size_t)h->cfg.n;
    if (u_seq) { CK(cudaMemcpyAsync(u_seq, j.useq, B * N * 16, cudaMemcpyDeviceToHost, h->stream)); h->stats.d2h_bytes += (long long)(B * N * 16); }
    if (x_seq) { CK(cudaMemcpyAsync(x_seq, j.xseq, B * N * 24, cudaMemcpyDeviceToHost, h->stream)); h->stats.d2h_bytes += (long long)(B * N * 24); }
    if (dt_out) { CK(cudaMemcpyAsync(dt_out, j.dt, B * 8, cudaMemcpyDeviceToHost, h->stream)); h->stats.d2h_bytes += (long long)(B * 8); }
    if (status) { CK(cudaMemcpyAsync(status, j.status, B * 4, cudaMemcpyDeviceToHost, h->stream)); h->stats.d2h_bytes += (long long)(B * 4); }
    if (kkt_err) { CK(cudaMemcpyAsync(kkt_err, j.kkt, B * 8, cudaMemcpyDeviceToHost, h->stream)); h->stats.d2h_bytes += (long long)(B * 8); }
    if (iters) { CK(cudaMemcpyAsync(iters, j.iters, B * 4, cudaMemcpyDeviceToHost, h->stream)); h->stats.d2h_bytes += (long long)(B * 4); }
    CK(cudaStreamSynchronize(h->stream));
    return 0;
}

// ---- queue solve: `total` cold instances through the persistent kernel (continuous batching) ----------------------
extern "C" int mpcb200_solve_stream(mpcb200_handle* h, int total, const double* x0, const double* xf, const double* u_prev, double u_prev_dt,
                                    const mpcb200_obstacles* obst, const mpcb200_viapoints* vp, double* u_seq, double* x_seq, double* dt_out,
                                    int* status, double* kkt_err, int* iters, double* solve_time_s)
{
    if (!h) return MPCB200_E_INVALID;
    if (total < 1 || !x0 || !xf) return set_err(h, MPCB200_E_INVALID, "total >= 1, x0 and xf are required");
    CK(cudaSetDevice(h->device));
    int rc = upload(h, h->queue, (size_t)total, x0, xf, u_prev, u_prev_dt, obst, vp, nullptr, nullptr);
    if (rc) return rc;
    if ((rc = solve_device(h, h->queue, 1, solve_time_s))) return rc;
    return fetch(h, h->queue, u_seq, x_seq, dt_out, status, kkt_err, iters);
}

extern "C" int mpcb200_step_batch(mpcb200_handle* h, int B, const double* x0, const double* xf, const double* u_prev, double u_prev_dt,
                                  const mpcb200_obstacles* obst, const mpcb200_viapoints* vp, const double* x_init,
                                  const unsigned char* reinit, double* u_seq, double* x_seq, double* dt_out, int* status,
                                  double* kkt_err, int* iters, double* solve_time_s)
{
    int rc = check_batch(h, B);
    if (rc) return rc;
    CK(cudaSetDevice(h->device));
    if ((rc = upload(h, h->batch, (size_t)B, x0, xf, u_prev, u_prev_dt, obst, vp, x_init, reinit))) return rc;
    // the phase kernels read the inputs from the instance blocks; the fused kernel reads the compact arrays itself
    if (h->solve_mode == 1 && (rc = scatter_batch(h))) return rc;
    if ((rc = solve_device(h, h->batch, 0, solve_time_s))) return rc;
    return fetch(h, h->batch, u_seq, x_seq, dt_out, status, kkt_err, iters);
}

extern "C" int mpcb200_upload_inputs(mpcb200_handle* h, int B, const double* x0, const double* xf, const double* u_prev, double u_prev_dt,
                                     const mpcb200_obstacles* obst, const mpcb200_viapoints* vp, const double* x_init)
{
    int rc = check_batch(h, B);
    if (rc) return rc;
    CK(cudaSetDevice(h->device));
    if ((rc = upload(h, h->batch, (size_t)B, x0, xf, u_prev, u_prev_dt, obst, vp, x_init, nullptr)) || (rc = scatter_batch(h))) return rc;
    CK(cudaStreamSynchronize(h->stream));
    return 0;
}

extern "C" int mpcb200_solve_resident(mpcb200_handle* h, int cold, double* solve_time_s)
{
    if (!h || h->batch.B < 1) return set_err(h, MPCB200_E_INVALID, "no resident inputs: call mpcb200_upload_inputs first");
    CK(cudaSetDevice(h->device));
    return solve_device(h, h->batch, cold ? 1 : 0, solve_time_s);
}

extern "C" int mpcb200_fetch_results(mpcb200_handle* h, double* u_seq, double* x_seq, double* dt_out, int* status, double* kkt_err, int* iters)
{
    if (!h || h->batch.B < 1) return set_err(h, MPCB200_E_INVALID, "nothing to fetch");
    CK(cudaSetDevice(h->device));
    return fetch(h, h->batch, u_seq, x_seq, dt_out, status, kkt_err, iters);
}

extern "C" int mpcb200_device_controls(mpcb200_handle* h, void** dev_ptr, long long* n_doubles)
{
    if (!h || h->batch.B < 1) return set_err(h, MPCB200_E_INVALID, "no batch solved yet");
    if (dev_ptr) *dev_ptr = h->batch.upacked;
    if (n_doubles) *n_doubles = (long long)h->batch.B * (h->cfg.n - 1) * 2;
    return 0;
}

extern "C" int mpcb200_reset(mpcb200_handle* h, const unsigned char* which, int B)
{
    if (!h) return MPCB200_E_INVALID;
    CK(cudaSetDevice(h->device));
    const int n = which ? B : h->max_batch;
    if (n < 1 || n > h->max_batch) return set_err(h, MPCB200_E_INVALID, "batch size out of range");
    if (which) CK(cudaMemcpyAsync(h->batch.reinit, which, (size_t)n, cudaMemcpyHostToDevice, h->stream));
    reset_kernel<<<(n + 127) / 128, 128, 0, h->stream>>>(h->L, h->ws, n, which ? h->batch.reinit.v : nullptr);
    CK(cudaGetLastError());
    CK(cudaStreamSynchronize(h->stream));
    return 0;
}

extern "C" int mpcb200_resample(mpcb200_handle* h, int n_new)
{
    if (!h) return MPCB200_E_INVALID;
    if (n_new < 3 || n_new > h->n_cap) return set_err(h, MPCB200_E_INVALID, "resample: horizon must be in [3, n the handle was created with]");
    if (n_new == h->cfg.n) return MPCB200_OK;
    CK(cudaSetDevice(h->device));
    const int B = h->max_batch, n_old = h->cfg.n;
    const int rec_words = MPCB200_SCAL_WORDS + 5 * h->n_cap;
    const int rc = grow(h, h->d_resample, h->resample_cap, (size_t)B * rec_words * sizeof(double));
    if (rc) return rc;
    resample_pack_kernel<<<(B + 127) / 128, 128, 0, h->stream>>>(h->L, h->ws, h->d_resample, rec_words, B);
    CK(cudaGetLastError());
    h->cfg.n = n_new;
    make_layout(&h->cfg, h->L.M, h->L.V, h->L);
    resample_unpack_kernel<<<(B + 127) / 128, 128, 0, h->stream>>>(h->L, h->ws, h->d_resample, rec_words, n_old, B);
    CK(cudaGetLastError());
    CK(cudaStreamSynchronize(h->stream));
    return MPCB200_OK;
}

extern "C" int mpcb200_get_horizon(const mpcb200_handle* h, int* n, int* n_capacity)
{
    if (!h) return MPCB200_E_INVALID;
    if (n) *n = h->cfg.n;
    if (n_capacity) *n_capacity = h->n_cap;
    return MPCB200_OK;
}

// ---- kernel-level access ------------------------------------------------------------------------------------
static int field_info(const mpcb200_handle* h, int field, int* off, int* cnt)
{
    const WsLayout& L = h->L;
    switch (field)
    {
        case MPCB200_F_X: *off = L.oX; *cnt = 3; return 0;
        case MPCB200_F_U: *off = L.oU; *cnt = 2; return 0;
        case MPCB200_F_NU: *off = L.oNU; *cnt = 3; return 0;
        case MPCB200_F_S: *off = L.oS; *cnt = L.RS; return 0;
        case MPCB200_F_LAM: *off = L.oLAM; *cnt = L.RS; return 0;
        case MPCB200_F_KKT: *off = L.oKKT; *cnt = KW; return 0;
        case MPCB200_F_STEP: *off = L.oSTEP; *cnt = 8; return 0;
        case MPCB200_F_SCAL: *off = L.oSCAL; *cnt = MPCB200_SCAL_WORDS; return 0;
        case MPCB200_F_OBSIDX: *off = L.oOBS; *cnt = L.K > 0 ? L.K : 1; return 0;
        case MPCB200_F_OBSGIDX: *off = L.oOGIDX; *cnt = L.M; return 0;
    }
    return -1;
}

extern "C" int mpcb200_ws_count(const mpcb200_handle* h, int field)
{
    int off, cnt;
    if (!h || field_info(h, field, &off, &cnt)) return MPCB200_E_INVALID;
    return cnt;
}

extern "C" int mpcb200_ws_read(mpcb200_handle* h, int field, int B, double* dst)
{
    int off, cnt, rc = check_batch(h, B);
    if (rc) return rc;
    if (!dst || field_info(h, field, &off, &cnt)) return set_err(h, MPCB200_E_INVALID, "bad field");
    CK(cudaSetDevice(h->device));
    const int N = h->L.N;
    if (field == MPCB200_F_KKT)
    {   // device layout: stage records [k][RSTR] inside the instance block; the API presents [B][42][N]
        std::vector<double> tmp((size_t)B * N * RSTR);
        CK(cudaMemcpy2DAsync(tmp.data(), (size_t)N * RSTR * 8, h->ws + off, (size_t)h->L.stride * 8, (size_t)N * RSTR * 8, (size_t)B, cudaMemcpyDeviceToHost, h->stream));
        CK(cudaStreamSynchronize(h->stream));
        for (int b = 0; b < B; ++b)
            for (int k = 0; k < N; ++k)
                for (int f = 0; f < KW; ++f) dst[((size_t)b * KW + f) * N + k] = tmp[((size_t)b * N + k) * RSTR + f];
        return 0;
    }
    if (field == MPCB200_F_OBSIDX)
    {   // device layout: one signed byte per (slot, stage); the API presents doubles [B][K][N]
        const size_t nb = (size_t)cnt * N;
        std::vector<signed char> tmp((size_t)B * nb);
        CK(cudaMemcpy2DAsync(tmp.data(), nb, h->ws + off, (size_t)h->L.stride * 8, nb, (size_t)B, cudaMemcpyDeviceToHost, h->stream));
        CK(cudaStreamSynchronize(h->stream));
        for (size_t i = 0; i < tmp.size(); ++i) dst[i] = (double)tmp[i];
        return 0;
    }
    const size_t words = (field == MPCB200_F_SCAL || field == MPCB200_F_OBSGIDX) ? (size_t)cnt : (size_t)cnt * N;
    CK(cudaMemcpy2DAsync(dst, words * 8, h->ws + off, (size_t)h->L.stride * 8, words * 8, (size_t)B, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    return 0;
}

extern "C" int mpcb200_ws_write(mpcb200_handle* h, int field, int B, const double* src)
{
    int off, cnt, rc = check_batch(h, B);
    if (rc) return rc;
    if (!src || field_info(h, field, &off, &cnt)) return set_err(h, MPCB200_E_INVALID, "bad field");
    CK(cudaSetDevice(h->device));
    const int N = h->L.N;
    if (field == MPCB200_F_KKT)
    {
        std::vector<double> tmp((size_t)B * N * RSTR, 0.0);
        for (int b = 0; b < B; ++b)
            for (int k = 0; k < N; ++k)
                for (int f = 0; f < KW; ++f) tmp[((size_t)b * N + k) * RSTR + f] = src[((size_t)b * KW + f) * N + k];
        CK(cudaMemcpy2DAsync(h->ws + off, (size_t)h->L.stride * 8, tmp.data(), (size_t)N * RSTR * 8, (size_t)N * RSTR * 8, (size_t)B, cudaMemcpyHostToDevice, h->stream));
        CK(cudaStreamSynchronize(h->stream));
        return 0;
    }
    if (field == MPCB200_F_OBSIDX)
    {
        const size_t nb = (size_t)cnt * N;
        std::vector<signed char> tmp((size_t)B * nb);
        for (size_t i = 0; i < tmp.size(); ++i) tmp[i] = (signed char)src[i];
        CK(cudaMemcpy2DAsync(h->ws + off, (size_t)h->L.stride * 8, tmp.data(), nb, nb, (size_t)B, cudaMemcpyHostToDevice, h->stream));
        CK(cudaStreamSynchronize(h->stream));
        return 0;
    }
    const size_t words = (field == MPCB200_F_SCAL || field == MPCB200_F_OBSGIDX) ? (size_t)cnt : (size_t)cnt * N;
    CK(cudaMemcpy2DAsync(h->ws + off, (size_t)h->L.stride * 8, src, words * 8, words * 8, (size_t)B, cudaMemcpyHostToDevice, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    return 0;
}

extern "C" int mpcb200_run_phase(mpcb200_handle* h, int phase, int B)
{
    int rc = check_batch(h, B);
    if (rc) return rc;
    CK(cudaSetDevice(h->device));
    if ((rc = launch_phase(h, phase, B, 0, 1, nullptr, true))) return rc;
    CK(cudaStreamSynchronize(h->stream));
    ev_collect(h);
    return 0;
}

extern "C" int mpcb200_set_stream(mpcb200_handle* h, void* cuda_stream)
{
    if (!h) return MPCB200_E_INVALID;
    CK(cudaSetDevice(h->device));
    CK(cudaStreamSynchronize(h->stream));
    h->stream = cuda_stream ? (cudaStream_t)cuda_stream : h->own_stream;
    return 0;
}

extern "C" int mpcb200_set_option(mpcb200_handle* h, int option, int value)
{
    if (!h) return MPCB200_E_INVALID;
    if (option == MPCB200_OPT_SOLVE_MODE && value >= 0 && value <= 1) { h->solve_mode = value; return 0; }
    if (option == MPCB200_OPT_CTAS_PER_SM && value >= 0 && value <= 32) { h->max_ctas_per_sm = value; return 0; }
    if (option == MPCB200_OPT_ORDER_BY_HISTORY && value >= 0 && value <= 1) { h->order_by_history = value; return 0; }
    if (option == MPCB200_OPT_SM_PHASE_SYNC && value >= -1 && value <= 2) { h->sm_phase_sync = value; return 0; }
    return set_err(h, MPCB200_E_INVALID, "unknown option or value");
}

extern "C" int mpcb200_set_timing(mpcb200_handle* h, unsigned phase_mask)
{
    if (!h) return MPCB200_E_INVALID;
    h->timing_mask = phase_mask;
    return 0;
}

extern "C" int mpcb200_time_phase(mpcb200_handle* h, int phase, int B, int reps, int flush_l2, double* ms_per_launch)
{
    int rc = check_batch(h, B);
    if (rc) return rc;
    if (reps < 1) reps = 1;
    CK(cudaSetDevice(h->device));
    double total = 0.0;
    for (int r = 0; r < reps; ++r)
    {
        if (flush_l2) { flush_kernel<<<148 * 8, 256, 0, h->stream>>>(h->d_flush, h->flush_n); CK(cudaGetLastError()); }
        CK(cudaEventRecord(h->t0, h->stream));
        if ((rc = launch_phase(h, phase, B, 0, 1, nullptr, false))) return rc;
        CK(cudaEventRecord(h->t1, h->stream));
        CK(cudaStreamSynchronize(h->stream));
        float ms = 0.f;
        CK(cudaEventElapsedTime(&ms, h->t0, h->t1));
        total += ms;
    }
    if (ms_per_launch) *ms_per_launch = total / reps;
    return 0;
}

extern "C" int mpcb200_stats_get(const mpcb200_handle* hc, mpcb200_stats* out)
{
    mpcb200_handle* h = const_cast<mpcb200_handle*>(hc);
    if (!h || !out) return MPCB200_E_INVALID;
    CK(cudaSetDevice(h->device));
    CK(cudaStreamSynchronize(h->stream));
    int rc = collect_fused_counters(h);   // also picks up the counters of phase-wise KKT launches
    if (rc) return rc;
    CK(cudaStreamSynchronize(h->stream));
    *out = h->stats;
    return 0;
}
extern "C" int mpcb200_stats_reset(mpcb200_handle* h)
{
    if (!h) return MPCB200_E_INVALID;
    memset(&h->stats, 0, sizeof(h->stats));
    CK(cudaSetDevice(h->device));
    CK(cudaMemsetAsync(h->d_counters, 0, CNT_WORDS * 8, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    return 0;
}
extern "C" int mpcb200_export_controls(mpcb200_handle* h, void* dst_dev)
{
    if (!h || h->batch.B < 1 || !dst_dev) return set_err(h, MPCB200_E_INVALID, "nothing to export");
    CK(cudaSetDevice(h->device));
    CK(cudaMemcpyAsync(dst_dev, h->batch.upacked, (size_t)h->batch.B * (h->cfg.n - 1) * 16, cudaMemcpyDeviceToDevice, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    return 0;
}
// costmap -> point obstacles on the device.  Poses come from the host (host_pose) or are already on the device (dev_pose: the x0 array
// of a step); lists go to d_count / d_type / d_params ([B], [B][M], [B][M][7]; nullptr: scratch of this call).
struct CostmapOut { int* count; int* found; int* type; double* params; };
static int costmap_run(mpcb200_handle* h, int B, const mpcb200_costmaps* maps, const double* host_pose, const double* dev_pose, double behind_robot_dist,
                       int max_per_instance, int* d_count, int* d_type, double* d_params, CostmapOut* out)
{
    if (B < 1 || !maps || !maps->cost || !maps->origin || max_per_instance < 1)
        return set_err(h, MPCB200_E_INVALID, "costmap_obstacles: B >= 1, maps, poses and output arrays are required");
    if (maps->size_x < 2 || maps->size_y < 2 || !(maps->resolution > 0)) return set_err(h, MPCB200_E_INVALID, "costmap_obstacles: maps of at least 2 x 2 cells with a positive resolution");
    const size_t W = (size_t)maps->size_x, H = (size_t)maps->size_y, M = (size_t)max_per_instance;
    const int nrb = (int)((H - 1 + 31) / 32);            // 32-row blocks of the rows the reference visits
    const int ncg = (int)((W + MARK_COLS - 1) / MARK_COLS); // 16-column groups per row
    const int Wp = ncg * MARK_COLS;                      // mask row pitch: sixteen columns per marking thread
    const size_t mask_words = (size_t)B * nrb * Wp;
    const size_t need = (size_t)B * W * H + 16 + (size_t)B * 5 * 8 + 2 * (size_t)B * 4 + (size_t)B * M * (MPCB200_OBST_STRIDE * 8 + 4) +
                        mask_words * 4 + 512;
    const int rc = grow(h, h->d_cm, h->cm_cap, need);
    if (rc) return rc;
    // carve the scratch: 16-byte aligned pieces first (mask rows are stored as uint4), then ints, then the maps
    char* p = h->d_cm;
    unsigned* d_mask = (unsigned*)p; p += mask_words * 4;
    double* s_params = (double*)p; p += (size_t)B * M * MPCB200_OBST_STRIDE * 8;
    double* d_origin = (double*)p; p += (size_t)B * 2 * 8;
    double* d_pose = (double*)p; p += (size_t)B * 3 * 8;
    int* s_count = (int*)p; p += (size_t)B * 4;
    int* d_found = (int*)p; p += (size_t)B * 4;
    int* s_type = (int*)p; p += (size_t)B * M * 4;
    p = (char*)(((uintptr_t)p + 15) & ~(uintptr_t)15);
    unsigned char* d_cost = (unsigned char*)p;            // 16-byte aligned (16-byte loads when size_x % 16 == 0)
    if (!d_count) d_count = s_count;
    if (!d_type) d_type = s_type;
    if (!d_params) d_params = s_params;
    CK(cudaMemcpyAsync(d_cost, maps->cost, (size_t)B * W * H, cudaMemcpyHostToDevice, h->stream));
    CK(cudaMemcpyAsync(d_origin, maps->origin, (size_t)B * 16, cudaMemcpyHostToDevice, h->stream));
    if (host_pose) CK(cudaMemcpyAsync(d_pose, host_pose, (size_t)B * 24, cudaMemcpyHostToDevice, h->stream));
    h->stats.h2d_bytes += (long long)((size_t)B * W * H + (size_t)B * (host_pose ? 40 : 16));
    CostmapArgs a{maps->size_x, maps->size_y, maps->resolution, behind_robot_dist, d_cost, d_origin, host_pose ? d_pose : dev_pose};
    const dim3 grid_mark((unsigned)(((size_t)B * ncg * nrb + 255) / 256));
    // slots behind count[b] are padding: zeroed, so that what goes back to the caller (and on into step_batch) is defined
    CK(cudaMemsetAsync(d_type, 0, (size_t)B * M * 4, h->stream));
    CK(cudaMemsetAsync(d_params, 0, (size_t)B * M * MPCB200_OBST_STRIDE * 8, h->stream));
    CK(cudaEventRecord(h->c0, h->stream));
    if (W % 16 == 0) costmap_mark_kernel<16><<<grid_mark, 256, 0, h->stream>>>(a, B, nrb, ncg, Wp, d_mask);
    else if (W % 4 == 0) costmap_mark_kernel<4><<<grid_mark, 256, 0, h->stream>>>(a, B, nrb, ncg, Wp, d_mask);
    else costmap_mark_kernel<1><<<grid_mark, 256, 0, h->stream>>>(a, B, nrb, ncg, Wp, d_mask);
    costmap_emit_kernel<<<B, 256, 0, h->stream>>>(a, B, nrb, Wp, d_mask, max_per_instance, d_count, d_found, d_params, d_type);
    CK(cudaGetLastError());
    CK(cudaEventRecord(h->c1, h->stream));
    h->stats.launches_total += 2;
    out->count = d_count; out->found = d_found; out->type = d_type; out->params = d_params;
    return 0;
}

extern "C" int mpcb200_costmap_obstacles(mpcb200_handle* h, int B, const mpcb200_costmaps* maps, const double* robot_pose, double behind_robot_dist,
                                         int max_per_instance, int* count, int* found, int* type, double* params)
{
    if (!h) return MPCB200_E_INVALID;
    if (!robot_pose || !count || !type || !params) return set_err(h, MPCB200_E_INVALID, "costmap_obstacles: B >= 1, maps, poses and output arrays are required");
    CK(cudaSetDevice(h->device));
    CostmapOut o;
    int rc = costmap_run(h, B, maps, robot_pose, nullptr, behind_robot_dist, max_per_instance, nullptr, nullptr, nullptr, &o);
    if (rc) return rc;
    const size_t M = (size_t)max_per_instance;
    CK(cudaMemcpyAsync(count, o.count, (size_t)B * 4, cudaMemcpyDeviceToHost, h->stream));
    if (found) CK(cudaMemcpyAsync(found, o.found, (size_t)B * 4, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaMemcpyAsync(type, o.type, (size_t)B * M * 4, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaMemcpyAsync(params, o.params, (size_t)B * M * MPCB200_OBST_STRIDE * 8, cudaMemcpyDeviceToHost, h->stream));
    h->stats.d2h_bytes += (long long)((size_t)B * 8 + (size_t)B * M * (4 + MPCB200_OBST_STRIDE * 8));
    CK(cudaStreamSynchronize(h->stream));
    float ms = 0.f;
    CK(cudaEventElapsedTime(&ms, h->c0, h->c1));
    h->costmap_ms = ms;
    return MPCB200_OK;
}

// One planning cycle from the costmaps: MpcLocalPlannerROS::computeVelocityCommands' updateObstacleContainerWithCostmap
// (mpc_local_planner_ros.cpp:474-499) followed by Controller::step, for B robots, without the obstacle lists leaving the device:
// maps H2D -> mark / emit into the batch's obstacle arrays (robot pose = x0) -> association over the lists -> solve.
extern "C" int mpcb200_step_batch_costmap(mpcb200_handle* h, int B, const double* x0, const double* xf, const double* u_prev, double u_prev_dt,
                                          const mpcb200_costmaps* maps, double behind_robot_dist, int max_per_instance, const mpcb200_viapoints* vp,
                                          const double* x_init, const unsigned char* reinit, double* u_seq, double* x_seq, double* dt_out, int* status,
                                          double* kkt_err, int* iters, int* obst_found, double* solve_time_s)
{
    int rc = check_batch(h, B);
    if (rc) return rc;
    if (max_per_instance < 1 || max_per_instance > MAX_OBST_LIST) return set_err(h, MPCB200_E_UNSUPPORTED, "step_batch_costmap: 1..2048 obstacles per instance");
    CK(cudaSetDevice(h->device));
    Job& j = h->batch;
    // room for the lists in the batch's obstacle arrays
    if ((rc = reserve(h, j, (size_t)B, max_per_instance))) return rc;
    if ((rc = upload(h, j, (size_t)B, x0, xf, u_prev, u_prev_dt, nullptr, vp, x_init, reinit))) return rc;
    CostmapOut o;
    if ((rc = costmap_run(h, B, maps, nullptr, j.x0, behind_robot_dist, max_per_instance, j.obst_count, j.obst_type, j.obst, &o))) return rc;
    j.obst_max = max_per_instance;   // point obstacles only: no line-obstacle kernel variant needed
    if (h->solve_mode == 1 && (rc = scatter_batch(h))) return rc;
    if ((rc = solve_device(h, j, 0, solve_time_s))) return rc;
    if (obst_found) CK(cudaMemcpyAsync(obst_found, o.found, (size_t)B * 4, cudaMemcpyDeviceToHost, h->stream));
    rc = fetch(h, j, u_seq, x_seq, dt_out, status, kkt_err, iters);
    float ms = 0.f;
    if (!rc && cudaEventElapsedTime(&ms, h->c0, h->c1) == cudaSuccess) h->costmap_ms = ms;
    return rc;
}

extern "C" int mpcb200_check_feasible(mpcb200_handle* h, int B, const mpcb200_costmaps* maps, const double* x_seq, int n_poses, const double* footprint_xy,
                                      int n_footprint, double inscribed_radius, double circumscribed_radius, double min_resolution_angular,
                                      int look_ahead_idx, unsigned char* feasible)
{
    (void)circumscribed_radius;   // CostmapModel::footprintCost does not use it either
    if (!h) return MPCB200_E_INVALID;
    if (B < 1 || !maps || !maps->cost || !maps->origin || !feasible || n_footprint < 0 || (n_footprint > 0 && !footprint_xy))
        return set_err(h, MPCB200_E_INVALID, "check_feasible: B >= 1, maps, footprint and the output array are required");
    if (maps->size_x < 1 || maps->size_y < 1 || !(maps->resolution > 0)) return set_err(h, MPCB200_E_INVALID, "check_feasible: bad map geometry");
    if (!(inscribed_radius > 0) || !(min_resolution_angular > 0)) return set_err(h, MPCB200_E_INVALID, "check_feasible: inscribed_radius and min_resolution_angular must be > 0");
    const int n = x_seq ? n_poses : h->cfg.n;
    if (n < 1) return set_err(h, MPCB200_E_INVALID, "check_feasible: n_poses >= 1 required");
    if (!x_seq && (h->batch.B < B)) return set_err(h, MPCB200_E_INVALID, "check_feasible: no solved batch of this size on the device (pass x_seq)");
    CK(cudaSetDevice(h->device));
    const size_t W = (size_t)maps->size_x, H = (size_t)maps->size_y;
    const size_t need = (size_t)B * n * 24 + (size_t)B * 16 + (size_t)(n_footprint > 0 ? n_footprint : 1) * 16 + (size_t)B * W * H + (size_t)B + 256;
    const int rc = grow(h, h->d_fz, h->fz_cap, need);
    if (rc) return rc;
    char* p = h->d_fz;
    double* d_x = (double*)p; p += (size_t)B * n * 24;
    double* d_origin = (double*)p; p += (size_t)B * 16;
    double* d_fp = (double*)p; p += (size_t)(n_footprint > 0 ? n_footprint : 1) * 16;
    unsigned char* d_cost = (unsigned char*)p; p += (size_t)B * W * H;
    unsigned char* d_ok = (unsigned char*)p;
    CK(cudaMemcpyAsync(d_cost, maps->cost, (size_t)B * W * H, cudaMemcpyHostToDevice, h->stream));
    CK(cudaMemcpyAsync(d_origin, maps->origin, (size_t)B * 16, cudaMemcpyHostToDevice, h->stream));
    if (n_footprint > 0) CK(cudaMemcpyAsync(d_fp, footprint_xy, (size_t)n_footprint * 16, cudaMemcpyHostToDevice, h->stream));
    if (x_seq) CK(cudaMemcpyAsync(d_x, x_seq, (size_t)B * n * 24, cudaMemcpyHostToDevice, h->stream));
    h->stats.h2d_bytes += (long long)((size_t)B * W * H + (size_t)B * 16 + (size_t)n_footprint * 16 + (x_seq ? (size_t)B * n * 24 : 0));
    FeasArgs a{maps->size_x, maps->size_y, maps->resolution, d_cost, d_origin, x_seq ? d_x : h->batch.xseq.v, n, d_fp, n_footprint,
               inscribed_radius, min_resolution_angular, look_ahead_idx};
    feasible_kernel<<<grid_for(B, WARPS_PER_CTA), WARPS_PER_CTA * 32, 0, h->stream>>>(a, B, d_ok);
    h->stats.launches_total += 1;
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(feasible, d_ok, (size_t)B, cudaMemcpyDeviceToHost, h->stream));
    h->stats.d2h_bytes += B;
    CK(cudaStreamSynchronize(h->stream));
    return MPCB200_OK;
}

extern "C" double mpcb200_costmap_last_ms(const mpcb200_handle* h) { return h ? h->costmap_ms : 0.0; }

extern "C" int mpcb200_flush_l2(mpcb200_handle* h)
{
    if (!h) return MPCB200_E_INVALID;
    CK(cudaSetDevice(h->device));
    flush_kernel<<<148 * 8, 256, 0, h->stream>>>(h->d_flush, h->flush_n);
    CK(cudaGetLastError());
    CK(cudaStreamSynchronize(h->stream));
    return 0;
}

// =================================================================================================================
// several devices of one node behind one handle (SURVEY 8e): instances are independent, so the batch is cut into contiguous
// blocks, one per device; every device solves its block with its own handle on its own stream (one host thread each), and ONE
// NCCL all-gather over NVLink leaves the packed optimal controls of the whole batch on every device.  No other collective.
// NCCL is loaded at run time (dlopen) when a multi-device handle is created: the single-device library has no NCCL dependency.
// =================================================================================================================
#include <dlfcn.h>
#include <thread>

struct NcclApi
{
    void* lib = nullptr;
    int (*CommInitAll)(void**, int, const int*) = nullptr;
    int (*CommDestroy)(void*) = nullptr;
    int (*AllGather)(const void*, void*, size_t, int, void*, cudaStream_t) = nullptr;
    int (*GroupStart)() = nullptr;
    int (*GroupEnd)() = nullptr;
    const char* (*GetErrorString)(int) = nullptr;
};
#define MPC_NCCL_FLOAT64 8   /* ncclFloat64 / ncclDouble (nccl.h) */

struct mpcb200_multi
{
    int n_dev = 0, max_per = 0, n = 0;
    std::vector<int> devices;
    std::vector<mpcb200_handle*> h;
    std::vector<void*> comm;
    std::vector<Dev<double>> d_all;  // per device: gathered packed controls [n_dev][max_per][N-1][2]
    NcclApi nccl;
    std::string err;
};
static std::string g_multi_err = "";
static int multi_err(mpcb200_multi* m, int code, const std::string& msg) { if (m) m->err = msg; else g_multi_err = msg; return code; }

static bool load_nccl(NcclApi& a, std::string& why)
{
    const char* names[] = {"libnccl.so.2", "libnccl.so"};
    for (const char* nm : names) { a.lib = dlopen(nm, RTLD_NOW | RTLD_GLOBAL); if (a.lib) break; }
    if (!a.lib) { why = std::string("NCCL not found (dlopen libnccl.so.2): ") + (dlerror() ? dlerror() : ""); return false; }
#define NSYM(field, name) a.field = (decltype(a.field))dlsym(a.lib, name); if (!a.field) { why = std::string("NCCL symbol missing: ") + name; return false; }
    NSYM(CommInitAll, "ncclCommInitAll") NSYM(CommDestroy, "ncclCommDestroy") NSYM(AllGather, "ncclAllGather")
    NSYM(GroupStart, "ncclGroupStart") NSYM(GroupEnd, "ncclGroupEnd") NSYM(GetErrorString, "ncclGetErrorString")
#undef NSYM
    return true;
}

extern "C" void mpcb200_destroy_multi(mpcb200_multi* m)
{
    if (!m) return;
    for (size_t r = 0; r < m->comm.size(); ++r) if (m->comm[r] && m->nccl.CommDestroy) m->nccl.CommDestroy(m->comm[r]);
    for (size_t r = 0; r < m->d_all.size(); ++r) { cudaSetDevice(m->devices[r]); m->d_all[r].reset(); }
    for (auto* h : m->h) if (h) mpcb200_destroy(h);
    delete m;
}

extern "C" int mpcb200_create_multi(const mpcb200_config* cfg, int max_batch_total, const int* devices, int n_devices, mpcb200_multi** out)
{
    if (!cfg || !out || max_batch_total < 1 || !devices || n_devices < 1) return multi_err(nullptr, MPCB200_E_INVALID, "bad arguments");
    mpcb200_multi* m = new mpcb200_multi();
    m->n_dev = n_devices; m->n = cfg->n;
    m->max_per = (max_batch_total + n_devices - 1) / n_devices;
    m->devices.assign(devices, devices + n_devices);
    m->h.assign(n_devices, nullptr); m->comm.assign(n_devices, nullptr); m->d_all = std::vector<Dev<double>>(n_devices);
    for (int r = 0; r < n_devices; ++r)
    {
        const int rc = mpcb200_create(cfg, m->max_per, devices[r], &m->h[r]);
        if (rc) { const std::string e = mpcb200_last_error(nullptr); mpcb200_destroy_multi(m); return multi_err(nullptr, rc, e); }
    }
    if (n_devices > 1)
    {
        std::string why;
        if (!load_nccl(m->nccl, why)) { mpcb200_destroy_multi(m); return multi_err(nullptr, MPCB200_E_UNSUPPORTED, why); }
        const int nrc = m->nccl.CommInitAll(m->comm.data(), n_devices, devices);
        if (nrc != 0) { const std::string e = std::string("ncclCommInitAll: ") + m->nccl.GetErrorString(nrc); mpcb200_destroy_multi(m); return multi_err(nullptr, MPCB200_E_CUDA, e); }
    }
    const size_t words = (size_t)n_devices * m->max_per * (cfg->n - 1) * 2;
    for (int r = 0; r < n_devices; ++r)
    {
        if (cudaSetDevice(devices[r]) != cudaSuccess || alloc(m->d_all[r], words) != cudaSuccess)
        { mpcb200_destroy_multi(m); return multi_err(nullptr, MPCB200_E_CUDA, "cudaMalloc of the gathered controls failed"); }
    }
    *out = m;
    return MPCB200_OK;
}

extern "C" const char* mpcb200_multi_last_error(const mpcb200_multi* m) { return m ? m->err.c_str() : g_multi_err.c_str(); }
extern "C" mpcb200_handle* mpcb200_multi_handle(mpcb200_multi* m, int rank) { return (m && rank >= 0 && rank < m->n_dev) ? m->h[rank] : nullptr; }
extern "C" int mpcb200_multi_device_controls(mpcb200_multi* m, int rank, void** dev_ptr, long long* n_doubles)
{
    if (!m || rank < 0 || rank >= m->n_dev) return MPCB200_E_INVALID;
    if (dev_ptr) *dev_ptr = m->d_all[rank];
    if (n_doubles) *n_doubles = (long long)m->n_dev * m->max_per * (m->n - 1) * 2;
    return MPCB200_OK;
}

extern "C" int mpcb200_multi_fetch_controls(mpcb200_multi* m, int rank, double* host)
{
    if (!m || rank < 0 || rank >= m->n_dev || !host) return MPCB200_E_INVALID;
    if (cudaSetDevice(m->devices[rank]) != cudaSuccess ||
        cudaMemcpy(host, m->d_all[rank], (size_t)m->n_dev * m->max_per * (m->n - 1) * 16, cudaMemcpyDeviceToHost) != cudaSuccess)
        return multi_err(m, MPCB200_E_CUDA, "copy of the gathered controls failed");
    return MPCB200_OK;
}

extern "C" int mpcb200_step_batch_multi(mpcb200_multi* m, int B, const double* x0, const double* xf, const double* u_prev, double u_prev_dt,
                                        const mpcb200_obstacles* obst, const mpcb200_viapoints* vp, const double* x_init, const unsigned char* reinit,
                                        double* u_seq, double* x_seq, double* dt_out, int* status, double* kkt_err, int* iters, double* solve_time_s)
{
    if (!m) return MPCB200_E_INVALID;
    if (B < 1 || B > m->n_dev * m->max_per) return multi_err(m, MPCB200_E_INVALID, "batch size out of range");
    const int G = m->n_dev, N = m->n;
    const int per = (B + G - 1) / G;   // contiguous blocks: device r gets instances [r per, min((r+1) per, B))
    std::vector<int> rcs(G, 0);
    std::vector<double> secs(G, 0.0);
    std::vector<std::thread> th;
    for (int r = 0; r < G; ++r)
    {
        const int b0 = r * per, nb = std::max(0, std::min(per, B - b0));
        if (nb == 0) continue;
        th.emplace_back([=, &rcs, &secs]() {
            mpcb200_obstacles ob; mpcb200_viapoints vv;
            const mpcb200_obstacles* pob = nullptr; const mpcb200_viapoints* pvp = nullptr;
            if (obst && obst->count && obst->max_per_instance > 0)
            {
                const size_t M = (size_t)obst->max_per_instance;
                ob.max_per_instance = obst->max_per_instance; ob.count = obst->count + b0; ob.type = obst->type + (size_t)b0 * M;
                ob.params = obst->params + (size_t)b0 * M * MPCB200_OBST_STRIDE;
                pob = &ob;
            }
            if (vp && vp->count && vp->max_per_instance > 0)
            {
                vv.max_per_instance = vp->max_per_instance; vv.count = vp->count + b0; vv.poses = vp->poses + (size_t)b0 * vp->max_per_instance * 3;
                pvp = &vv;
            }
            rcs[r] = mpcb200_step_batch(m->h[r], nb, x0 + (size_t)b0 * 3, xf + (size_t)b0 * 3, u_prev ? u_prev + (size_t)b0 * 2 : nullptr, u_prev_dt, pob, pvp,
                                        x_init ? x_init + (size_t)b0 * N * 3 : nullptr, reinit ? reinit + b0 : nullptr,
                                        u_seq ? u_seq + (size_t)b0 * N * 2 : nullptr, x_seq ? x_seq + (size_t)b0 * N * 3 : nullptr, dt_out ? dt_out + b0 : nullptr,
                                        status ? status + b0 : nullptr, kkt_err ? kkt_err + b0 : nullptr, iters ? iters + b0 : nullptr, &secs[r]);
        });
    }
    for (auto& t : th) t.join();
    for (int r = 0; r < G; ++r)
        if (rcs[r]) return multi_err(m, rcs[r], std::string("device ") + std::to_string(m->devices[r]) + ": " + mpcb200_last_error(m->h[r]));
    // ---- all-gather of the packed optimal controls: every device ends up with u* of every instance ----
    const size_t count = (size_t)per * (N - 1) * 2;
    if (G > 1)
    {
        int nrc = m->nccl.GroupStart();
        for (int r = 0; r < G && nrc == 0; ++r)
        {
            cudaSetDevice(m->devices[r]);
            nrc = m->nccl.AllGather(m->h[r]->batch.upacked, m->d_all[r], count, MPC_NCCL_FLOAT64, m->comm[r], m->h[r]->stream);
        }
        const int erc = m->nccl.GroupEnd();
        if (nrc == 0) nrc = erc;
        if (nrc != 0) return multi_err(m, MPCB200_E_CUDA, std::string("ncclAllGather: ") + m->nccl.GetErrorString(nrc));
        for (int r = 0; r < G; ++r)
        {
            cudaSetDevice(m->devices[r]);
            if (cudaStreamSynchronize(m->h[r]->stream) != cudaSuccess) return multi_err(m, MPCB200_E_CUDA, "stream synchronisation after the all-gather failed");
        }
    }
    else
    {
        cudaSetDevice(m->devices[0]);
        if (cudaMemcpyAsync(m->d_all[0], m->h[0]->batch.upacked, count * 8, cudaMemcpyDeviceToDevice, m->h[0]->stream) != cudaSuccess ||
            cudaStreamSynchronize(m->h[0]->stream) != cudaSuccess)
            return multi_err(m, MPCB200_E_CUDA, "copy of the controls failed");
    }
    if (solve_time_s) { double mx = 0.0; for (double s_ : secs) mx = s_ > mx ? s_ : mx; *solve_time_s = mx; }
    return MPCB200_OK;
}
