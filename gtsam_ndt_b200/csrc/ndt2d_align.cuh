// The align machinery shared by the kernels that run SPEC 5 on the device (k_align, k_align_block in ndt2d_kernels.cu;
// k_pairs_fused in ndt2d_pairs.cu): the per-warp LM state, one evaluation into it, THE Levenberg-Marquardt loop and the
// result write-back. Reference file:line: none (the mount is /root/reference/README.md:1 only); arithmetic follows SPEC.md.
#pragma once
#include "ndt2d_device.cuh"

namespace ndt2d {

// SPEC 5, one pyramid level. Every lane carries the same f64 state (the butterfly reduction gives
// all lanes identical sums), so the control flow is warp-uniform and needs no broadcast.
// where a warp reads its scan from: its padded shared-memory slot or global memory
struct ScanView {
    const float2 *pts;
    int n;
};

// Per-warp LM state. Every lane computes the same f64 values (the butterfly gives all lanes identical sums), so one
// copy per warp in shared memory is the whole solver state: nothing but a few ints stays live in registers
// across the evaluation call (register spills of warp-uniform doubles would cost 32 lanes x 8 B of local memory each).
struct WarpState {
    double v[10];   // the last accepted evaluation (SPEC 5's E)
    double t[10];   // the trial evaluation
    double p[3];    // the current pose
    double pn[3];   // the trial pose
    double lambda;
    int count, tcount;
};

// ------------------------------------------------------------------------------------------------
// Helper warps (k_align<..., HELP>). The batch is a queue of scans, one warp per scan; a scan takes 10-90 evaluations, so a
// launch ends with a few long scans running alone (and a batch of fewer scans than resident warps never fills the GPU).
// A warp that finds the queue empty therefore does not exit: it attaches itself to a warp of its block that still
// holds a scan (its OWNER) and, for every evaluation the owner posts, computes the SPEC 4 factors of the last few 64-point
// steps and parks them in its own - now unused - shared-memory slot. The owner evaluates the first steps itself and then
// applies the parked factors in step order, so the partial sums are the bits of the unhelped evaluation (the same
// mechanism as k_align_block, with the number of helpers changing from one evaluation to the next).
// Protocol, all in shared memory of the block (volatile accesses + __threadfence_block):
//   helper -> owner: claims entry h of desk.helper[] by atomicCAS (entries fill from the front and are never released);
//   owner -> helpers: one word desk.post = (evaluation number << 8 | helpers counted on << 4 | steps per helper), written
//            after desk.level / desk.n / the trial pose ws->pn; a helper with h >= helpers counted on skips that evaluation;
//   helper -> owner: desk.done[h] = evaluation number once its factors are parked.
// A warp turns helper only after it has seen the queue empty, and the queue head only grows: an owner that has helpers
// never starts another scan, so desks are initialised once per launch. desk.active is 1 from the start of the launch
// until the warp has seen the empty queue itself (a helper must not mistake a warp between two scans for a finished one).
// ------------------------------------------------------------------------------------------------
static constexpr int ALIGN_THREADS = 128;
static constexpr unsigned kHelpSleepNs = 64;   // a waiting helper sleeps between two polls of its owner's desk
static constexpr int kAlignWarps = ALIGN_THREADS / 32;
static constexpr int kMaxHelpers = kAlignWarps - 1 < 7 ? kAlignWarps - 1 : 7;
static constexpr unsigned kNoHelper = 0xffffffffu;

struct HelpDesk {
    unsigned post;                 // the evaluation helpers are wanted for (0: none yet); written by the owner only
    unsigned cur;                  // owner-private: `post` if the evaluation in progress is helped, else 0
    unsigned active;               // the warp may still own a scan (it has not seen the queue empty yet)
    unsigned slot_bytes;           // bytes of one warp's scan slot (= where a helper parks its factors)
    int level, n;                  // of the posted evaluation
    unsigned helper[7];            // warp number of helper h
    unsigned done[7];              // evaluation number of helper h's latest parked factors
};
static_assert(sizeof(HelpDesk) % 16 == 0, "scan slots follow the desks and must stay 16-byte aligned");

__device__ __forceinline__ unsigned lds_volatile(const unsigned *p) { return *reinterpret_cast<const volatile unsigned *>(p); }
__device__ __forceinline__ void sts_volatile(unsigned *p, unsigned v) { *reinterpret_cast<volatile unsigned *>(p) = v; }

// dynamic shared memory of a k_align block: [WarpState x warps][HelpDesk x warps (HELP)][scan slot x warps]
__device__ __forceinline__ unsigned char *align_smem()
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    return smem_raw;
}
__device__ __forceinline__ HelpDesk *help_desk(int warp)
{
    return reinterpret_cast<HelpDesk *>(align_smem() + kAlignWarps * sizeof(WarpState)) + warp;
}
__device__ __forceinline__ unsigned char *help_slots() { return align_smem() + kAlignWarps * (sizeof(WarpState) + sizeof(HelpDesk)); }

// The owner's side of one helped evaluation. Nothing of it stays in registers across the point loop: finish() re-reads the
// plan from the desk.
struct HelpPlan {
    static constexpr bool on = true;
    unsigned helped_steps;         // steps left to the helpers (0: nobody helps)
    __device__ __forceinline__ unsigned own_steps(unsigned nsteps) const { return nsteps - helped_steps; }
    __device__ __forceinline__ void finish(Partials &S, int &cnt, int lane) const
    {
        const HelpDesk *d = help_desk(threadIdx.x >> 5);
        const unsigned cur = d->cur;
        if (cur == 0) return;
        const unsigned nh = (cur >> 4) & 15u, hs = cur & 15u, seq = cur >> 8;
        const unsigned sb = d->slot_bytes;
#pragma unroll 1
        for (unsigned h = 0; h < nh; ++h) {
            while (lds_volatile(&d->done[h]) != seq) { }
            __threadfence_block();
            const u64 *fac = reinterpret_cast<const u64 *>(help_slots() + (size_t)d->helper[h] * sb) + lane;
#pragma unroll 1
            for (unsigned e = 0; e < hs; ++e) apply_parked(fac + (size_t)e * FACTOR_WORDS * 32, S, cnt);
        }
    }
};

// Owner, before an evaluation of `n` points on pyramid level `level` at ws->pn: count the helpers that have attached
// themselves, split the steps and post the evaluation.
__device__ __forceinline__ HelpPlan post_help(int level, int n)
{
    const int lane = threadIdx.x & 31;
    HelpDesk *d = help_desk(threadIdx.x >> 5);
    const unsigned nsteps = (unsigned)(n + 63) >> 6;
    unsigned nh = 0;
#pragma unroll
    for (int h = 0; h < kMaxHelpers; ++h) nh += (nh == (unsigned)h && lds_volatile(&d->helper[h]) != kNoHelper) ? 1u : 0u;
    unsigned hs = min(min(d->slot_bytes / kFactorBytes, 15u), nsteps / (nh + 1u));
    if (hs == 0) nh = 0;
    const unsigned cur = nh ? ((((d->post >> 8) + 1u) << 8) | (nh << 4) | hs) : 0u;
    __syncwarp();
    if (lane == 0) {
        d->cur = cur;
        if (nh) {
            d->level = level;
            d->n = n;
            __threadfence_block();       // level, n and the trial pose (ws->pn, written before the warp barrier above) first
            sts_volatile(&d->post, cur);
        }
    }
    __syncwarp();
    HelpPlan hp;
    hp.helped_steps = nh * hs;
    return hp;
}

// A warp without a scan: serve the owners of this block until none is left. lv = the launch's pyramid levels.
template <int OV>
__device__ __noinline__ void help_others(const LevelDev *lv)
{
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (;;) {
        int o = -1;
        unsigned hidx = 0;
        if (lane == 0) {
            for (int tries = 0; tries < 2 * kAlignWarps && o < 0; ++tries) {
                int best = -1;
                unsigned bestc = kMaxHelpers;
                for (int w = 0; w < kAlignWarps; ++w) {           // the owner with the fewest helpers
                    if (w == warp || !lds_volatile(&help_desk(w)->active)) continue;
                    unsigned c = 0;
                    for (int h = 0; h < kMaxHelpers; ++h) c += lds_volatile(&help_desk(w)->helper[h]) != kNoHelper ? 1u : 0u;
                    if (c < bestc) { best = w; bestc = c; }
                }
                if (best < 0) break;
                for (unsigned h = bestc; h < (unsigned)kMaxHelpers; ++h)
                    if (atomicCAS(&help_desk(best)->helper[h], kNoHelper, (unsigned)warp) == kNoHelper) { o = best; hidx = h; break; }
            }
        }
        o = __shfl_sync(0xffffffffu, o, 0);
        hidx = __shfl_sync(0xffffffffu, hidx, 0);
        if (o < 0) return;
        HelpDesk *d = help_desk(o);
        const unsigned sb = d->slot_bytes;
        const volatile double *opose = reinterpret_cast<const WarpState *>(align_smem())[o].pn;
        const float2 *opts = reinterpret_cast<const float2 *>(help_slots() + (size_t)o * sb);
        u64 *mine = reinterpret_cast<u64 *>(help_slots() + (size_t)warp * sb) + lane;
        unsigned last = 0;
        for (;;) {
            unsigned post;
            while ((post = lds_volatile(&d->post)) == last && lds_volatile(&d->active)) __nanosleep(kHelpSleepNs);
            if (post == last) break;                              // the owner has finished its scan
            last = post;
            const unsigned nh = (post >> 4) & 15u, hs = post & 15u;
            if (hidx >= nh) continue;                             // attached after this evaluation was planned
            __threadfence_block();
            const int level = *reinterpret_cast<const volatile int *>(&d->level), n = *reinterpret_cast<const volatile int *>(&d->n);
            const LevelDev *L = lv + level;
            const PosePk P = pose_pack(pose_for_level(opose[0], opose[1], opose[2], *L));
            const LatticePk G = lattice_pack<OV>(*L, TABLE_DENSE);
            const float4 *__restrict__ cells = L->cells;
            const unsigned first = (((unsigned)(n + 63) >> 6) - nh * hs) + hidx * hs;
#pragma unroll 1
            for (unsigned e = 0; e < hs; ++e) {
                Fetched<OV> F;
                fetch<OV, true, TABLE_DENSE>(cells, G, P, opts, n, (int)((first + e) << 6) + lane, F);
                Factors X;
                int c = 0;
                F.A.XY = local_xy(G, F.A.df, 0);
                F.B.XY = local_xy(G, F.B.df, 0);
                cell_factors<true>(F.cA[0], F.cB[0], F.A, F.B, X, c);
                park_factors(X, mine + (size_t)e * FACTOR_WORDS * 32);
            }
            __syncwarp();
            __threadfence_block();
            if (lane == 0) sts_volatile(&d->done[hidx], post >> 8);
        }
    }
}

// One SPEC 4 evaluation at the trial pose ws->pn, result to ws->t / ws->tcount; lane t stores sum t.
// HELP: `level` is L's number in the launch's pyramid (helpers look the level up themselves)
template <int OV, bool STAGED, int TABLE, bool HELP = false>
__device__ __forceinline__ void eval_to_smem_body(const LevelDev *L, const float2 *pts, int n, WarpState *ws, int level = 0)
{
    const int lane = threadIdx.x & 31;
    const double *pose = ws->pn;
    Eval E;
    if (HELP) {
        const HelpPlan hp = post_help(level, n);
        eval_warp<OV, true, STAGED, true, TABLE, false, HelpPlan>(*L, pts, n, pose_for_level(pose[0], pose[1], pose[2], *L), lane, E, hp);
    } else {
        eval_warp<OV, true, STAGED, true, TABLE>(*L, pts, n, pose_for_level(pose[0], pose[1], pose[2], *L), lane, E);
    }
    __syncwarp();
    ws->t[E.slot] = E.v[0]; // lanes holding the same sum store the same bits
    if (lane == 0) ws->tcount = E.count;
    __syncwarp();
}
// ... as a function of its own (the point loop then gets a register allocation independent of the f64 solver)
template <int OV, bool STAGED, int TABLE>
__device__ __noinline__ void eval_to_smem_call(const LevelDev *L, const float2 *pts, int n, WarpState *ws)
{
    eval_to_smem_body<OV, STAGED, TABLE>(L, pts, n, ws);
}
// k_align inlines the evaluation into the LM loop (r2g: 18.70 vs 18.17 M matches/s against the call - no spills at 80
// registers and both gathers of a step issue back to back). The fused pairs kernel calls it as a function: inlined, its
// code outgrows the instruction cache (r2h: 9.7 vs 10.8 M pairs/s).
template <int OV, bool STAGED, int TABLE, bool HELP = false>
__device__ __forceinline__ void eval_to_smem(const LevelDev *L, const float2 *pts, int n, WarpState *ws, int level = 0)
{
    if (HELP) eval_to_smem_body<OV, STAGED, TABLE, true>(L, pts, n, ws, level);
    else if (TABLE != TABLE_SHASH) eval_to_smem_body<OV, STAGED, TABLE>(L, pts, n, ws);
    else eval_to_smem_call<OV, STAGED, TABLE>(L, pts, n, ws);
}

// The threads that share one WarpState: a warp (k_align) or a whole block (k_align_block)
struct WarpScope {
    static __device__ __forceinline__ void sync() { __syncwarp(); }
    static __device__ __forceinline__ int id() { return threadIdx.x & 31; }
};
struct BlockScope {
    static __device__ __forceinline__ void sync() { __syncthreads(); }
    static __device__ __forceinline__ int id() { return threadIdx.x; }
};

// SPEC 5, one pyramid level, starting from and finishing in ws->p: THE Levenberg-Marquardt loop, shared by the
// warp-per-scan and the block-per-scan kernels. Every thread of the scope computes the same f64 values from the shared
// state, so the control flow is uniform. eval() evaluates the trial pose ws->pn into ws->t / ws->tcount and ends with a
// Scope::sync(). There is ONE call site: the first evaluation (at ws->p) runs as a trial at pn = p that is accepted
// unconditionally, so an inlined evaluation exists once in the kernel (round 2: the second copy had the worse register
// allocation - ten accumulator moves per 64 points - and it was the one that ran 11 times out of 12).
template <class Scope, class EvalFn>
__device__ __forceinline__ int lm_level(const ndt2d_params &P, int n, WarpState *ws, int &evals_total, EvalFn eval)
{
    const int id = Scope::id();
    if (id == 0) ws->lambda = P.lambda_init;
    if (id < 3) ws->pn[id] = ws->p[id];
    Scope::sync();
    int evals = 0, status = NDT2D_MAX_ITERATIONS;
    bool small = false;
    for (;;) {
        eval();
        evals += 1;
        double lambda = ws->lambda;
        const bool first = evals == 1;
        const bool better = first || ws->t[0] > ws->v[0];
        Scope::sync();
        if (better) {
            if (id < 10) ws->v[id] = ws->t[id];
            if (id == 10) ws->count = ws->tcount;
            if (id >= 11 && id < 14) ws->p[id - 11] = ws->pn[id - 11];
            if (!first) {
                lambda = fmax(lambda / P.lambda_down, P.lambda_min);
                if (id == 14) ws->lambda = lambda;
            }
            Scope::sync();
            if (first) {
                if (n == 0 || ws->count == 0) { status = NDT2D_NO_OVERLAP; break; }
            } else if (small) { status = NDT2D_CONVERGED; break; }
        } else {
            if (small) { status = NDT2D_CONVERGED; break; }
            lambda = lambda * P.lambda_up;
            if (id == 14) ws->lambda = lambda;
            Scope::sync();
            if (lambda > P.lambda_max) { status = NDT2D_STALLED; break; }
        }
        if (evals >= P.max_iterations) break;
        double d[3];
        bool stalled = false;
        {
            double g[3] = {ws->v[1], ws->v[2], ws->v[3]};
            double H6[6] = {ws->v[4], ws->v[5], ws->v[6], ws->v[7], ws->v[8], ws->v[9]};
            while (!solve3(g, H6, lambda, d)) {
                lambda = lambda * P.lambda_fail_up;
                if (lambda > P.lambda_max) { stalled = true; break; }
            }
        }
        if (stalled) { status = NDT2D_STALLED; break; }
        double n2 = d[0] * d[0] + d[1] * d[1]; // squared translation step: no sqrt unless the step is clamped
        if (n2 > P.max_step_trans * P.max_step_trans) {
            double sc = P.max_step_trans / sqrt(n2);
            d[0] *= sc; d[1] *= sc; d[2] *= sc; n2 = P.max_step_trans * P.max_step_trans;
        }
        if (fabs(d[2]) > P.max_step_rot) {
            double sc = P.max_step_rot / fabs(d[2]);
            d[0] *= sc; d[1] *= sc; d[2] *= sc; n2 = n2 * (sc * sc);
        }
        small = (n2 < P.eps_trans * P.eps_trans) && (fabs(d[2]) < P.eps_rot);
        Scope::sync();
        if (id == 0) {
            ws->pn[0] = ws->p[0] + d[0];
            ws->pn[1] = ws->p[1] + d[1];
            ws->pn[2] = ws->p[2] + d[2];
            ws->lambda = lambda;
        }
        Scope::sync();
    }
    evals_total += evals;
    return status;
}

// what align returns (SPEC 5): the state after the finest level, theta wrapped
__device__ __forceinline__ void write_result(const WarpState &E, int evals, int status, ndt2d_result *r)
{
    const double TWO_PI = 6.283185307179586476925286766559;
    r->pose[0] = E.p[0];
    r->pose[1] = E.p[1];
    r->pose[2] = E.p[2] - TWO_PI * rint(E.p[2] / TWO_PI);
    r->score = E.v[0];
    r->grad[0] = E.v[1]; r->grad[1] = E.v[2]; r->grad[2] = E.v[3];
    r->hessian[0] = E.v[4]; r->hessian[1] = E.v[5]; r->hessian[2] = E.v[6];
    r->hessian[3] = E.v[5]; r->hessian[4] = E.v[7]; r->hessian[5] = E.v[8];
    r->hessian[6] = E.v[6]; r->hessian[7] = E.v[8]; r->hessian[8] = E.v[9];
    r->iterations = evals;
    r->status = status;
    r->count = E.count;
    r->reserved = 0;
}

template <int OV, bool STAGED, int TABLE, bool HELP = false>
__device__ __forceinline__ int align_level(const LevelDev *L, const ndt2d_params &P, const ScanView &v, WarpState *ws,
                                           int &evals_total, int level = 0)
{
    return lm_level<WarpScope>(P, v.n, ws, evals_total, [&]() { eval_to_smem<OV, STAGED, TABLE, HELP>(L, v.pts, v.n, ws, level); });
}


} // namespace ndt2d
