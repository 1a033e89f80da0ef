// C-ABI layer of libndt2d.so (include/ndt2d.h): handle, device buffers, host<->device copies and
// kernel launches. No CPU compute path exists here: without a CUDA device ndt2d_create fails.
// Reference interface: none citable (/root/reference/README.md:1 is the whole mount); the entry points
// implement the matcher operations BASELINE.json's north_star names.
#include "ndt2d_host.h"

using namespace ndt2d;

namespace {

thread_local std::string g_create_error;

} // namespace

// helpers shared with the other host translation units are declared in ndt2d_host.h
namespace ndt2d {

int fail(ndt2d_matcher *m, int code, const char *fmt, ...)
{
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    if (m) m->err = buf; else g_create_error = buf;
    return code;
}


// forget the target; keep_memory: the per-level allocations stay for the next target (set_target after set_target)
void drop_target(ndt2d_matcher *m, bool keep_memory = false)
{
    for (int l = 0; l < NDT2D_MAX_LEVELS; ++l) {
        if (!keep_memory) m->mem[l].release();
        m->lv[l] = LevelDev{};
    }
    m->has_target = false;
    m->sums_valid = false;
}

// device memory of level l for the lattice in m->lv[l]: tables allocated and cleared
static int install_level(ndt2d_matcher *m, int l)
{
    LevelDev &L = m->lv[l];
    const int64_t nc = (int64_t)L.njx * L.njy;
    LevelMem &M = m->mem[l];
    const int64_t pad = LevelMem::zero_pad(L.njx);
    CK(m, M.ensure(nc, pad));
    // records, sums and counts share one allocation and are cleared by one memset (three launches fewer per level: a
    // target scan's tables are small, the launches were most of the clearing); the all-zero records after the table are
    // the gather targets of points outside the lattice and are never written again
    CK(m, cudaMemsetAsync(M.base, 0, M.bytes, m->cfg.stream));
    L.cells = M.cells;
    L.cnt = M.cnt;
    L.sums = M.sums;
    return NDT2D_OK;
}

// SPEC 2: geometry and tables of every level. bbox = {xmin, ymin, xmax, ymax}, used for auto-fit only. On failure the
// target is dropped.
static int setup_levels(ndt2d_matcher *m, const float bbox[4])
{
    for (int l = 0; l < m->nlevels; ++l) {
        LevelDev &L = m->lv[l];
        L = LevelDev{};
        int rc;
        if (level_geometry(L, m->res[l], m->prm.overlap, m->explicit_grid, m->gox, m->goy, m->gex, m->gey, bbox[0], bbox[1], bbox[2],
                           bbox[3]))
            rc = install_level(m, l);
        else if (L.nhx < 1 || L.nhy < 1)
            rc = fail(m, NDT2D_EINVAL, "level %d: empty lattice (%d x %d)", l, L.nhx, L.nhy);
        else
            rc = fail(m, NDT2D_EINVAL, "level %d: %lld cells exceed 2^31", l, (long long)L.njx * L.njy);
        if (rc) {
            drop_target(m);
            return rc;
        }
    }
    return NDT2D_OK;
}

// SPEC 3: accumulate src into every level of the target and finalise. touch (incremental update): finalise only the
// cells the points touch, with one list of them per level in b_idx (after the per-level list lengths)
static int accumulate_and_finalize(ndt2d_matcher *m, const TargetSrc &src, bool touch = false)
{
    const int64_t list_cap = src.n * (m->prm.overlap ? 4 : 1);
    LevelSet S;
    memset(&S, 0, sizeof(S));
    S.nlevels = m->nlevels;
    if (touch) {
        CK(m, m->b_idx.ensure(((size_t)list_cap * m->nlevels + NDT2D_MAX_LEVELS) * 4));
        S.nlist = m->b_idx.as<unsigned>();
    }
    for (int l = 0; l < m->nlevels; ++l) {
        LevelMem &M = m->mem[l];
        if (touch && !M.dirty) {
            CK(m, cudaMalloc(&M.dirty, (size_t)M.cap * 4));
            CK(m, cudaMemsetAsync(M.dirty, 0, (size_t)M.cap * 4, m->cfg.stream));
        }
        S.lv[l] = m->lv[l];
        S.cells[l] = M.cells;
        S.dirty[l] = M.dirty;
        if (touch) S.list[l] = S.nlist + NDT2D_MAX_LEVELS + l * list_cap;
    }
    CK(m, launch_build(m->cfg, S, m->prm, src, touch, &m->launches));
    return NDT2D_OK;
}

int check_level(ndt2d_matcher *m, int level)
{
    if (!m) return NDT2D_EINVAL;
    if (!m->has_target) return fail(m, NDT2D_ENOTARGET, "no target set");
    if (level < 0 || level >= m->nlevels) return fail(m, NDT2D_EINVAL, "level %d out of range [0, %d)", level, m->nlevels);
    return NDT2D_OK;
}

int upload(ndt2d_matcher *m, DevBuf &b, const void *src, size_t bytes)
{
    CK(m, b.ensure(bytes ? bytes : 16));
    if (bytes) CK(m, cudaMemcpyAsync(b.p, src, bytes, cudaMemcpyHostToDevice, m->cfg.stream));
    return NDT2D_OK;
}

// shared-memory slot capacity (points per warp) for the align kernel; 0 = read scans from global memory
static int align_cap_points(const ndt2d_matcher *m, int max_points)
{
    int cap = (max_points + 63) & ~63; // two NaN-padded planes per warp, 64 points per warp iteration
    if (cap < 64) cap = 64;
    if (align_smem_bytes(cap) > (size_t)m->cfg.max_smem_optin) return 0;
    return cap;
}

// SPEC 8 beam table, computed on the host with libm in f64 and rounded once, then cached on the device
int ensure_beams(ndt2d_matcher *m, int nbeams, double angle_min, double angle_inc)
{
    if (m->beams_n == nbeams && m->beams_amin == angle_min && m->beams_ainc == angle_inc) return NDT2D_OK;
    std::vector<float> tab((size_t)nbeams * 2);
    for (int i = 0; i < nbeams; ++i) {
        double phi = angle_min + (double)i * angle_inc;
        tab[2 * i] = (float)cos(phi);
        tab[2 * i + 1] = (float)sin(phi);
    }
    int rc = upload(m, m->b_beams, tab.data(), tab.size() * 4);
    if (rc) return rc;
    CK(m, cudaStreamSynchronize(m->cfg.stream)); // tab goes out of scope
    m->beams_n = nbeams; m->beams_amin = angle_min; m->beams_ainc = angle_inc;
    return NDT2D_OK;
}

int align_device(ndt2d_matcher *m, AlignArgs a, int max_points, double angle_min, double angle_inc)
{
    a.cap_points = align_cap_points(m, max_points);
    if (a.ranges) {     // LaserScan ranges are converted in the staging step, so they need the shared-memory slot
        if (a.cap_points == 0) return fail(m, NDT2D_EINVAL, "nbeams %d exceeds the shared-memory staging limit", a.nbeams);
        int rc = ensure_beams(m, a.nbeams, angle_min, angle_inc);
        if (rc) return rc;
        a.beams = m->b_beams.as<float2>();
    }
    for (int l = 0; l < m->nlevels; ++l) a.lv[l] = m->lv[l];
    a.nlevels = m->nlevels;
    a.prm = m->prm;
    if (!a.counter) a.counter = m->b_counter.as<unsigned int>();
    CK(m, launch_align(m->cfg, a, &m->launches));
    return NDT2D_OK;
}

// Host-buffer batch driver shared by the xy and ranges entry points. The input is cut into chunks; chunk
// copies run back to back on copy_stream, chunk kernels alternate between two work streams (so the tail
// of one chunk overlaps the head of the next) and each chunk's results are copied back as it finishes.
// The call returns after everything has completed (host-synchronous, like the rest of the host API).
struct ChunkPlan {
    int nchunks, per;
};

// Chunk size: a copy-bound call (f32 ranges, float2 points) wants small chunks, which shorten the un-overlapped first
// copy and last kernel (measured on PCIe 5 x16, 65 536 scans: 8192-scan chunks 10.1 M matches/s, 4096-scan chunks
// 10.7-11.5 M); a kernel-bound call (u16 ranges) wants large ones, since every chunk is a launch with its own partial
// last wave (15.9 M vs 15.1 M). About 18 MB per chunk gives 16 chunks for the former and 8 for the latter.
ChunkPlan plan_chunks(int nscans, size_t total_bytes)
{
    ChunkPlan p;
    p.nchunks = (int)((total_bytes + (18u << 20) - 1) / (18u << 20));
    if (p.nchunks > ndt2d_matcher::MAX_CHUNKS) p.nchunks = ndt2d_matcher::MAX_CHUNKS;
    if (p.nchunks < 1) p.nchunks = 1;
    p.per = (nscans + p.nchunks - 1) / p.nchunks;
    return p;
}

// chunk_desc(s0, s1, &dst, &src, &bytes): where the input of scans [s0, s1) goes on the device, where it comes from on the
// host, and how long it is. With an upload relay (ndt2d_set_upload_relay) about relay_frac of the chunks take the detour
// host -> relay GPU -> this GPU: their ev_chunk is recorded after the peer copy instead of after the direct one.
static void release_relay(ndt2d_matcher *m)
{
    if (m->relay_dev < 0) return;
    {
        DeviceGuard g(m->relay_dev);
        if (m->relay_stream) { cudaStreamSynchronize(m->relay_stream); cudaStreamDestroy(m->relay_stream); }
        for (cudaEvent_t &e : m->ev_relay) { if (e) cudaEventDestroy(e); e = nullptr; }
        if (m->relay_buf) cudaFree(m->relay_buf);
    }
    if (m->relay_peer_stream) {
        DeviceGuard g(m->device);
        cudaStreamSynchronize(m->relay_peer_stream);
        cudaStreamDestroy(m->relay_peer_stream);
    }
    m->relay_stream = m->relay_peer_stream = nullptr;
    m->relay_buf = nullptr;
    m->relay_cap = 0;
    m->relay_dev = -1;
    m->relay_frac = 0.0;
}

template <typename DescFn, typename LaunchFn>
int run_pipeline(ndt2d_matcher *m, int nscans, size_t total_bytes, ndt2d_result *res, DescFn chunk_desc, LaunchFn launch_chunk)
{
    const ChunkPlan pl = plan_chunks(nscans, total_bytes);
    const bool relay = m->relay_dev >= 0 && pl.nchunks > 1;
    if (relay && m->relay_cap < total_bytes) {          // the relay GPU mirrors the call's input buffer
        DeviceGuard g(m->relay_dev);
        if (m->relay_buf) { cudaStreamSynchronize(m->relay_stream); cudaFree(m->relay_buf); m->relay_buf = nullptr; m->relay_cap = 0; }
        CK(m, cudaMalloc(&m->relay_buf, total_bytes + total_bytes / 8));
        m->relay_cap = total_bytes + total_bytes / 8;
    }
    CK(m, cudaEventRecord(m->ev_begin, m->cfg.stream)); // earlier work on the handle's stream comes first
    CK(m, cudaStreamWaitEvent(m->copy_stream, m->ev_begin, 0));
    for (int i = 0; i < 2; ++i) CK(m, cudaStreamWaitEvent(m->work_stream[i], m->ev_begin, 0));
    if (relay) {
        CK(m, cudaStreamWaitEvent(m->relay_stream, m->ev_begin, 0));
        CK(m, cudaStreamWaitEvent(m->relay_peer_stream, m->ev_begin, 0));
    }
    unsigned char *base_dst = nullptr;
    for (int c = 0; c < pl.nchunks; ++c) {
        int s0 = c * pl.per, s1 = s0 + pl.per < nscans ? s0 + pl.per : nscans;
        void *dst = nullptr;
        const void *src = nullptr;
        size_t bytes = 0;
        if (s1 > s0) chunk_desc(s0, s1, &dst, &src, &bytes);
        if (c == 0) base_dst = static_cast<unsigned char *>(dst);
        // chunk c is relayed when the running share of relayed chunks falls behind relay_frac; the half-step phase keeps the
        // first chunk (it gates the start) and the last ones (a relayed chunk arrives after two hops) on the direct link
        const bool via = relay && bytes > 0 && c > 0 && (int)((c + 1) * m->relay_frac + 0.5) > (int)(c * m->relay_frac + 0.5);
        if (via) {
            unsigned char *mid = static_cast<unsigned char *>(m->relay_buf) + (static_cast<unsigned char *>(dst) - base_dst);
            {
                DeviceGuard g(m->relay_dev);
                CK(m, cudaMemcpyAsync(mid, src, bytes, cudaMemcpyHostToDevice, m->relay_stream));
                CK(m, cudaEventRecord(m->ev_relay[c], m->relay_stream));
            }
            CK(m, cudaStreamWaitEvent(m->relay_peer_stream, m->ev_relay[c], 0));
            CK(m, cudaMemcpyPeerAsync(dst, m->device, mid, m->relay_dev, bytes, m->relay_peer_stream));
            CK(m, cudaEventRecord(m->ev_chunk[c], m->relay_peer_stream));
        } else {
            if (bytes > 0) CK(m, cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, m->copy_stream));
            CK(m, cudaEventRecord(m->ev_chunk[c], m->copy_stream));
        }
    }
    const cudaStream_t main_stream = m->cfg.stream;
    int rc = NDT2D_OK;
    for (int c = 0; c < pl.nchunks && rc == NDT2D_OK; ++c) {
        int s0 = c * pl.per, s1 = s0 + pl.per < nscans ? s0 + pl.per : nscans;
        if (s1 <= s0) break;
        cudaStream_t ws = m->work_stream[c & 1];
        CK(m, cudaStreamWaitEvent(ws, m->ev_chunk[c], 0));
        m->cfg.stream = ws; // launches below go to the work stream
        rc = launch_chunk(s0, s1, m->b_counter.as<unsigned int>() + 1 + c);
        m->cfg.stream = main_stream;
        if (rc) break;
        cudaError_t e = cudaMemcpyAsync(res + s0, m->b_res.as<ndt2d_result>() + s0, (size_t)(s1 - s0) * sizeof(ndt2d_result),
                                        cudaMemcpyDeviceToHost, ws);
        if (e != cudaSuccess) rc = fail(m, NDT2D_ECUDA, "result copy: %s", cudaGetErrorString(e));
    }
    for (int i = 0; i < 2; ++i) {
        cudaEventRecord(m->ev_done[i], m->work_stream[i]);
        cudaStreamWaitEvent(main_stream, m->ev_done[i], 0);
    }
    int rs = ndt2d_synchronize(m);
    return rc ? rc : rs;
}

} // namespace ndt2d

extern "C" {

int ndt2d_version(void) { return NDT2D_VERSION; }

void ndt2d_default_params(ndt2d_params *p)
{
    if (!p) return;
    p->eig_ratio = 0.01; p->eps_trans = 1e-4; p->eps_rot = 1e-5;
    p->max_step_trans = 0.5; p->max_step_rot = 0.2;
    p->lambda_init = 1e-3; p->lambda_min = 1e-9; p->lambda_max = 1e7;
    p->lambda_up = 10.0; p->lambda_down = 5.0; p->lambda_fail_up = 3.0;
    p->min_points = 3; p->max_iterations = 30; p->overlap = 0; p->reserved = 0;
}

int ndt2d_create_on_stream(int device, void *cuda_stream, ndt2d_matcher **out)
{
    if (!out) return fail(nullptr, NDT2D_EINVAL, "out is NULL");
    *out = nullptr;
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0)
        return fail(nullptr, NDT2D_ECUDA, "no CUDA device available (%s); this library has no CPU fallback",
                    e != cudaSuccess ? cudaGetErrorString(e) : "device count is 0");
    if (device < 0 || device >= ndev) return fail(nullptr, NDT2D_EINVAL, "device %d out of range [0, %d)", device, ndev);
    DeviceGuard g(device);
    cudaDeviceProp prop;
    e = cudaGetDeviceProperties(&prop, device);
    if (e != cudaSuccess) return fail(nullptr, NDT2D_ECUDA, "cudaGetDeviceProperties: %s", cudaGetErrorString(e));
    if (prop.major < 10)
        return fail(nullptr, NDT2D_ECUDA, "device %d is sm_%d%d; libndt2d is built for sm_100a (B200) only", device, prop.major,
                    prop.minor);
    ndt2d_matcher *m = new ndt2d_matcher();
    m->device = device;
    m->cfg.sm_count = prop.multiProcessorCount;
    m->cfg.max_smem_optin = (int)prop.sharedMemPerBlockOptin;
    if (cuda_stream == (void *)-1) {
        e = cudaStreamCreateWithFlags(&m->cfg.stream, cudaStreamNonBlocking);
        if (e != cudaSuccess) {
            delete m;
            return fail(nullptr, NDT2D_ECUDA, "cudaStreamCreate: %s", cudaGetErrorString(e));
        }
        m->own_stream = true;
    } else {
        m->cfg.stream = (cudaStream_t)cuda_stream;
    }
    ndt2d_default_params(&m->prm);
    {
        bool ok = cudaStreamCreateWithFlags(&m->copy_stream, cudaStreamNonBlocking) == cudaSuccess;
        ok = ok && cudaEventCreateWithFlags(&m->ev_begin, cudaEventDisableTiming) == cudaSuccess;
        for (int i = 0; i < 2 && ok; ++i) {
            ok = cudaStreamCreateWithFlags(&m->work_stream[i], cudaStreamNonBlocking) == cudaSuccess;
            ok = ok && cudaEventCreateWithFlags(&m->ev_done[i], cudaEventDisableTiming) == cudaSuccess;
        }
        for (int i = 0; i < ndt2d_matcher::MAX_CHUNKS && ok; ++i)
            ok = cudaEventCreateWithFlags(&m->ev_chunk[i], cudaEventDisableTiming) == cudaSuccess;
        if (!ok) {
            ndt2d_destroy(m);
            return fail(nullptr, NDT2D_ECUDA, "stream/event creation failed: %s", cudaGetErrorString(cudaGetLastError()));
        }
        m->cfg.block_align_max = -1;
        if (const char *e = getenv("NDT2D_BLOCK_ALIGN_MAX")) m->cfg.block_align_max = atoi(e); // 0: always one warp per scan
        m->cfg.align_help = -1;
        if (const char *e = getenv("NDT2D_ALIGN_HELP")) m->cfg.align_help = atoi(e);             // 0: never, 1: always
    }
    if (m->b_counter.ensure(4 * (ndt2d_matcher::MAX_CHUNKS + 1)) != cudaSuccess || m->b_box.ensure(16) != cudaSuccess ||
        m->b_scratch.ensure(sizeof(unsigned long long) * (size_t)topk_scratch_words(m->cfg.sm_count)) != cudaSuccess) {
        ndt2d_destroy(m);
        return fail(nullptr, NDT2D_ENOMEM, "device allocation failed");
    }
    *out = m;
    return NDT2D_OK;
}

int ndt2d_create(int device, ndt2d_matcher **out) { return ndt2d_create_on_stream(device, (void *)-1, out); }

void ndt2d_destroy(ndt2d_matcher *m)
{
    if (!m) return;
    DeviceGuard g(m->device);
    cudaStreamSynchronize(m->cfg.stream);
    drop_target(m);
    ndt2d_exchange_close(m);
    ndt2d_reloc_close(m);
    if (m->fast_host) cudaFreeHost(m->fast_host);
    if (m->fast_res) cudaFreeHost(m->fast_res);
    m->b_fast.release();
    m->b_ring.release();
    DevBuf *bufs[] = {&m->b_xy, &m->b_off, &m->b_init, &m->b_res, &m->b_pose, &m->b_out, &m->b_cnt, &m->b_idx, &m->b_terms,
                      &m->b_hyp, &m->b_scores, &m->b_tki, &m->b_tkv, &m->b_scratch, &m->b_counter, &m->b_beams, &m->b_ranges,
                      &m->b_box, &m->b_ptab, &m->b_pcnt, &m->b_psums, &m->b_pgeo, &m->b_ptargets, &m->b_ppairs, &m->b_perr, &m->b_reloc,
                      &m->b_scand, &m->b_sjobs, &m->b_sinit, &m->b_slevels, &m->b_tpose, &m->b_sm_off, &m->b_sm_start,
                      &m->b_sm_base, &m->b_sm_pose, &m->b_sm_tab};
    for (DevBuf *b : bufs) b->release();
    release_relay(m);
    if (m->copy_stream) {
        cudaStreamSynchronize(m->copy_stream);
        cudaStreamDestroy(m->copy_stream);
    }
    if (m->ev_begin) cudaEventDestroy(m->ev_begin);
    for (int i = 0; i < 2; ++i) {
        if (m->work_stream[i]) {
            cudaStreamSynchronize(m->work_stream[i]);
            cudaStreamDestroy(m->work_stream[i]);
        }
        if (m->ev_done[i]) cudaEventDestroy(m->ev_done[i]);
    }
    for (cudaEvent_t e : m->ev_chunk)
        if (e) cudaEventDestroy(e);
    if (m->own_stream) cudaStreamDestroy(m->cfg.stream);
    delete m;
}

const char *ndt2d_last_error(const ndt2d_matcher *m) { return m ? m->err.c_str() : g_create_error.c_str(); }
void *ndt2d_stream(const ndt2d_matcher *m) { return m ? (void *)m->cfg.stream : nullptr; }
int64_t ndt2d_kernel_launches(const ndt2d_matcher *m) { return m ? m->launches : 0; }

int ndt2d_synchronize(ndt2d_matcher *m)
{
    if (!m) return NDT2D_EINVAL;
    DeviceGuard g(m->device);
    CK(m, cudaStreamSynchronize(m->cfg.stream));
    return NDT2D_OK;
}

int ndt2d_set_params(ndt2d_matcher *m, const ndt2d_params *p)
{
    if (!m || !p) return NDT2D_EINVAL;
    if (p->min_points < 2 || p->max_iterations < 1 || (p->overlap != 0 && p->overlap != 1))
        return fail(m, NDT2D_EINVAL, "bad params: min_points >= 2, max_iterations >= 1, overlap in {0,1}");
    if (!(p->lambda_up > 1.0) || !(p->lambda_fail_up > 1.0) || !(p->lambda_down >= 1.0))
        return fail(m, NDT2D_EINVAL, "bad params: lambda_up > 1, lambda_fail_up > 1, lambda_down >= 1");
    DeviceGuard g(m->device);
    if (m->has_target && p->overlap != m->prm.overlap) {
        cudaStreamSynchronize(m->cfg.stream);
        drop_target(m);
    }
    m->prm = *p;
    return NDT2D_OK;
}

int ndt2d_get_params(const ndt2d_matcher *m, ndt2d_params *p)
{
    if (!m || !p) return NDT2D_EINVAL;
    *p = m->prm;
    return NDT2D_OK;
}

int ndt2d_set_resolutions(ndt2d_matcher *m, const float *res, int nlevels)
{
    if (!m || !res) return NDT2D_EINVAL;
    if (nlevels < 1 || nlevels > NDT2D_MAX_LEVELS) return fail(m, NDT2D_EINVAL, "nlevels %d not in [1, %d]", nlevels, NDT2D_MAX_LEVELS);
    for (int l = 0; l < nlevels; ++l)
        if (!(res[l] > 0.0f) || res[l] > 8.0f) return fail(m, NDT2D_EINVAL, "resolution %g not in (0, 8] m", (double)res[l]);
    DeviceGuard g(m->device);
    cudaStreamSynchronize(m->cfg.stream);
    drop_target(m);
    m->nlevels = nlevels;
    for (int l = 0; l < nlevels; ++l) m->res[l] = res[l];
    return NDT2D_OK;
}

int ndt2d_set_resolution(ndt2d_matcher *m, float res) { return ndt2d_set_resolutions(m, &res, 1); }

int ndt2d_set_grid(ndt2d_matcher *m, float ox, float oy, float ex, float ey)
{
    if (!m) return NDT2D_EINVAL;
    DeviceGuard g(m->device);
    cudaStreamSynchronize(m->cfg.stream);
    drop_target(m);
    m->explicit_grid = (ex > 0.0f && ey > 0.0f);
    m->gox = ox; m->goy = oy; m->gex = ex; m->gey = ey;
    return NDT2D_OK;
}

static TargetSrc point_src(const float *d_xy, int64_t n)
{
    TargetSrc s{};
    s.xy = reinterpret_cast<const float2 *>(d_xy);
    s.n = n;
    return s;
}

// Posed sources (SPEC 7.2): their per-scan {cos, sin, p0, p1} table, made from the f64 poses on the device
static int pose_table(ndt2d_matcher *m, TargetSrc &src, const double *d_poses)
{
    CK(m, m->b_tpose.ensure((size_t)(src.nscans > 0 ? src.nscans : 1) * 32));
    CK(m, launch_pose_table(m->cfg, d_poses, src.nscans, m->b_tpose.as<double>(), &m->launches));
    src.pose = m->b_tpose.as<double>();
    return NDT2D_OK;
}

// Build (replace) the target from `src`, after the caller's argument checks. d_poses: the scans' poses on the device (posed
// sources), nullptr for map-frame points. host_bbox: the caller already knows the bounding box of the finite points
// (ndt2d_set_target computes it on the host for small targets while the points are still in its hands: no bbox kernel,
// no read-back, no synchronisation)
static int set_target_impl(ndt2d_matcher *m, TargetSrc src, const double *d_poses, const float *host_bbox)
{
    DeviceGuard g(m->device);
    CK(m, cudaStreamSynchronize(m->cfg.stream));
    drop_target(m, /*keep_memory=*/true);
    if (d_poses) {
        int rc = pose_table(m, src, d_poses);
        if (rc) return rc;
    }
    float bbox[4] = {0, 0, 0, 0};
    if (host_bbox) {
        for (int i = 0; i < 4; ++i) bbox[i] = host_bbox[i];
    } else if (!m->explicit_grid) {
        int box[4];
        CK(m, launch_bbox(m->cfg, src, m->b_box.as<int>(), &m->launches));
        CK(m, cudaMemcpyAsync(box, m->b_box.p, sizeof(box), cudaMemcpyDeviceToHost, m->cfg.stream));
        CK(m, cudaStreamSynchronize(m->cfg.stream));
        for (int i = 0; i < 4; ++i) bbox[i] = bbox_decode(box[i]);
    }
    int rc = setup_levels(m, bbox);
    if (!rc) rc = accumulate_and_finalize(m, src);
    if (rc) return rc;
    m->has_target = true;
    m->sums_valid = true;
    return NDT2D_OK;
}

// Extend the target with `src` (SPEC 7), after the caller's argument checks; without a target, set_target_impl
static int add_target_impl(ndt2d_matcher *m, TargetSrc src, const double *d_poses)
{
    if (!m->has_target) return set_target_impl(m, src, d_poses, nullptr);
    if (!m->sums_valid) return fail(m, NDT2D_EINVAL, "target was loaded with ndt2d_set_cells; it has no sums to extend");
    DeviceGuard g(m->device);
    if (d_poses) {
        int rc = pose_table(m, src, d_poses);
        if (rc) return rc;
    }
    // small additions (a scan into a large map) finalise only the cells they touch; large ones take the dense pass
    const int64_t n = src.n;
    const int K = m->prm.overlap ? 4 : 1;
    bool sparse = n > 0;
    for (int l = 0; l < m->nlevels; ++l) sparse = sparse && n * K * 8 < (int64_t)m->lv[l].njx * m->lv[l].njy;
    return accumulate_and_finalize(m, src, sparse);
}

int ndt2d_set_target_device(ndt2d_matcher *m, const float *d_xy, int64_t n)
{
    if (!m || n < 0 || (n > 0 && !d_xy)) return m ? fail(m, NDT2D_EINVAL, "bad target arguments") : NDT2D_EINVAL;
    return set_target_impl(m, point_src(d_xy, n), nullptr, nullptr);
}

int ndt2d_add_target_device(ndt2d_matcher *m, const float *d_xy, int64_t n)
{
    if (!m || n < 0 || (n > 0 && !d_xy)) return m ? fail(m, NDT2D_EINVAL, "bad target arguments") : NDT2D_EINVAL;
    return add_target_impl(m, point_src(d_xy, n), nullptr);
}

int ndt2d_set_target(ndt2d_matcher *m, const float *xy, int64_t n)
{
    if (!m || n < 0 || (n > 0 && !xy)) return m ? fail(m, NDT2D_EINVAL, "bad target arguments") : NDT2D_EINVAL;
    DeviceGuard g(m->device);
    int rc = upload(m, m->b_xy, xy, (size_t)n * 8);
    if (rc) return rc;
    // a target scan: the auto-fit bounding box (SPEC 2: min and max over the finite points - exact, order independent) is
    // cheaper to take here than with a kernel, a copy back and a synchronisation; a map cloud goes to the GPU
    float bbox[4] = {INFINITY, INFINITY, -INFINITY, -INFINITY};
    const bool on_host = !m->explicit_grid && n <= 16384;
    if (on_host) {
        for (int64_t i = 0; i < n; ++i) {
            const float x = xy[2 * i], y = xy[2 * i + 1];
            if (!std::isfinite(x) || !std::isfinite(y)) continue;
            bbox[0] = fminf(bbox[0], x); bbox[2] = fmaxf(bbox[2], x);
            bbox[1] = fminf(bbox[1], y); bbox[3] = fmaxf(bbox[3], y);
        }
    }
    rc = set_target_impl(m, point_src(m->b_xy.as<float>(), n), nullptr, on_host ? bbox : nullptr);
    if (rc) return rc;
    return ndt2d_synchronize(m);
}

int ndt2d_add_target(ndt2d_matcher *m, const float *xy, int64_t n)
{
    if (!m || n < 0 || (n > 0 && !xy)) return m ? fail(m, NDT2D_EINVAL, "bad target arguments") : NDT2D_EINVAL;
    DeviceGuard g(m->device);
    int rc = upload(m, m->b_xy, xy, (size_t)n * 8);
    if (rc) return rc;
    rc = ndt2d_add_target_device(m, m->b_xy.as<float>(), n);
    if (rc) return rc;
    return ndt2d_synchronize(m);
}

// ---- targets from posed scans (SPEC 7.2): one implementation for packed points and LaserScan ranges, host and device
// buffers, set and add. The checks come first, so a refused call leaves the target as it was.

// packed scans: d_offsets[0..nscans] index d_xy[0..npoints); host: the arrays are host memory (checked, then uploaded)
static int scans_target(ndt2d_matcher *m, bool add, const float *xy, const int64_t *offsets, int nscans, int64_t npoints,
                        const double *poses, bool host)
{
    if (!m) return NDT2D_EINVAL;
    if (nscans < 0 || (nscans > 0 && (!offsets || !poses))) return fail(m, NDT2D_EINVAL, "bad arguments");
    if (host) {
        if (nscans > 0 && offsets[0] != 0) return fail(m, NDT2D_EINVAL, "offsets[0] = %lld, not 0", (long long)offsets[0]);
        for (int b = 0; b < nscans; ++b)
            if (offsets[b + 1] < offsets[b]) return fail(m, NDT2D_EINVAL, "offsets not monotone at scan %d", b);
        npoints = nscans > 0 ? offsets[nscans] : 0;
        for (int64_t i = 0; i < 3 * (int64_t)nscans; ++i)
            if (!std::isfinite(poses[i])) return fail(m, NDT2D_EINVAL, "pose of scan %lld is not finite", (long long)(i / 3));
    }
    if (npoints < 0 || (npoints > 0 && (!xy || nscans == 0))) return fail(m, NDT2D_EINVAL, "bad arguments");
    DeviceGuard g(m->device);
    if (host) {
        int rc = upload(m, m->b_xy, xy, (size_t)npoints * 8);
        if (!rc) rc = upload(m, m->b_off, offsets, nscans > 0 ? (size_t)(nscans + 1) * 8 : 0);
        if (!rc) rc = upload(m, m->b_pose, poses, (size_t)nscans * 24);
        if (rc) return rc;
        xy = m->b_xy.as<float>();
        offsets = m->b_off.as<int64_t>();
        poses = m->b_pose.as<double>();
    }
    TargetSrc src{};
    src.xy = reinterpret_cast<const float2 *>(xy);
    src.n = npoints;
    src.offsets = offsets;
    src.nscans = nscans;
    int rc = add ? add_target_impl(m, src, poses) : set_target_impl(m, src, poses, nullptr);
    if (rc || !host) return rc;
    return ndt2d_synchronize(m);
}

// LaserScan scans (SPEC 8): nscans rows of nbeams ranges
static int ranges_target(ndt2d_matcher *m, bool add, const void *ranges, int ranges_are_u16, int nscans, int nbeams, double angle_min,
                         double angle_inc, float range_scale, float range_min, float range_max, const double *poses, bool host)
{
    if (!m) return NDT2D_EINVAL;
    if (nscans < 0 || nbeams < 1 || (nscans > 0 && (!ranges || !poses))) return fail(m, NDT2D_EINVAL, "bad arguments");
    if (host)
        for (int64_t i = 0; i < 3 * (int64_t)nscans; ++i)
            if (!std::isfinite(poses[i])) return fail(m, NDT2D_EINVAL, "pose of scan %lld is not finite", (long long)(i / 3));
    DeviceGuard g(m->device);
    int rc = ensure_beams(m, nbeams, angle_min, angle_inc);
    if (rc) return rc;
    const size_t bytes = (size_t)nscans * nbeams * (ranges_are_u16 ? 2 : 4);
    if (host) {
        rc = upload(m, m->b_ranges, ranges, bytes);
        if (!rc) rc = upload(m, m->b_pose, poses, (size_t)nscans * 24);
        if (rc) return rc;
        ranges = m->b_ranges.p;
        poses = m->b_pose.as<double>();
    }
    TargetSrc src{};
    src.n = (int64_t)nscans * nbeams;
    src.nscans = nscans;
    src.ranges = ranges;
    src.beams = m->b_beams.as<float2>();
    src.ranges_u16 = ranges_are_u16 ? 1 : 0;
    src.nbeams = nbeams;
    src.range_scale = range_scale; src.range_min = range_min; src.range_max = range_max;
    rc = add ? add_target_impl(m, src, poses) : set_target_impl(m, src, poses, nullptr);
    if (rc || !host) return rc;
    return ndt2d_synchronize(m);
}

int ndt2d_set_target_scans(ndt2d_matcher *m, const float *xy, const int64_t *offsets, int nscans, const double *poses)
{
    return scans_target(m, false, xy, offsets, nscans, 0, poses, true);
}

int ndt2d_add_target_scans(ndt2d_matcher *m, const float *xy, const int64_t *offsets, int nscans, const double *poses)
{
    return scans_target(m, true, xy, offsets, nscans, 0, poses, true);
}

int ndt2d_set_target_scans_device(ndt2d_matcher *m, const float *d_xy, const int64_t *d_offsets, int nscans, int64_t npoints,
                                  const double *d_poses)
{
    return scans_target(m, false, d_xy, d_offsets, nscans, npoints, d_poses, false);
}

int ndt2d_add_target_scans_device(ndt2d_matcher *m, const float *d_xy, const int64_t *d_offsets, int nscans, int64_t npoints,
                                  const double *d_poses)
{
    return scans_target(m, true, d_xy, d_offsets, nscans, npoints, d_poses, false);
}

int ndt2d_set_target_ranges(ndt2d_matcher *m, const void *ranges, int ranges_are_u16, int nscans, int nbeams, double angle_min,
                            double angle_inc, float range_scale, float range_min, float range_max, const double *poses)
{
    return ranges_target(m, false, ranges, ranges_are_u16, nscans, nbeams, angle_min, angle_inc, range_scale, range_min, range_max,
                         poses, true);
}

int ndt2d_add_target_ranges(ndt2d_matcher *m, const void *ranges, int ranges_are_u16, int nscans, int nbeams, double angle_min,
                            double angle_inc, float range_scale, float range_min, float range_max, const double *poses)
{
    return ranges_target(m, true, ranges, ranges_are_u16, nscans, nbeams, angle_min, angle_inc, range_scale, range_min, range_max,
                         poses, true);
}

int ndt2d_set_target_ranges_device(ndt2d_matcher *m, const void *d_ranges, int ranges_are_u16, int nscans, int nbeams,
                                   double angle_min, double angle_inc, float range_scale, float range_min, float range_max,
                                   const double *d_poses)
{
    return ranges_target(m, false, d_ranges, ranges_are_u16, nscans, nbeams, angle_min, angle_inc, range_scale, range_min,
                         range_max, d_poses, false);
}

int ndt2d_add_target_ranges_device(ndt2d_matcher *m, const void *d_ranges, int ranges_are_u16, int nscans, int nbeams,
                                   double angle_min, double angle_inc, float range_scale, float range_min, float range_max,
                                   const double *d_poses)
{
    return ranges_target(m, true, d_ranges, ranges_are_u16, nscans, nbeams, angle_min, angle_inc, range_scale, range_min,
                         range_max, d_poses, false);
}

int ndt2d_level_geometry(const ndt2d_matcher *m, int level, float geom[5], int32_t dims[4])
{
    if (!m || !m->has_target || level < 0 || level >= m->nlevels) return NDT2D_EINVAL;
    const LevelDev &L = m->lv[level];
    geom[0] = L.res; geom[1] = L.st; geom[2] = L.inv_st; geom[3] = L.ox; geom[4] = L.oy;
    dims[0] = L.nhx; dims[1] = L.nhy; dims[2] = L.njx; dims[3] = L.njy;
    return NDT2D_OK;
}

int ndt2d_get_cells(ndt2d_matcher *m, int level, float *cells)
{
    int rc = check_level(m, level);
    if (rc) return rc;
    DeviceGuard g(m->device);
    const LevelDev &L = m->lv[level];
    CK(m, cudaMemcpyAsync(cells, L.cells, (size_t)L.njx * L.njy * 32, cudaMemcpyDeviceToHost, m->cfg.stream));
    return ndt2d_synchronize(m);
}

int ndt2d_get_sums(ndt2d_matcher *m, int level, uint32_t *n, int64_t *sums)
{
    int rc = check_level(m, level);
    if (rc) return rc;
    if (!m->sums_valid) return fail(m, NDT2D_EINVAL, "target was loaded with ndt2d_set_cells; no sums");
    DeviceGuard g(m->device);
    const LevelDev &L = m->lv[level];
    size_t nc = (size_t)L.njx * L.njy;
    CK(m, cudaMemcpyAsync(n, L.cnt, nc * 4, cudaMemcpyDeviceToHost, m->cfg.stream));
    CK(m, cudaMemcpyAsync(sums, L.sums, nc * 40, cudaMemcpyDeviceToHost, m->cfg.stream));
    return ndt2d_synchronize(m);
}

const float *ndt2d_cells_device(const ndt2d_matcher *m, int level)
{
    if (!m || !m->has_target || level < 0 || level >= m->nlevels) return nullptr;
    return reinterpret_cast<const float *>(m->lv[level].cells);
}

int ndt2d_set_cells(ndt2d_matcher *m, int level, const float *cells, int64_t nrecords)
{
    if (!m || !cells) return NDT2D_EINVAL;
    DeviceGuard g(m->device);
    if (!m->has_target) {
        if (!m->explicit_grid) return fail(m, NDT2D_EINVAL, "ndt2d_set_cells needs ndt2d_set_grid first");
        const float bbox[4] = {0, 0, 0, 0};
        int rc = setup_levels(m, bbox);
        if (rc) return rc;
        m->has_target = true;
    }
    if (level < 0 || level >= m->nlevels) return fail(m, NDT2D_EINVAL, "level %d out of range", level);
    const LevelDev &L = m->lv[level];
    if (nrecords != (int64_t)L.njx * L.njy)
        return fail(m, NDT2D_EINVAL, "set_cells: level %d holds %d x %d = %lld records, caller passed %lld", level, L.njx, L.njy,
                    (long long)((int64_t)L.njx * L.njy), (long long)nrecords);
    m->sums_valid = false;
    CK(m, cudaMemcpyAsync(m->mem[level].cells, cells, (size_t)L.njx * L.njy * 32, cudaMemcpyHostToDevice, m->cfg.stream));
    return ndt2d_synchronize(m);
}

// ---- map files (SURVEY 8(f) rank 4). Layout: MapFileHeader, nlevels x MapFileLevel, then per level the cell records
// (njx*njy*32 B) and, when has_sums, the counts (u32) and the five i64 sums of every cell. Little endian, no padding games:
// both structs are made of 4- and 8-byte fields in natural alignment.
namespace {
struct MapFileHeader {
    char magic[8];          // "NDT2DMAP"
    uint32_t version;       // file layout, 1
    uint32_t spec_version;  // SPEC.md version of the records (4): records of another version are not interchangeable
    int32_t nlevels, overlap, min_points, explicit_grid;
    double eig_ratio;
    float gox, goy, gex, gey;
    uint32_t has_sums, reserved;
};
struct MapFileLevel {
    float res, ox, oy, reserved;
    int32_t nhx, nhy, njx, njy;
};
constexpr uint32_t kMapFileVersion = 1, kSpecVersion = 4;
} // namespace

int ndt2d_save_map(ndt2d_matcher *m, const char *path, int with_sums)
{
    if (!m || !path) return NDT2D_EINVAL;
    if (!m->has_target) return fail(m, NDT2D_ENOTARGET, "no target set");
    if (with_sums && !m->sums_valid) return fail(m, NDT2D_EINVAL, "save_map: the target has no sums (it was loaded without them)");
    DeviceGuard g(m->device);
    FILE *f = fopen(path, "wb");
    if (!f) return fail(m, NDT2D_EINVAL, "save_map: cannot open %s for writing", path);
    MapFileHeader h;
    memset(&h, 0, sizeof(h));
    memcpy(h.magic, "NDT2DMAP", 8);
    h.version = kMapFileVersion; h.spec_version = kSpecVersion;
    h.nlevels = m->nlevels; h.overlap = m->prm.overlap; h.min_points = m->prm.min_points; h.explicit_grid = m->explicit_grid ? 1 : 0;
    h.eig_ratio = m->prm.eig_ratio;
    h.gox = m->gox; h.goy = m->goy; h.gex = m->gex; h.gey = m->gey;
    h.has_sums = with_sums ? 1u : 0u;
    bool ok = fwrite(&h, sizeof(h), 1, f) == 1;
    for (int l = 0; l < m->nlevels && ok; ++l) {
        const LevelDev &L = m->lv[l];
        MapFileLevel v = {L.res, L.ox, L.oy, 0.0f, L.nhx, L.nhy, L.njx, L.njy};
        ok = fwrite(&v, sizeof(v), 1, f) == 1;
    }
    std::vector<unsigned char> buf;
    for (int l = 0; l < m->nlevels && ok; ++l) {
        const LevelDev &L = m->lv[l];
        const size_t nc = (size_t)L.njx * L.njy;
        const void *src[3] = {L.cells, L.cnt, L.sums};
        const size_t bytes[3] = {nc * 32, nc * 4, nc * 40};
        for (int part = 0; part < (with_sums ? 3 : 1) && ok; ++part) {
            buf.resize(bytes[part]);
            cudaError_t e = cudaMemcpyAsync(buf.data(), src[part], bytes[part], cudaMemcpyDeviceToHost, m->cfg.stream);
            if (e == cudaSuccess) e = cudaStreamSynchronize(m->cfg.stream);
            if (e != cudaSuccess) {
                fclose(f);
                return fail(m, NDT2D_ECUDA, "save_map: %s", cudaGetErrorString(e));
            }
            ok = fwrite(buf.data(), 1, bytes[part], f) == bytes[part];
        }
    }
    ok = (fclose(f) == 0) && ok;
    return ok ? NDT2D_OK : fail(m, NDT2D_EINVAL, "save_map: short write to %s", path);
}

int ndt2d_load_map(ndt2d_matcher *m, const char *path)
{
    if (!m || !path) return NDT2D_EINVAL;
    DeviceGuard g(m->device);
    FILE *f = fopen(path, "rb");
    if (!f) return fail(m, NDT2D_EINVAL, "load_map: cannot open %s", path);
    MapFileHeader h;
    MapFileLevel lv[NDT2D_MAX_LEVELS];
    bool ok = fread(&h, sizeof(h), 1, f) == 1 && memcmp(h.magic, "NDT2DMAP", 8) == 0;
    if (!ok || h.version != kMapFileVersion || h.spec_version != kSpecVersion || h.nlevels < 1 || h.nlevels > NDT2D_MAX_LEVELS ||
        (h.overlap != 0 && h.overlap != 1) || h.min_points < 2) {
        fclose(f);
        return fail(m, NDT2D_EINVAL, "load_map: %s is not an NDT2DMAP file of layout %u / SPEC v%u", path, kMapFileVersion, kSpecVersion);
    }
    ok = fread(lv, sizeof(MapFileLevel), (size_t)h.nlevels, f) == (size_t)h.nlevels;
    for (int l = 0; l < h.nlevels && ok; ++l)
        ok = lv[l].res > 0.0f && lv[l].res <= 8.0f && lv[l].nhx >= 1 && lv[l].nhy >= 1 && lv[l].njx == lv[l].nhx + h.overlap &&
             lv[l].njy == lv[l].nhy + h.overlap && (int64_t)lv[l].njx * lv[l].njy < ((int64_t)1 << 31);
    if (!ok) {
        fclose(f);
        return fail(m, NDT2D_EINVAL, "load_map: %s: bad level table", path);
    }
    cudaStreamSynchronize(m->cfg.stream);
    drop_target(m, /*keep_memory=*/true);
    m->prm.overlap = h.overlap; m->prm.min_points = h.min_points; m->prm.eig_ratio = h.eig_ratio;
    m->nlevels = h.nlevels;
    m->explicit_grid = h.explicit_grid != 0;
    m->gox = h.gox; m->goy = h.goy; m->gex = h.gex; m->gey = h.gey;
    std::vector<unsigned char> buf;
    int rc = NDT2D_OK;
    for (int l = 0; l < h.nlevels && rc == NDT2D_OK; ++l) {
        m->res[l] = lv[l].res;
        LevelDev &L = m->lv[l];
        L = LevelDev{};
        level_strides(L, lv[l].res, h.overlap);
        L.ox = lv[l].ox; L.oy = lv[l].oy;   // the saved lattice, exactly (auto-fitted or explicit)
        L.nhx = lv[l].nhx; L.nhy = lv[l].nhy; L.njx = lv[l].njx; L.njy = lv[l].njy;
        rc = install_level(m, l);
        if (rc) break;
        const size_t nc = (size_t)L.njx * L.njy;
        void *dst[3] = {m->mem[l].cells, m->mem[l].cnt, m->mem[l].sums};
        const size_t bytes[3] = {nc * 32, nc * 4, nc * 40};
        for (int part = 0; part < (h.has_sums ? 3 : 1) && rc == NDT2D_OK; ++part) {
            buf.resize(bytes[part]);
            if (fread(buf.data(), 1, bytes[part], f) != bytes[part]) {
                rc = fail(m, NDT2D_EINVAL, "load_map: %s is truncated (level %d)", path, l);
                break;
            }
            cudaError_t e = cudaMemcpyAsync(dst[part], buf.data(), bytes[part], cudaMemcpyHostToDevice, m->cfg.stream);
            if (e == cudaSuccess) e = cudaStreamSynchronize(m->cfg.stream);
            if (e != cudaSuccess) rc = fail(m, NDT2D_ECUDA, "load_map: %s", cudaGetErrorString(e));
        }
    }
    fclose(f);
    if (rc) {
        drop_target(m);
        return rc;
    }
    m->has_target = true;
    m->sums_valid = h.has_sums != 0;
    return NDT2D_OK;
}

int ndt2d_cell_index(ndt2d_matcher *m, int level, const float *xy, int n, const double *pose, int32_t *idx)
{
    int rc = check_level(m, level);
    if (rc) return rc;
    if (n < 0 || (n > 0 && (!xy || !idx))) return fail(m, NDT2D_EINVAL, "bad arguments");
    if (n == 0) return NDT2D_OK;
    DeviceGuard g(m->device);
    if ((rc = upload(m, m->b_xy, xy, (size_t)n * 8))) return rc;
    if (pose && (rc = upload(m, m->b_pose, pose, 24))) return rc;
    CK(m, m->b_idx.ensure((size_t)n * 4));
    CK(m, launch_cell_index(m->cfg, m->lv[level], m->b_xy.as<float2>(), n, pose ? m->b_pose.as<double>() : nullptr,
                            m->b_idx.as<int32_t>(), &m->launches));
    CK(m, cudaMemcpyAsync(idx, m->b_idx.p, (size_t)n * 4, cudaMemcpyDeviceToHost, m->cfg.stream));
    return ndt2d_synchronize(m);
}

int ndt2d_evaluate_device(ndt2d_matcher *m, int level, const float *d_xy, int n, const double *d_poses, int npose,
                          double *d_out, int32_t *d_count)
{
    int rc = check_level(m, level);
    if (rc) return rc;
    if (n < 0 || npose < 0 || !d_out || (npose > 0 && !d_poses)) return fail(m, NDT2D_EINVAL, "bad arguments");
    DeviceGuard g(m->device);
    CK(m, launch_eval_poses(m->cfg, m->lv[level], reinterpret_cast<const float2 *>(d_xy), n, d_poses, 0, npose, 1, d_out, 10,
                            d_count, &m->launches));
    return NDT2D_OK;
}

int ndt2d_evaluate(ndt2d_matcher *m, int level, const float *xy, int n, const double *poses, int npose, double *out,
                   int32_t *count)
{
    int rc = check_level(m, level);
    if (rc) return rc;
    if (n < 0 || npose < 0 || !out || (npose > 0 && !poses) || (n > 0 && !xy)) return fail(m, NDT2D_EINVAL, "bad arguments");
    if (npose == 0) return NDT2D_OK;
    DeviceGuard g(m->device);
    if ((rc = upload(m, m->b_xy, xy, (size_t)n * 8))) return rc;
    if ((rc = upload(m, m->b_pose, poses, (size_t)npose * 24))) return rc;
    CK(m, m->b_out.ensure((size_t)npose * 80));
    CK(m, m->b_cnt.ensure((size_t)npose * 4));
    rc = ndt2d_evaluate_device(m, level, m->b_xy.as<float>(), n, m->b_pose.as<double>(), npose, m->b_out.as<double>(),
                               m->b_cnt.as<int32_t>());
    if (rc) return rc;
    CK(m, cudaMemcpyAsync(out, m->b_out.p, (size_t)npose * 80, cudaMemcpyDeviceToHost, m->cfg.stream));
    if (count) CK(m, cudaMemcpyAsync(count, m->b_cnt.p, (size_t)npose * 4, cudaMemcpyDeviceToHost, m->cfg.stream));
    return ndt2d_synchronize(m);
}

int ndt2d_point_terms(ndt2d_matcher *m, int level, const float *xy, int n, const double *pose, float *terms)
{
    int rc = check_level(m, level);
    if (rc) return rc;
    if (n < 0 || !pose || (n > 0 && (!xy || !terms))) return fail(m, NDT2D_EINVAL, "bad arguments");
    if (n == 0) return NDT2D_OK;
    DeviceGuard g(m->device);
    const int K = m->prm.overlap ? 4 : 1;
    if ((rc = upload(m, m->b_xy, xy, (size_t)n * 8))) return rc;
    if ((rc = upload(m, m->b_pose, pose, 24))) return rc;
    CK(m, m->b_terms.ensure((size_t)n * K * 40));
    CK(m, launch_point_terms(m->cfg, m->lv[level], m->b_xy.as<float2>(), n, m->b_pose.as<double>(), m->b_terms.as<float>(),
                             &m->launches));
    CK(m, cudaMemcpyAsync(terms, m->b_terms.p, (size_t)n * K * 40, cudaMemcpyDeviceToHost, m->cfg.stream));
    return ndt2d_synchronize(m);
}

int ndt2d_align_batch_device(ndt2d_matcher *m, const float *d_xy, const int64_t *d_offsets, int nscans, int max_points,
                             const double *d_init, ndt2d_result *d_res)
{
    if (!m) return NDT2D_EINVAL;
    if (!m->has_target) return fail(m, NDT2D_ENOTARGET, "no target set");
    if (nscans < 0 || max_points < 0 || (nscans > 0 && (!d_offsets || !d_init || !d_res)))
        return fail(m, NDT2D_EINVAL, "bad arguments");
    if (nscans == 0) return NDT2D_OK;
    DeviceGuard g(m->device);
    AlignArgs a{};
    a.xy = reinterpret_cast<const float2 *>(d_xy);
    a.offsets = d_offsets;
    a.init = d_init;
    a.res = d_res;
    a.nscans = nscans;
    return align_device(m, a, max_points);
}

// Small host-buffer batches (a single align above all): offsets, initial poses and scans are packed into one pinned
// buffer and go up in ONE upload, the kernel writes its results into mapped pinned memory, the queue counter comes from a
// pre-zeroed ring: upload, launch, synchronise - instead of the ~15 calls of the chunked pipeline.
// the buffers of the small-call path (align_small), and a zeroed work-queue counter from the ring
static int fast_prepare(ndt2d_matcher *m)
{
    if (!m->fast_ready) {   // set only after every allocation below has succeeded: a failed attempt is simply repeated
        if (!m->fast_host) CK(m, cudaHostAlloc(reinterpret_cast<void **>(&m->fast_host), ndt2d_matcher::FAST_BYTES, cudaHostAllocMapped));
        CK(m, cudaHostGetDevicePointer(reinterpret_cast<void **>(&m->fast_host_dev), m->fast_host, 0));
        if (!m->fast_res) CK(m, cudaHostAlloc(reinterpret_cast<void **>(&m->fast_res), ndt2d_matcher::FAST_SCANS * sizeof(ndt2d_result), cudaHostAllocMapped));
        CK(m, cudaHostGetDevicePointer(reinterpret_cast<void **>(&m->fast_res_dev), m->fast_res, 0));
        CK(m, m->b_fast.ensure(ndt2d_matcher::FAST_BYTES));
        CK(m, m->b_ring.ensure(ndt2d_matcher::RING * 4));
        CK(m, cudaMemsetAsync(m->b_ring.p, 0, ndt2d_matcher::RING * 4, m->cfg.stream));
        m->ring_pos = 0;
        m->fast_ready = true;
    }
    if (m->ring_pos == ndt2d_matcher::RING) {   // every slot used once: zero the ring again (stream-ordered after its last user)
        CK(m, cudaMemsetAsync(m->b_ring.p, 0, ndt2d_matcher::RING * 4, m->cfg.stream));
        m->ring_pos = 0;
    }
    return NDT2D_OK;
}

// `a`: the call's input in host memory, as align_host takes it; scan_bytes: its scans. Packed layout: offsets (points
// only) | init | scans, every section at a multiple of 8 bytes.
static int align_small(ndt2d_matcher *m, AlignArgs a, size_t scan_bytes, int max_points, const double *init, ndt2d_result *res,
                       double angle_min, double angle_inc)
{
    int rc = fast_prepare(m);
    if (rc) return rc;
    const bool ranges = a.ranges != nullptr;
    const size_t off_bytes = ranges ? 0 : (size_t)(a.nscans + 1) * 8, init_bytes = (size_t)a.nscans * 24;
    unsigned char *h = m->fast_host;
    if (off_bytes) memcpy(h, a.offsets, off_bytes);
    memcpy(h + off_bytes, init, init_bytes);
    if (scan_bytes) memcpy(h + off_bytes + init_bytes, ranges ? a.ranges : static_cast<const void *>(a.xy), scan_bytes);
    // Point scans are staged by the block kernel straight from the mapped staging buffer (8.6 KB over PCIe, every thread
    // with a load in flight): one copy operation fewer per call, 66.7 -> 62.3 us for a 1080-point align. LaserScan ranges
    // are copied first: one warp converts the beams, and from mapped memory its 34 dependent PCIe round trips measured
    // 102 us against 83 us.
    unsigned char *d = ranges ? m->b_fast.as<unsigned char>() : m->fast_host_dev;
    if (ranges) CK(m, cudaMemcpyAsync(d, h, init_bytes + scan_bytes, cudaMemcpyHostToDevice, m->cfg.stream));
    const unsigned char *scans = d + off_bytes + init_bytes;
    if (ranges) {
        a.ranges = scans;
    } else {
        a.offsets = reinterpret_cast<const int64_t *>(d);
        a.xy = reinterpret_cast<const float2 *>(scans);
    }
    a.init = reinterpret_cast<const double *>(d + off_bytes);
    a.res = m->fast_res_dev;
    a.counter = m->b_ring.as<unsigned int>() + m->ring_pos++;
    a.counter_is_zero = 1;
    if ((rc = align_device(m, a, max_points, angle_min, angle_inc))) return rc;
    if ((rc = ndt2d_synchronize(m))) return rc;
    memcpy(res, m->fast_res, (size_t)a.nscans * sizeof(ndt2d_result));
    return NDT2D_OK;
}

// The host-buffer batch of ndt2d_align_batch and ndt2d_align_batch_ranges, after their argument checks. `in` is the call's
// input as the caller passed it, in host memory: in.nscans scans of at most max_points points each, as xy and offsets or as
// ranges with their beam fields. Small calls take align_small, the others the chunked pipeline.
static int align_host(ndt2d_matcher *m, const AlignArgs &in, int max_points, const double *init, ndt2d_result *res,
                      double angle_min = 0.0, double angle_inc = 0.0)
{
    const int nscans = in.nscans;
    const bool ranges = in.ranges != nullptr;
    const unsigned char *src = static_cast<const unsigned char *>(ranges ? in.ranges : static_cast<const void *>(in.xy));
    const size_t row = (size_t)in.nbeams * (in.ranges_u16 ? 2 : 4);
    auto pos = [&](int s) { return ranges ? (size_t)s * row : (size_t)in.offsets[s] * 8; };  // first byte of scan s in src
    const size_t off_bytes = ranges ? 0 : (size_t)(nscans + 1) * 8, init_bytes = (size_t)nscans * 24;
    if (nscans <= ndt2d_matcher::FAST_SCANS && pos(0) == 0 && off_bytes + init_bytes + pos(nscans) <= ndt2d_matcher::FAST_BYTES)
        return align_small(m, in, pos(nscans), max_points, init, res, angle_min, angle_inc);
    DevBuf &buf = ranges ? m->b_ranges : m->b_xy;
    int rc;
    CK(m, buf.ensure(std::max<size_t>(pos(nscans), 8)));
    CK(m, m->b_res.ensure((size_t)nscans * sizeof(ndt2d_result)));
    if (!ranges && (rc = upload(m, m->b_off, in.offsets, off_bytes))) return rc;
    if ((rc = upload(m, m->b_init, init, init_bytes))) return rc;
    if (ranges && (rc = ensure_beams(m, in.nbeams, angle_min, angle_inc))) return rc; // on the main stream, before the work streams fork
    unsigned char *dev = buf.as<unsigned char>();
    return run_pipeline(
        m, nscans, pos(nscans), res,
        [&](int s0, int s1, void **dst, const void **from, size_t *bytes) {
            *dst = dev + pos(s0);
            *from = src + pos(s0);
            *bytes = pos(s1) - pos(s0);
        },
        [&](int s0, int s1, unsigned int *counter) -> int {
            AlignArgs a = in;
            if (ranges) {
                a.ranges = dev + pos(s0);
            } else {            // the points keep their place in the batch: the offsets index them
                a.xy = reinterpret_cast<const float2 *>(dev);
                a.offsets = m->b_off.as<int64_t>() + s0;
            }
            a.init = m->b_init.as<double>() + 3 * (size_t)s0;
            a.res = m->b_res.as<ndt2d_result>() + s0;
            a.nscans = s1 - s0;
            a.counter = counter;
            a.batch_scans = nscans;
            return align_device(m, a, max_points, angle_min, angle_inc);
        });
}

int ndt2d_align_batch(ndt2d_matcher *m, const float *xy, const int64_t *offsets, int nscans, const double *init,
                      ndt2d_result *res)
{
    if (!m) return NDT2D_EINVAL;
    if (!m->has_target) return fail(m, NDT2D_ENOTARGET, "no target set");
    if (nscans < 0 || (nscans > 0 && (!offsets || !init || !res))) return fail(m, NDT2D_EINVAL, "bad arguments");
    if (nscans == 0) return NDT2D_OK;
    int64_t maxn = 0;
    for (int b = 0; b < nscans; ++b) {
        int64_t nb = offsets[b + 1] - offsets[b];
        if (nb < 0 || nb > 0x7fffffff) return fail(m, NDT2D_EINVAL, "offsets not monotone at scan %d", b);
        if (nb > maxn) maxn = nb;
    }
    int64_t total = offsets[nscans];
    if (offsets[0] < 0 || (total > 0 && !xy)) return fail(m, NDT2D_EINVAL, "bad offsets / xy");
    DeviceGuard g(m->device);
    AlignArgs in{};
    in.xy = reinterpret_cast<const float2 *>(xy);
    in.offsets = offsets;
    in.nscans = nscans;
    return align_host(m, in, (int)maxn, init, res);
}

int ndt2d_align(ndt2d_matcher *m, const float *xy, int n, const double init[3], ndt2d_result *res)
{
    if (n < 0) return m ? fail(m, NDT2D_EINVAL, "n < 0") : NDT2D_EINVAL;
    int64_t off[2] = {0, n};
    return ndt2d_align_batch(m, xy, off, 1, init, res);
}

// the LaserScan input of an align (SPEC 8); align_device adds the beam table
static AlignArgs ranges_input(const void *ranges, int ranges_are_u16, int nscans, int nbeams, float range_scale, float range_min,
                              float range_max)
{
    AlignArgs a{};
    a.ranges = ranges;
    a.ranges_u16 = ranges_are_u16 ? 1 : 0;
    a.nbeams = nbeams;
    a.range_scale = range_scale; a.range_min = range_min; a.range_max = range_max;
    a.nscans = nscans;
    return a;
}

int ndt2d_align_batch_ranges_device(ndt2d_matcher *m, const void *d_ranges, int ranges_are_u16, int nscans, int nbeams,
                                    double angle_min, double angle_inc, float range_scale, float range_min, float range_max,
                                    const double *d_init, ndt2d_result *d_res)
{
    if (!m) return NDT2D_EINVAL;
    if (!m->has_target) return fail(m, NDT2D_ENOTARGET, "no target set");
    if (nscans < 0 || nbeams < 1 || (nscans > 0 && (!d_ranges || !d_init || !d_res)))
        return fail(m, NDT2D_EINVAL, "bad arguments");
    if (nscans == 0) return NDT2D_OK;
    DeviceGuard g(m->device);
    AlignArgs a = ranges_input(d_ranges, ranges_are_u16, nscans, nbeams, range_scale, range_min, range_max);
    a.init = d_init;
    a.res = d_res;
    return align_device(m, a, nbeams, angle_min, angle_inc);
}

int ndt2d_align_batch_ranges(ndt2d_matcher *m, const void *ranges, int ranges_are_u16, int nscans, int nbeams,
                             double angle_min, double angle_inc, float range_scale, float range_min, float range_max,
                             const double *init, ndt2d_result *res)
{
    if (!m) return NDT2D_EINVAL;
    if (!m->has_target) return fail(m, NDT2D_ENOTARGET, "no target set");
    if (nscans < 0 || nbeams < 1 || (nscans > 0 && (!ranges || !init || !res))) return fail(m, NDT2D_EINVAL, "bad arguments");
    if (nscans == 0) return NDT2D_OK;
    DeviceGuard g(m->device);
    return align_host(m, ranges_input(ranges, ranges_are_u16, nscans, nbeams, range_scale, range_min, range_max), nbeams, init,
                      res, angle_min, angle_inc);
}

int ndt2d_sweep_device(ndt2d_matcher *m, int level, const float *d_xy, int n, const float *d_hyp, int64_t nhyp,
                       double *d_scores, int k, int64_t *d_best_idx, double *d_best_score)
{
    int rc = check_level(m, level);
    if (rc) return rc;
    if (n < 0 || nhyp < 0 || k < 0 || k > 1024 || (nhyp > 0 && !d_hyp) || (k > 0 && (!d_best_idx || !d_best_score)))
        return fail(m, NDT2D_EINVAL, "bad arguments");
    DeviceGuard g(m->device);
    if (!d_scores) {
        CK(m, m->b_scores.ensure((size_t)(nhyp ? nhyp : 1) * 8));
        d_scores = m->b_scores.as<double>();
    }
    CK(m, launch_eval_poses(m->cfg, m->lv[level], reinterpret_cast<const float2 *>(d_xy), n, d_hyp, 1, nhyp, 0, d_scores, 1,
                            nullptr, &m->launches));
    if (k > 0) CK(m, launch_topk(m->cfg, d_scores, nhyp, k, d_best_idx, d_best_score, m->b_scratch.as<unsigned long long>(), &m->launches));
    return NDT2D_OK;
}

int ndt2d_sweep(ndt2d_matcher *m, int level, const float *xy, int n, const float *hyp, int64_t nhyp, double *scores, int k,
                int64_t *best_idx, double *best_score)
{
    int rc = check_level(m, level);
    if (rc) return rc;
    if (n < 0 || nhyp < 0 || k < 0 || k > 1024 || (n > 0 && !xy) || (nhyp > 0 && !hyp) || (k > 0 && (!best_idx || !best_score)))
        return fail(m, NDT2D_EINVAL, "bad arguments");
    DeviceGuard g(m->device);
    if ((rc = upload(m, m->b_xy, xy, (size_t)n * 8))) return rc;
    if ((rc = upload(m, m->b_hyp, hyp, (size_t)nhyp * 12))) return rc;
    CK(m, m->b_scores.ensure((size_t)(nhyp ? nhyp : 1) * 8));
    CK(m, m->b_tki.ensure((size_t)(k ? k : 1) * 8));
    CK(m, m->b_tkv.ensure((size_t)(k ? k : 1) * 8));
    rc = ndt2d_sweep_device(m, level, m->b_xy.as<float>(), n, m->b_hyp.as<float>(), nhyp, m->b_scores.as<double>(), k,
                            m->b_tki.as<int64_t>(), m->b_tkv.as<double>());
    if (rc) return rc;
    if (scores && nhyp) CK(m, cudaMemcpyAsync(scores, m->b_scores.p, (size_t)nhyp * 8, cudaMemcpyDeviceToHost, m->cfg.stream));
    if (k > 0) {
        CK(m, cudaMemcpyAsync(best_idx, m->b_tki.p, (size_t)k * 8, cudaMemcpyDeviceToHost, m->cfg.stream));
        CK(m, cudaMemcpyAsync(best_score, m->b_tkv.p, (size_t)k * 8, cudaMemcpyDeviceToHost, m->cfg.stream));
    }
    return ndt2d_synchronize(m);
}

// Everything on the device, nothing synchronised: sweep of the level, top-k, then the k candidates become k refinement
// jobs of the SAME scan (AlignArgs::job_scan) - no copy of the scan, no trip to the host in between.
int ndt2d_relocalize_device(ndt2d_matcher *m, int level, const float *d_xy, int n, const float *d_hyp, int64_t nhyp, int k,
                            int64_t *d_best_idx, ndt2d_result *d_res)
{
    int rc = check_level(m, level);
    if (rc) return rc;
    if (k < 1 || k > 1024 || n < 0 || nhyp < 0 || !d_best_idx || !d_res || (nhyp > 0 && !d_hyp))
        return fail(m, NDT2D_EINVAL, "bad arguments");
    DeviceGuard g(m->device);
    CK(m, m->b_tkv.ensure((size_t)k * 8));
    CK(m, m->b_reloc.ensure((size_t)k * (24 + 4) + 16 + 64));
    rc = ndt2d_sweep_device(m, level, d_xy, n, d_hyp, nhyp, nullptr, k, d_best_idx, m->b_tkv.as<double>());
    if (rc) return rc;
    // layout of b_reloc: offsets[2] (i64) | init[3k] (f64) | job_scan[k] (i32)
    int64_t *d_off = m->b_reloc.as<int64_t>();
    double *d_init = reinterpret_cast<double *>(d_off + 2);
    int32_t *d_jobs = reinterpret_cast<int32_t *>(d_init + 3 * (size_t)k);
    m->reloc_off[0] = 0;
    m->reloc_off[1] = n;
    CK(m, cudaMemcpyAsync(d_off, m->reloc_off, 16, cudaMemcpyHostToDevice, m->cfg.stream));
    CK(m, launch_topk_to_jobs(m->cfg, d_hyp, d_best_idx, k, d_init, d_jobs, &m->launches));
    AlignArgs a{};
    a.xy = reinterpret_cast<const float2 *>(d_xy);
    a.offsets = d_off;
    a.job_scan = d_jobs;
    a.init = d_init;
    a.res = d_res;
    a.nscans = k;
    return align_device(m, a, n);
}

int ndt2d_relocalize(ndt2d_matcher *m, int level, const float *xy, int n, const float *hyp, int64_t nhyp, int k,
                     int64_t *best_idx, ndt2d_result *res)
{
    if (!m) return NDT2D_EINVAL;
    if (k < 1 || k > 1024 || !best_idx || !res || n < 0 || nhyp < 0 || (n > 0 && !xy) || (nhyp > 0 && !hyp))
        return fail(m, NDT2D_EINVAL, "bad arguments");
    int rc = check_level(m, level);
    if (rc) return rc;
    DeviceGuard g(m->device);
    if ((rc = upload(m, m->b_xy, xy, (size_t)n * 8))) return rc;
    if ((rc = upload(m, m->b_hyp, hyp, (size_t)nhyp * 12))) return rc;
    CK(m, m->b_tki.ensure((size_t)k * 8));
    CK(m, m->b_res.ensure((size_t)k * sizeof(ndt2d_result)));
    rc = ndt2d_relocalize_device(m, level, m->b_xy.as<float>(), n, m->b_hyp.as<float>(), nhyp, k, m->b_tki.as<int64_t>(),
                                 m->b_res.as<ndt2d_result>());
    if (rc) return rc;
    CK(m, cudaMemcpyAsync(best_idx, m->b_tki.p, (size_t)k * 8, cudaMemcpyDeviceToHost, m->cfg.stream));
    CK(m, cudaMemcpyAsync(res, m->b_res.p, (size_t)k * sizeof(ndt2d_result), cudaMemcpyDeviceToHost, m->cfg.stream));
    rc = ndt2d_synchronize(m);          // the one synchronisation of the call
    if (rc) return rc;
    for (int j = 0; j < k; ++j)
        if (best_idx[j] < 0) {          // fewer than k hypotheses: no candidate, no result
            memset(res + j, 0, sizeof(ndt2d_result));
            res[j].status = NDT2D_NO_OVERLAP;
        }
    return NDT2D_OK;
}

int ndt2d_set_upload_relay(ndt2d_matcher *m, int relay_device, double fraction)
{
    if (!m) return NDT2D_EINVAL;
    int rs = ndt2d_synchronize(m);
    if (rs) return rs;
    release_relay(m);
    if (relay_device < 0) return NDT2D_OK;
    int ndev = 0;
    CK(m, cudaGetDeviceCount(&ndev));
    if (relay_device >= ndev || relay_device == m->device || !(fraction > 0.0) || !(fraction < 1.0))
        return fail(m, NDT2D_EINVAL, "upload relay: device %d (this handle: %d, %d devices), fraction %g (0 < f < 1)", relay_device, m->device,
                    ndev, fraction);
    int can = 0;
    CK(m, cudaDeviceCanAccessPeer(&can, m->device, relay_device));
    if (!can) return fail(m, NDT2D_EINVAL, "upload relay: device %d cannot access device %d as a peer", m->device, relay_device);
    {
        DeviceGuard g(m->device);
        cudaError_t e = cudaDeviceEnablePeerAccess(relay_device, 0);
        if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) CK(m, e);
        cudaGetLastError();
        CK(m, cudaStreamCreateWithFlags(&m->relay_peer_stream, cudaStreamNonBlocking));
    }
    m->relay_dev = relay_device;        // from here on release_relay() undoes a partial set-up
    {
        DeviceGuard g(relay_device);
        cudaError_t e = cudaDeviceEnablePeerAccess(m->device, 0);
        if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) { release_relay(m); CK(m, e); }
        cudaGetLastError();
        e = cudaStreamCreateWithFlags(&m->relay_stream, cudaStreamNonBlocking);
        for (int i = 0; i < ndt2d_matcher::MAX_CHUNKS && e == cudaSuccess; ++i) e = cudaEventCreateWithFlags(&m->ev_relay[i], cudaEventDisableTiming);
        if (e != cudaSuccess) { release_relay(m); CK(m, e); }
    }
    m->relay_frac = fraction;
    return NDT2D_OK;
}

int ndt2d_host_alloc(void **p, size_t bytes) { return ndt2d_host_alloc_flags(p, bytes, 0); }

int ndt2d_host_alloc_flags(void **p, size_t bytes, int flags)
{
    if (!p) return NDT2D_EINVAL;
    cudaError_t e = cudaHostAlloc(p, bytes ? bytes : 1, (flags & NDT2D_HOST_WRITE_COMBINED) ? cudaHostAllocWriteCombined : cudaHostAllocDefault);
    if (e != cudaSuccess) {
        fail(nullptr, NDT2D_ENOMEM, "cudaHostAlloc(%zu): %s", bytes, cudaGetErrorString(e));
        return NDT2D_ENOMEM;
    }
    return NDT2D_OK;
}

int ndt2d_host_free(void *p)
{
    if (!p) return NDT2D_OK;
    return cudaFreeHost(p) == cudaSuccess ? NDT2D_OK : NDT2D_ECUDA;
}

} // extern "C"
