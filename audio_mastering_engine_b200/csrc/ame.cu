// libame host side: plan construction (job tables, workspace, waves) and the C ABI of include/ame.h.
#include <algorithm>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <dlfcn.h>
#include <mutex>
#include <string>
#include <vector>

#include "ame_kernels.cuh"

using namespace ame;

namespace {

thread_local std::string g_err;

int fail(int code, const char *fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    g_err = buf;
    return code;
}

#define CU(call)                                                                                   \
    do {                                                                                           \
        cudaError_t e_ = (call);                                                                   \
        if (e_ != cudaSuccess)                                                                     \
            return fail(AME_E_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__); \
    } while (0)

// Every entry point works on its plan's device and leaves the caller's current device as it found it (a process may
// drive plans on several GPUs, and torch allocates on the current device).
struct DeviceGuard {
    int prev = -1;
    cudaError_t err;
    explicit DeviceGuard(int dev) {
        err = cudaGetDevice(&prev);
        if (err == cudaSuccess && prev != dev) err = cudaSetDevice(dev);
    }
    ~DeviceGuard() {
        int cur = -1;
        if (prev >= 0 && cudaGetDevice(&cur) == cudaSuccess && cur != prev) cudaSetDevice(prev);
    }
};
#define GUARD(dev)                                                                                 \
    DeviceGuard guard_(dev);                                                                       \
    if (guard_.err != cudaSuccess) return fail(AME_E_CUDA, "cannot select CUDA device %d: %s", (int)(dev), cudaGetErrorString(guard_.err))

// Device memory comes from one stream-ordered pool per device whose release threshold is lifted: the workspace of a
// destroyed plan stays in the pool and the next plan gets it back in microseconds.  (cudaMalloc + cudaFree of the
// ~25 buffers of a plan cost 50 - 150 ms, several times what mastering a 3 min track takes; profiles/r01e_summary.md.)
// Allocation and release are ordered on the legacy default stream, which every entry point that allocates
// synchronises before it returns; ame_release_cached_memory() hands the pool back to the driver.
constexpr int kMaxDevices = 64;
std::mutex g_pool_mutex;
cudaMemPool_t g_pools[kMaxDevices] = {};
bool g_pool_tried[kMaxDevices] = {};

cudaMemPool_t device_pool() {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= kMaxDevices) return nullptr;
    std::lock_guard<std::mutex> lock(g_pool_mutex);
    if (!g_pool_tried[dev]) {
        g_pool_tried[dev] = true;
        int ok = 0;
        cudaDeviceGetAttribute(&ok, cudaDevAttrMemoryPoolsSupported, dev);
        if (ok) {
            cudaMemPoolProps props = {};
            props.allocType = cudaMemAllocationTypePinned;
            props.handleTypes = cudaMemHandleTypeNone;
            props.location.type = cudaMemLocationTypeDevice;
            props.location.id = dev;
            cudaMemPool_t pool = nullptr;
            unsigned long long keep = ~0ull;
            if (cudaMemPoolCreate(&pool, &props) == cudaSuccess &&
                cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep) == cudaSuccess)
                g_pools[dev] = pool;
            else
                cudaGetLastError();
        }
    }
    return g_pools[dev];
}

cudaError_t dev_alloc(void **ptr, size_t bytes) {
    if (cudaMemPool_t pool = device_pool()) return cudaMallocFromPoolAsync(ptr, bytes, pool, 0);
    return cudaMalloc(ptr, bytes);
}

void dev_free(void *ptr) {
    if (!ptr) return;
    if (device_pool()) cudaFreeAsync(ptr, 0); else cudaFree(ptr);
}

constexpr int kEqBlock = 256;            // k_eq: 8 warps in ONE CTA per SM (two 4-warp CTAs were slower, see build_layout)
constexpr int kMaxTimedSteps = 8;
constexpr int kMaxTimedWaves = 128;
constexpr int kTimedSlots = kMaxTimedWaves * AME_N_KERNELS;   // per step
const char *const kKernelNames[AME_N_KERNELS] = {"k_eq", "k_band_split", "k_window_flag", "k_att_chain",
    "k_compress_apply", "k_kweight_energy", "k_tail_peak", "k_block_hist", "k_finalize", "k_apply_gain", "k_limiter", "k_true_peak"};
enum { S_EQ = 0, S_SPLIT, S_FLAG, S_CHAIN, S_APPLY, S_KW, S_TAIL, S_HIST, S_FIN, S_GAIN, S_LIM, S_TP };

// Per-wave workspace.  A plan has n_slots of them; wave w runs in slot w % n_slots on that slot's stream, so a slot is
// recycled in stream order and a plan over many waves needs the intermediate buffers of only n_slots waves.
struct Slot {
    int16_t *pre = nullptr;      // pre-normalisation int16 of the wave (the signal the reference materialises at the concat)
    int16_t *bands = nullptr;    // 3 planes of mb_frames frames
    uint16_t *rms = nullptr;     // 3 planes: integer window rms of flagged frames, 0 elsewhere
    uint16_t *list = nullptr;    // 3 planes: per chain the rms values of its flagged frames, dense
    int *tile_cnt = nullptr;     // flagged frames per k_window_flag tile
    int *n_flagged = nullptr;    // flagged frames per chain
    GrpRec *grp = nullptr;       // per 32-frame group of every chain
    double *att = nullptr;       // 3 planes: attenuation after every flagged frame, dense per chain
    int16_t *norm = nullptr;     // the normalised signal of tracks with the limiter stage (k_apply_gain -> k_limiter)
    long long *lim_last = nullptr;   // per k_apply_gain tile: last frame over the limiter's limit, or -1
    LimStore lim_in{}, lim_out{};    // per tile: the limiter state it started from / ended in
    int *lim_need = nullptr;         // per tile: its start is not its predecessor's end (yet)
    cudaStream_t stream = nullptr;
};

}  // namespace

// A plan is its layout (ame_layout.h) plus the device state built from it.
struct ame_plan : Layout {
    int device = 0;
    int n_tracks = 0;
    int n_sm = 148, chain_warps = 0;      // see chain_lanes()
    int precision = 0;                    // 1 = the FP32 EQ experiment
    std::vector<void *> allocs;           // every device allocation of the plan (plan_alloc), freed by ame_plan_destroy
    size_t ws_bytes = 0;
    int64_t launches = 0;
    // device
    ame_track_params *d_tracks = nullptr;
    TrackDev *d_tdev = nullptr;
    int64_t *d_mb_delta = nullptr;
    TileJob *d_eq_jobs = nullptr, *d_split_jobs = nullptr;
    ChainJob *d_chain_jobs = nullptr;
    WfJob *d_wf_jobs = nullptr;
    MbChunk *d_mb_chunks = nullptr;
    KwJob *d_kw_jobs = nullptr;
    GainJob *d_gain_jobs = nullptr, *d_lim_jobs = nullptr;
    AttEntry *d_tables = nullptr;
    double *d_luts = nullptr;
    int n_luts = 0;
    int16_t *d_in = nullptr, *d_out = nullptr;
    std::vector<Slot> slots;
    double *d_energy = nullptr;
    int *d_chain_stats = nullptr;          // per chain: {flagged steps, passes} of the last k_att_chain
    long long *d_hist = nullptr;
    int *d_hist_st = nullptr;               // short-term (3 s) histogram per track, for loudness range
    int *d_peak = nullptr;
    unsigned *d_tp = nullptr;               // per track: float bits of the oversampled peak (k_true_peak)
    int *d_lim_stats = nullptr;             // open tiles after the limiter's round 0 / 1 / 2, accumulated
    int lim_guess = -1;                     // frames of the limiter's round-0 guess; -1 = 2 G (ame_plan_set_limiter_guess)
    ame_track_result *d_results = nullptr;
    // output meter (tracks with AME_F_MEASURE_OUTPUT; none of it exists without such a track)
    KwJob *d_meter_kw = nullptr;
    GainJob *d_meter_peak = nullptr;
    int32_t *d_meter_tracks = nullptr;
    TrackDev *d_meter_tdev = nullptr;
    double *d_meter_energy = nullptr;       // sub-block energies of the flagged tracks (meter_tdev[t].sb_offset)
    int *d_meter_sp = nullptr;              // per track: sample peak
    unsigned *d_meter_tp = nullptr;         // per track: float bits of the oversampled peak
    ame_loudness *d_loud_out = nullptr;     // per track: meter of the last ame_master_* / ame_normalize_device call
    ame_loudness *d_loud_any = nullptr;     // per track: the last ame_measure_loudness
    cudaStream_t s_in = nullptr, s_out = nullptr;                       // host path: copy-in / copy-out
    std::vector<cudaEvent_t> ev_in, ev_run;                             // per wave
    std::vector<cudaEvent_t> ev_meter;                                  // host path with the meter: per slot, its last meter done
    // optional per-kernel CUDA-event timing (ame_plan_set_timing)
    bool timing = false;
    int t_step = -1, t_wave = 0;
    std::vector<cudaEvent_t> t_ev;        // [kMaxTimedSteps][kMaxTimedWaves][AME_N_KERNELS][2]
    std::vector<char> t_used;             // [kMaxTimedSteps][kMaxTimedWaves][AME_N_KERNELS]
    std::vector<cudaEvent_t> tl_ev;       // host-path timeline of the last timed ame_master_host: start, then per wave
    int tl_waves = 0;                     //   {H2D done, first kernel may start, kernels done, D2H done}
};

namespace {

inline bool t_on(const ame_plan *p) {
    return p->timing && p->t_step >= 0 && p->t_step < kMaxTimedSteps && p->t_wave < kMaxTimedWaves;
}
inline size_t t_slot(const ame_plan *p, int kernel) {
    return ((size_t)p->t_step * kMaxTimedWaves + p->t_wave) * AME_N_KERNELS + kernel;
}
inline void t_begin(ame_plan *p, int kernel, cudaStream_t s) {
    if (t_on(p)) cudaEventRecord(p->t_ev[t_slot(p, kernel) * 2], s);
}
inline void t_end(ame_plan *p, int kernel, cudaStream_t s) {
    if (t_on(p)) {
        cudaEventRecord(p->t_ev[t_slot(p, kernel) * 2 + 1], s);
        p->t_used[t_slot(p, kernel)] = 1;
    }
}

// The one allocator of a plan's device memory: it records every pointer, and ame_plan_destroy frees what it recorded.
int plan_alloc(ame_plan *p, void **ptr, size_t bytes) {
    *ptr = nullptr;
    if (bytes == 0) return AME_OK;
    cudaError_t e = dev_alloc(ptr, bytes);
    if (e != cudaSuccess) {
        *ptr = nullptr;
        return fail(AME_E_NOMEM, "device allocation of %zu bytes failed: %s", bytes, cudaGetErrorString(e));
    }
    p->allocs.push_back(*ptr);
    return AME_OK;
}

// workspace: counted by ame_plan_workspace_bytes, which leaves the uploaded tables out
int dmalloc(ame_plan *p, void **ptr, size_t bytes) {
    const int rc = plan_alloc(p, ptr, bytes);
    if (rc == AME_OK) p->ws_bytes += bytes;
    return rc;
}

template <class T>
int upload(ame_plan *p, T **dptr, const std::vector<T> &v) {
    if (int rc = plan_alloc(p, (void **)dptr, v.size() * sizeof(T))) return rc;
    if (!v.empty()) CU(cudaMemcpy(*dptr, v.data(), v.size() * sizeof(T), cudaMemcpyHostToDevice));
    return AME_OK;
}

#define LAUNCH_CHECK(p)                                                                            \
    do {                                                                                           \
        cudaError_t e_ = cudaGetLastError();                                                       \
        if (e_ != cudaSuccess) return fail(AME_E_CUDA, "kernel launch failed: %s (%s:%d)", cudaGetErrorString(e_), __FILE__, __LINE__); \
        ++(p)->launches;                                                                           \
    } while (0)

int check_warmth(const ame_plan *p) {
    for (int t = 0; t < p->n_tracks; ++t)
        if (p->tracks[t].flags & AME_F_WARMTH) {
            const int l = p->tracks[t].warm_lut;
            if (l < 0 || l >= p->n_luts) return fail(AME_E_INVALID, "track %d needs warmth table %d but %d are set", t, l, p->n_luts);
        }
    return AME_OK;
}

// ---- stage launches over one wave ------------------------------------------------------------------
// `pre` is addressed with ABSOLUTE packed-buffer frame indices everywhere: for a slot the pointer handed in is
// slot.pre - 2 * wave.frame_lo (never dereferenced outside the wave's own range).
struct Bufs {
    const int16_t *in = nullptr;
    int16_t *pre = nullptr, *bands = nullptr, *out = nullptr;
    uint16_t *rms = nullptr, *list = nullptr;
    int *tile_cnt = nullptr, *n_flagged = nullptr;
    GrpRec *grp = nullptr;
    double *att = nullptr;
    int64_t *hist = nullptr;
    int16_t *norm = nullptr;
    long long *lim_last = nullptr;
    LimStore lim_in{}, lim_out{};
    int *lim_need = nullptr;
};

Bufs slot_bufs(ame_plan *p, const Wave &w, const int16_t *d_in, int16_t *d_out) {
    const Slot &sl = p->slots[w.slot];
    Bufs b;
    b.in = d_in; b.out = d_out;
    b.pre = sl.pre - 2 * w.frame_lo;
    b.bands = sl.bands; b.rms = sl.rms; b.list = sl.list; b.tile_cnt = sl.tile_cnt; b.n_flagged = sl.n_flagged;
    b.grp = sl.grp; b.att = sl.att;
    b.norm = sl.norm ? sl.norm - 2 * w.frame_lo : nullptr;
    b.lim_last = sl.lim_last; b.lim_in = sl.lim_in; b.lim_out = sl.lim_out; b.lim_need = sl.lim_need;
    b.hist = (int64_t *)p->d_hist;
    return b;
}

int run_eq(ame_plan *p, const Wave &w, const int16_t *d_in, int16_t *d_pre, cudaStream_t s) {
    if (!w.eq.n) return AME_OK;
    t_begin(p, S_EQ, s);
    if (p->precision == 1)
        k_eq_f32<<<(w.eq.n + 127) / 128, 128, 0, s>>>(p->d_eq_jobs + w.eq.lo, w.eq.n, p->d_tracks, p->d_luts, d_in, d_pre);
    else
        k_eq<<<(w.eq.n + kEqBlock - 1) / kEqBlock, kEqBlock, 0, s>>>(p->d_eq_jobs + w.eq.lo, w.eq.n, p->d_tracks, p->d_luts, d_in, d_pre);
    LAUNCH_CHECK(p);
    t_end(p, S_EQ, s);
    return AME_OK;
}

int run_split(ame_plan *p, const Wave &w, const int16_t *d_pre, int16_t *d_bands, cudaStream_t s) {
    if (!w.split.n) return AME_OK;
    t_begin(p, S_SPLIT, s);
    if (w.xover_uni)
        k_band_split<true><<<(w.split.n + 127) / 128, 128, 0, s>>>(w.xover, p->d_split_jobs + w.split.lo, w.split.n, p->d_tracks, p->d_mb_delta,
                                                                   d_pre, d_bands, p->mb_frames);
    else
        k_band_split<false><<<(w.split.n + 127) / 128, 128, 0, s>>>(w.xover, p->d_split_jobs + w.split.lo, w.split.n, p->d_tracks, p->d_mb_delta,
                                                                    d_pre, d_bands, p->mb_frames);
    LAUNCH_CHECK(p);
    t_end(p, S_SPLIT, s);
    return AME_OK;
}

// Lanes (time segments) per chain of k_att_chain.  More lanes = shorter segments = cheaper passes but more of them once
// a segment is shorter than the distance after which trajectories meet.  Alone on the GPU a chain is fastest with 8
// warps (few chains) or 4; in a batch, where launches of several waves share the SMs, a 216-register lane is worth
// more as room for the other kernels than as a shorter segment: 2 warps (1024 tracks: 223-225 ms per step against
// 228 with 4 warps and 239 with 6, profiles/r02/scheduling_experiments.txt).
int chain_lanes(const ame_plan *p, int n_chains) {
    if (p->chain_warps < 0) return 1;                       // ONE lane per chain: the sequential loop
    if (p->chain_warps > 0) return 32 * p->chain_warps;
    if (n_chains * 2 <= p->n_sm) return 256;
    return (n_chains >= p->n_sm && p->slots.size() > 1) ? 64 : 128;
}

int run_compress(ame_plan *p, const Wave &w, const Bufs &b, cudaStream_t s) {
    if (!w.chain.n) return AME_OK;
    t_begin(p, S_FLAG, s);
    int *tile_base = b.tile_cnt + std::max(p->slot_tiles, 1);
    k_window_flag<<<w.wf.n, kWfThreads, 0, s>>>(p->d_wf_jobs + w.wf.lo, b.bands, b.rms, b.tile_cnt, b.grp);
    LAUNCH_CHECK(p);
    k_tile_prefix<<<w.chain.n, kWfThreads, 0, s>>>(p->d_chain_jobs + w.chain.lo, b.tile_cnt, tile_base, b.n_flagged);
    LAUNCH_CHECK(p);
    k_compact<<<(w.wf.n + kWfThreads / 32 - 1) / (kWfThreads / 32), kWfThreads, 0, s>>>(p->d_wf_jobs + w.wf.lo, w.wf.n, b.rms, b.tile_cnt,
                                                                                          tile_base, b.list, b.grp);
    LAUNCH_CHECK(p);
    t_end(p, S_FLAG, s);
    t_begin(p, S_CHAIN, s);
    const int lanes = chain_lanes(p, w.chain.n);
    k_att_chain<<<w.chain.n, std::max(lanes, 32), 0, s>>>(p->d_chain_jobs + w.chain.lo, b.list, b.n_flagged, p->d_tables, b.att, p->mb_frames,
                                            lanes, p->d_chain_stats + 2 * (size_t)w.chain.lo);
    LAUNCH_CHECK(p);
    t_end(p, S_CHAIN, s);
    t_begin(p, S_APPLY, s);
    k_compress_apply<<<(unsigned)((w.seg_hi - w.seg_lo + 3) / 4), 128, 0, s>>>(p->d_mb_chunks + w.mb_chunks.lo, w.mb_chunks.n, w.seg_lo, w.seg_hi,
                                                                                b.bands, b.grp, b.att, b.pre, p->mb_frames);
    LAUNCH_CHECK(p);
    t_end(p, S_APPLY, s);
    return AME_OK;
}

int run_hist(ame_plan *p, const Wave &w, const int16_t *d_pre, int64_t *d_hist, cudaStream_t s) {
    const int nt = w.track_hi - w.track_lo;
    if (nt <= 0) return AME_OK;
    CU(cudaMemsetAsync(p->d_peak + w.track_lo, 0, (size_t)nt * 4, s));
    if (w.kw.n) {
        t_begin(p, S_KW, s);
        if (w.kw_uni)
            k_kweight_energy<true><<<(w.kw.n + 127) / 128, 128, 0, s>>>(w.kw_cfg, p->d_kw_jobs + w.kw.lo, w.kw.n, p->d_tracks, p->d_tdev, d_pre,
                                                                        p->d_energy, p->d_peak);
        else
            k_kweight_energy<false><<<(w.kw.n + 127) / 128, 128, 0, s>>>(w.kw_cfg, p->d_kw_jobs + w.kw.lo, w.kw.n, p->d_tracks, p->d_tdev, d_pre,
                                                                         p->d_energy, p->d_peak);
        LAUNCH_CHECK(p);
        t_end(p, S_KW, s);
    }
    t_begin(p, S_TAIL, s);
    k_tail_peak<<<nt, 128, 0, s>>>(p->d_tracks, p->d_tdev, w.track_lo, w.track_hi, d_pre, p->d_peak);
    LAUNCH_CHECK(p);
    t_end(p, S_TAIL, s);
    CU(cudaMemsetAsync(p->d_tp + w.track_lo, 0, (size_t)nt * 4, s));
    if (w.true_peak && w.gain.n) {
        t_begin(p, S_TP, s);
        k_true_peak<<<w.gain.n, 256, 0, s>>>(p->d_gain_jobs + w.gain.lo, p->d_tracks, d_pre, p->d_tp);
        LAUNCH_CHECK(p);
        t_end(p, S_TP, s);
    }
    t_begin(p, S_HIST, s);
    k_block_hist<<<nt, 256, 0, s>>>(p->d_tdev, w.track_lo, p->d_energy, (long long *)d_hist, p->d_hist_st);
    LAUNCH_CHECK(p);
    t_end(p, S_HIST, s);
    return AME_OK;
}

// static gain (+ the limiter's input and per-tile "last frame over the limit") and the limiter; needs d_results
int run_apply(ame_plan *p, const Wave &w, const int16_t *d_pre, int16_t *d_out, const Bufs &b, cudaStream_t s) {
    int16_t *d_norm = b.norm;
    long long *lim_last = b.lim_last;
    if (!w.gain.n) return AME_OK;
    t_begin(p, S_GAIN, s);
    if (w.limiter) CU(cudaMemsetAsync(lim_last, 0xff, (size_t)w.lim.n * sizeof(long long), s));      // -1: no frame over the limit
    k_apply_gain<<<w.gain.n, 256, 0, s>>>(p->d_gain_jobs + w.gain.lo, p->d_results, p->d_tracks, p->d_tdev, d_pre, d_out, d_norm, lim_last);
    LAUNCH_CHECK(p);
    t_end(p, S_GAIN, s);
    if (w.limiter) {
        t_begin(p, S_LIM, s);
        const GainJob *gj = p->d_lim_jobs + w.lim.lo;
        constexpr int kLimRounds = 2;                 // repair rounds before the sequential fallback
        int cap = 64;
        while (cap < p->lim_keep + 2) cap *= 2;       // queue capacity in shared memory: a power of two
        const size_t smem = lim_smem_bytes(cap);
        for (int round = 0; round <= kLimRounds; ++round) {
            if (round == 0) {                         // the elementwise tiles, 256 threads each
                k_limiter<<<w.lim.n, 256, smem, s>>>(gj, w.lim.n, lim_last, p->d_tracks, d_norm, d_out, b.lim_in, b.lim_out, b.lim_need, 0, cap, p->lim_guess);
                LAUNCH_CHECK(p);
            }
            k_limiter<<<w.lim.n, 32, smem, s>>>(gj, w.lim.n, lim_last, p->d_tracks, d_norm, d_out, b.lim_in, b.lim_out, b.lim_need, round, cap, p->lim_guess);
            LAUNCH_CHECK(p);
            k_lim_verify<<<(w.lim.n + 3) / 4, 128, 0, s>>>(gj, w.lim.n, p->d_tracks, b.lim_in, b.lim_out, b.lim_need,
                                                             p->d_lim_stats + round);
            LAUNCH_CHECK(p);
        }
        k_lim_fallback<<<w.lim.n, 32, smem, s>>>(gj, w.lim.n, p->d_tracks, d_norm, d_out, b.lim_in, b.lim_out, b.lim_need, cap);
        LAUNCH_CHECK(p);
        t_end(p, S_LIM, s);
    }
    return AME_OK;
}

int run_gain(ame_plan *p, const Wave &w, const int16_t *d_pre, const int64_t *d_hist, int16_t *d_out, const Bufs &b, cudaStream_t s) {
    const int nt = w.track_hi - w.track_lo;
    if (nt <= 0) return AME_OK;
    t_begin(p, S_FIN, s);
    k_finalize<<<nt, 128, 0, s>>>(p->d_tracks, w.track_lo, w.track_hi, (const long long *)d_hist, p->d_hist_st, p->d_peak,
                                             p->d_tp, p->d_results);
    LAUNCH_CHECK(p);
    t_end(p, S_FIN, s);
    return run_apply(p, w, d_pre, d_out, b, s);
}

// the output meter over the flagged tracks of wave w, read from `buf` (absolute packed-buffer addressing), into `res`
int run_meter(ame_plan *p, const Wave &w, const int16_t *buf, ame_loudness *res, cudaStream_t s) {
    if (!w.meter_tracks.n) return AME_OK;
    const int nt = w.track_hi - w.track_lo;
    CU(cudaMemsetAsync(p->d_meter_sp + w.track_lo, 0, (size_t)nt * 4, s));
    CU(cudaMemsetAsync(p->d_meter_tp + w.track_lo, 0, (size_t)nt * 4, s));
    if (w.meter_kw.n) {
        if (w.kw_uni)
            k_kweight_energy<true><<<(w.meter_kw.n + 127) / 128, 128, 0, s>>>(w.kw_cfg, p->d_meter_kw + w.meter_kw.lo, w.meter_kw.n, p->d_tracks,
                                                                              p->d_meter_tdev, buf, p->d_meter_energy, p->d_meter_sp);
        else
            k_kweight_energy<false><<<(w.meter_kw.n + 127) / 128, 128, 0, s>>>(w.kw_cfg, p->d_meter_kw + w.meter_kw.lo, w.meter_kw.n, p->d_tracks,
                                                                               p->d_meter_tdev, buf, p->d_meter_energy, p->d_meter_sp);
        LAUNCH_CHECK(p);
    }
    if (w.meter_peak.n) {
        k_meter_peak<<<w.meter_peak.n, 256, 0, s>>>(p->d_meter_peak + w.meter_peak.lo, p->d_tracks, buf, p->d_meter_tp, p->d_meter_sp);
        LAUNCH_CHECK(p);
    }
    k_meter_finalize<<<w.meter_tracks.n, 256, 0, s>>>(p->d_meter_tracks + w.meter_tracks.lo, p->d_tracks, p->d_meter_tdev, p->d_meter_energy,
                                                      p->d_meter_sp, p->d_meter_tp, res);
    LAUNCH_CHECK(p);
    return AME_OK;
}

int run_measure(ame_plan *p, const Wave &w, const Bufs &b, cudaStream_t s) {
    int rc;
    if ((rc = run_eq(p, w, b.in, b.pre, s))) return rc;
    if ((rc = run_split(p, w, b.pre, b.bands, s))) return rc;
    if ((rc = run_compress(p, w, b, s))) return rc;
    return run_hist(p, w, b.pre, b.hist, s);
}

int run_chain_of_stages(ame_plan *p, const Wave &w, const Bufs &b, cudaStream_t s) {
    int rc = run_measure(p, w, b, s);
    if (rc) return rc;
    return run_gain(p, w, b.pre, b.hist, b.out, b, s);
}

// after a failure in the middle of a pipelined call nothing may still be reading the caller's buffers when we return
int drain(ame_plan *p, int rc) {
    (void)p;
    if (rc != AME_OK) cudaDeviceSynchronize();
    return rc;
}

}  // namespace

extern "C" {

int ame_abi_version(void) { return AME_ABI_VERSION; }
size_t ame_sizeof_track_params(void) { return sizeof(ame_track_params); }
size_t ame_sizeof_track_result(void) { return sizeof(ame_track_result); }
size_t ame_sizeof_plan_options(void) { return sizeof(ame_plan_options); }
size_t ame_sizeof_loudness(void) { return sizeof(ame_loudness); }
const char *ame_last_error(void) { return g_err.c_str(); }
const char *ame_kernel_name(int slot) { return (slot >= 0 && slot < AME_N_KERNELS) ? kKernelNames[slot] : ""; }

int ame_device_count(int *count) {
    if (!count) return fail(AME_E_INVALID, "count is NULL");
    *count = 0;
    CU(cudaGetDeviceCount(count));
    return AME_OK;
}

void ame_plan_destroy(ame_plan *p) {
    if (!p) return;
    DeviceGuard guard(p->device);
    cudaDeviceSynchronize();            // nothing of this plan may still be running when its memory goes back to the pool
    for (void *q : p->allocs) dev_free(q);
    for (Slot &sl : p->slots)
        if (sl.stream) cudaStreamDestroy(sl.stream);
    for (cudaStream_t s : {p->s_in, p->s_out})
        if (s) cudaStreamDestroy(s);
    for (cudaEvent_t e : p->ev_in) cudaEventDestroy(e);
    for (cudaEvent_t e : p->ev_run) cudaEventDestroy(e);
    for (cudaEvent_t e : p->ev_meter) cudaEventDestroy(e);
    for (cudaEvent_t e : p->t_ev) cudaEventDestroy(e);
    for (cudaEvent_t e : p->tl_ev) cudaEventDestroy(e);
    delete p;
}

int ame_plan_create(int device, const ame_track_params *tracks, int32_t n_tracks, const ame_plan_options *opt,
                    ame_plan **out) {
    if (!out) return fail(AME_E_INVALID, "plan out-pointer is NULL");
    *out = nullptr;
    if (!tracks || n_tracks <= 0) return fail(AME_E_INVALID, "no tracks");
    int ndev = 0;
    CU(cudaGetDeviceCount(&ndev));
    if (device < 0 || device >= ndev) return fail(AME_E_CUDA, "CUDA device %d not available (%d devices)", device, ndev);
    GUARD(device);
    ame_plan_options o{};
    if (opt) o = *opt;

    ame_plan *p = new ame_plan();
    p->device = device;
    p->n_tracks = n_tracks;
    p->chain_warps = std::max(-1, std::min(o.chain_warps, kChainMaxThreads / 32));
    p->precision = o.precision == 1 ? 1 : 0;
    auto bail = [&](int code) { ame_plan_destroy(p); return code; };

    // ---- layout: tiles are sized for the resident 128-thread CTAs of k_eq and k_band_split -------------
    DeviceShape shape{148, 2, 3};
    cudaDeviceGetAttribute(&shape.n_sm, cudaDevAttrMultiProcessorCount, device);
    if (p->precision == 1) cudaOccupancyMaxActiveBlocksPerMultiprocessor(&shape.occ_eq, k_eq_f32, 128, 0);
    else cudaOccupancyMaxActiveBlocksPerMultiprocessor(&shape.occ_eq, k_eq, 128, 0);
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&shape.occ_split, k_band_split<true>, 128, 0);
    p->n_sm = shape.n_sm;
    JobTables jobs;
    std::string err;
    int rc = build_layout(tracks, n_tracks, o, shape, *p, jobs, err);
    if (rc) {
        g_err = err;
        return bail(rc);
    }

    // ---- device state -------------------------------------------------------------------------
    if ((rc = upload(p, &p->d_tracks, p->tracks)) || (rc = upload(p, &p->d_tdev, p->tdev)) || (rc = upload(p, &p->d_mb_delta, jobs.mb_delta)) ||
        (rc = upload(p, &p->d_eq_jobs, jobs.eq)) || (rc = upload(p, &p->d_split_jobs, jobs.split)) ||
        (rc = upload(p, &p->d_chain_jobs, jobs.chain)) || (rc = upload(p, &p->d_wf_jobs, jobs.wf)) ||
        (rc = upload(p, &p->d_mb_chunks, jobs.mb_chunks)) || (rc = upload(p, &p->d_kw_jobs, jobs.kw)) ||
        (rc = upload(p, &p->d_gain_jobs, jobs.gain)) || (rc = upload(p, &p->d_lim_jobs, jobs.lim)) || (rc = upload(p, &p->d_tables, jobs.att)))
        return bail(rc);
    if (p->any_meter &&
        ((rc = upload(p, &p->d_meter_kw, jobs.meter_kw)) || (rc = upload(p, &p->d_meter_peak, jobs.meter_peak)) ||
         (rc = upload(p, &p->d_meter_tracks, jobs.meter_tracks)) || (rc = upload(p, &p->d_meter_tdev, p->meter_tdev))))
        return bail(rc);
    const size_t fb = (size_t)p->total_frames * 4;
    p->slots.resize(p->n_slots);
    for (Slot &sl : p->slots) {
        if ((rc = dmalloc(p, (void **)&sl.pre, (size_t)p->slot_frames * 4)) ||
            (rc = dmalloc(p, (void **)&sl.bands, (size_t)p->mb_frames * 4 * 3)) ||
            (rc = dmalloc(p, (void **)&sl.rms, (size_t)p->mb_frames * 2 * 3)) ||
            (rc = dmalloc(p, (void **)&sl.list, (size_t)p->mb_frames * 2 * 3)) ||
            (rc = dmalloc(p, (void **)&sl.tile_cnt, (size_t)std::max(p->slot_tiles, 1) * 2 * sizeof(int))) ||     // counts, then ranks
            (rc = dmalloc(p, (void **)&sl.n_flagged, (size_t)std::max(p->slot_chains, 1) * sizeof(int))) ||
            (rc = dmalloc(p, (void **)&sl.grp, (size_t)p->slot_groups * sizeof(GrpRec))) ||
            (rc = dmalloc(p, (void **)&sl.att, (size_t)p->mb_frames * 8 * 3)))
            return bail(rc);
        if (p->any_limiter &&
            ((rc = dmalloc(p, (void **)&sl.norm, (size_t)p->slot_frames * 4)) ||
             (rc = dmalloc(p, (void **)&sl.lim_last, (size_t)std::max(p->slot_lim_jobs, 1) * sizeof(long long))) ||
             (rc = dmalloc(p, (void **)&sl.lim_in.st, (size_t)std::max(p->slot_lim_jobs, 1) * sizeof(LimState))) ||
             (rc = dmalloc(p, (void **)&sl.lim_out.st, (size_t)std::max(p->slot_lim_jobs, 1) * sizeof(LimState))) ||
             (rc = dmalloc(p, (void **)&sl.lim_in.qframe, (size_t)std::max(p->slot_lim_jobs, 1) * p->lim_keep * sizeof(int))) ||
             (rc = dmalloc(p, (void **)&sl.lim_out.qframe, (size_t)std::max(p->slot_lim_jobs, 1) * p->lim_keep * sizeof(int))) ||
             (rc = dmalloc(p, (void **)&sl.lim_in.qdelta, (size_t)std::max(p->slot_lim_jobs, 1) * p->lim_keep * sizeof(double))) ||
             (rc = dmalloc(p, (void **)&sl.lim_out.qdelta, (size_t)std::max(p->slot_lim_jobs, 1) * p->lim_keep * sizeof(double))) ||
             (rc = dmalloc(p, (void **)&sl.lim_need, (size_t)std::max(p->slot_lim_jobs, 1) * sizeof(int)))))
            return bail(rc);
        sl.lim_in.keep = sl.lim_out.keep = p->lim_keep;
        // the filters read a few frames past a track's end (whole 16 / 32-byte groups, never stored): keep them defined
        if (cudaMemsetAsync(sl.pre, 0, (size_t)p->slot_frames * 4, 0) != cudaSuccess ||
            (p->mb_frames && cudaMemsetAsync(sl.bands, 0, (size_t)p->mb_frames * 12, 0) != cudaSuccess))
            return bail(fail(AME_E_CUDA, "cudaMemset failed"));
    }
    if ((rc = dmalloc(p, (void **)&p->d_chain_stats, std::max<size_t>(jobs.chain.size(), 1) * 2 * sizeof(int))) ||
        (rc = dmalloc(p, (void **)&p->d_energy, (size_t)std::max<int64_t>(p->n_sb_total, 1) * 8)) ||
        (rc = dmalloc(p, (void **)&p->d_hist, (size_t)n_tracks * 1000 * 8)) ||
        (rc = dmalloc(p, (void **)&p->d_hist_st, (size_t)n_tracks * 1000 * 4)) ||
        (rc = dmalloc(p, (void **)&p->d_peak, (size_t)n_tracks * 4)) ||
        (rc = dmalloc(p, (void **)&p->d_tp, (size_t)n_tracks * 4)) ||
        (rc = dmalloc(p, (void **)&p->d_lim_stats, 4 * sizeof(int))) ||
        (rc = dmalloc(p, (void **)&p->d_results, (size_t)n_tracks * sizeof(ame_track_result))))
        return bail(rc);
    if (cudaMemsetAsync(p->d_lim_stats, 0, 4 * sizeof(int), 0) != cudaSuccess) return bail(fail(AME_E_CUDA, "cudaMemset failed"));
    if (p->any_meter) {
        const size_t lb = (size_t)n_tracks * sizeof(ame_loudness);
        if ((rc = dmalloc(p, (void **)&p->d_meter_energy, (size_t)std::max<int64_t>(p->meter_sb_total, 1) * 8)) ||
            (rc = dmalloc(p, (void **)&p->d_meter_sp, (size_t)n_tracks * 4)) ||
            (rc = dmalloc(p, (void **)&p->d_meter_tp, (size_t)n_tracks * 4)) ||
            (rc = dmalloc(p, (void **)&p->d_loud_out, lb)) || (rc = dmalloc(p, (void **)&p->d_loud_any, lb)))
            return bail(rc);
        // measured = 0 everywhere until a call meters
        if (cudaMemsetAsync(p->d_loud_out, 0, lb, 0) != cudaSuccess || cudaMemsetAsync(p->d_loud_any, 0, lb, 0) != cudaSuccess)
            return bail(fail(AME_E_CUDA, "cudaMemset failed"));
    }
    if (cudaMemsetAsync(p->d_chain_stats, 0, std::max<size_t>(jobs.chain.size(), 1) * 2 * sizeof(int), 0) != cudaSuccess)
        return bail(fail(AME_E_CUDA, "cudaMemset failed"));
    if (o.host_io) {
        if ((rc = dmalloc(p, (void **)&p->d_in, fb)) || (rc = dmalloc(p, (void **)&p->d_out, fb))) return bail(rc);
        // pool memory is recycled: the padding between tracks is copied back to the caller with the wave, so it must
        // not carry another plan's audio
        if (cudaMemsetAsync(p->d_in, 0, fb, 0) != cudaSuccess || cudaMemsetAsync(p->d_out, 0, fb, 0) != cudaSuccess)
            return bail(fail(AME_E_CUDA, "cudaMemset failed"));
        if (cudaStreamCreateWithFlags(&p->s_in, cudaStreamNonBlocking) != cudaSuccess ||
            cudaStreamCreateWithFlags(&p->s_out, cudaStreamNonBlocking) != cudaSuccess)
            return bail(fail(AME_E_CUDA, "cudaStreamCreate failed"));
    }
    const int n_waves = (int)p->waves.size();
    if (o.host_io || n_waves > 1) {
        p->ev_in.resize(n_waves);
        p->ev_run.resize(n_waves);
        for (Slot &sl : p->slots)
            if (cudaStreamCreateWithFlags(&sl.stream, cudaStreamNonBlocking) != cudaSuccess)
                return bail(fail(AME_E_CUDA, "cudaStreamCreate failed"));
        for (int w = 0; w < n_waves; ++w)
            if (cudaEventCreateWithFlags(&p->ev_in[w], cudaEventDisableTiming) != cudaSuccess ||
                cudaEventCreateWithFlags(&p->ev_run[w], cudaEventDisableTiming) != cudaSuccess)
                return bail(fail(AME_E_CUDA, "cudaEventCreate failed"));
        if (o.host_io && p->any_meter) {
            p->ev_meter.resize(p->slots.size());
            for (cudaEvent_t &e : p->ev_meter)
                if (cudaEventCreateWithFlags(&e, cudaEventDisableTiming) != cudaSuccess) return bail(fail(AME_E_CUDA, "cudaEventCreate failed"));
        }
    }

    // ebur128.c histogram tables (same libm calls as the C library)
    {
        static double bounds[1001], energies[1000];
        bounds[0] = std::pow(10.0, (-70.0 + 0.691) / 10.0);
        for (int i = 0; i < 1000; ++i) energies[i] = std::pow(10.0, ((double)i / 10.0 - 69.95 + 0.691) / 10.0);
        for (int i = 1; i < 1001; ++i) bounds[i] = std::pow(10.0, ((double)i / 10.0 - 70.0 + 0.691) / 10.0);
        if (cudaMemcpyToSymbol(c_hist_bounds, bounds, sizeof bounds) != cudaSuccess ||
            cudaMemcpyToSymbol(c_hist_energy, energies, sizeof energies) != cudaSuccess)
            return bail(fail(AME_E_CUDA, "cudaMemcpyToSymbol failed: %s", cudaGetErrorString(cudaGetLastError())));
    }
    // allocations and clears are ordered on the default stream; the plan runs on others
    if (cudaError_t e = cudaStreamSynchronize(0); e != cudaSuccess)
        return bail(fail(AME_E_CUDA, "cudaStreamSynchronize failed: %s", cudaGetErrorString(e)));
    *out = p;
    return AME_OK;
}

int ame_release_cached_memory(int device) {
    GUARD(device);
    CU(cudaDeviceSynchronize());
    if (cudaMemPool_t pool = device_pool()) CU(cudaMemPoolTrimTo(pool, 0));
    return AME_OK;
}

int ame_plan_set_warm_luts(ame_plan *p, const float *luts, int32_t n_luts) {
    if (!p || !luts || n_luts <= 0) return fail(AME_E_INVALID, "bad warm lut arguments");
    GUARD(p->device);
    if (p->d_luts) {
        CU(cudaDeviceSynchronize());
        p->allocs.erase(std::find(p->allocs.begin(), p->allocs.end(), (void *)p->d_luts));
        dev_free(p->d_luts);
        p->d_luts = nullptr;
        p->ws_bytes -= (size_t)p->n_luts * 65536 * sizeof(double);
        p->n_luts = 0;
    }
    // widened exactly to double on the host so the kernel needs no float->double conversion per sample
    std::vector<double> wide((size_t)n_luts * 65536);
    for (size_t i = 0; i < wide.size(); ++i) wide[i] = (double)luts[i];
    int rc = dmalloc(p, (void **)&p->d_luts, wide.size() * sizeof(double));
    if (rc) return rc;
    CU(cudaMemcpy(p->d_luts, wide.data(), wide.size() * sizeof(double), cudaMemcpyHostToDevice));
    CU(cudaStreamSynchronize(0));
    p->n_luts = n_luts;
    return AME_OK;
}

int64_t ame_plan_total_frames(const ame_plan *p) { return p ? p->total_frames : 0; }
size_t ame_plan_workspace_bytes(const ame_plan *p) { return p ? p->ws_bytes : 0; }
int64_t ame_plan_launch_count(const ame_plan *p) { return p ? p->launches : 0; }
int32_t ame_plan_wave_count(const ame_plan *p) { return p ? (int32_t)p->waves.size() : 0; }
int32_t ame_plan_slot_count(const ame_plan *p) { return p ? (int32_t)p->slots.size() : 0; }
const int16_t *ame_plan_tap_pre(const ame_plan *p) { return (p && p->waves.size() == 1) ? p->slots[0].pre : nullptr; }
const int16_t *ame_plan_tap_bands(const ame_plan *p) { return (p && p->waves.size() == 1) ? p->slots[0].bands : nullptr; }
const double *ame_plan_tap_subblock_energy(const ame_plan *p) { return p ? p->d_energy : nullptr; }
int64_t ame_plan_mb_frames(const ame_plan *p) { return p ? p->mb_frames : 0; }
int64_t ame_plan_mb_offset(const ame_plan *p, int32_t t) { return (!p || t < 0 || t >= p->n_tracks) ? -1 : p->mb_offset[t]; }
int64_t ame_plan_subblock_offset(const ame_plan *p, int32_t t) { return (!p || t < 0 || t >= p->n_tracks) ? -1 : p->tdev[t].sb_offset; }

int ame_plan_read_device(ame_plan *p, void *h_dst, const void *d_src, size_t bytes) {
    if (!p || !h_dst || !d_src) return fail(AME_E_INVALID, "NULL argument");
    GUARD(p->device);
    CU(cudaDeviceSynchronize());
    CU(cudaMemcpy(h_dst, d_src, bytes, cudaMemcpyDeviceToHost));
    return AME_OK;
}

int ame_plan_chain_stats(ame_plan *p, int64_t *n_chains, int64_t *steps, int64_t *max_steps, int64_t *passes, int32_t *max_passes) {
    if (!p) return fail(AME_E_INVALID, "NULL plan");
    GUARD(p->device);
    CU(cudaDeviceSynchronize());
    int64_t nc = 0;
    for (const Wave &w : p->waves) nc += w.chain.n;
    std::vector<int> h((size_t)std::max<int64_t>(nc, 1) * 2, 0);
    if (nc) CU(cudaMemcpy(h.data(), p->d_chain_stats, (size_t)nc * 2 * sizeof(int), cudaMemcpyDeviceToHost));
    int64_t st = 0, mx = 0, ps = 0;
    int mp = 0;
    for (int64_t c = 0; c < nc; ++c) {
        st += h[2 * c]; mx = std::max<int64_t>(mx, h[2 * c]);
        ps += h[2 * c + 1]; mp = std::max(mp, h[2 * c + 1]);
    }
    if (n_chains) *n_chains = nc;
    if (steps) *steps = st;
    if (max_steps) *max_steps = mx;
    if (passes) *passes = ps;
    if (max_passes) *max_passes = mp;
    return AME_OK;
}

int ame_plan_limiter_stats(ame_plan *p, int64_t *open_tiles) {
    if (!p || !open_tiles) return fail(AME_E_INVALID, "NULL argument");
    GUARD(p->device);
    CU(cudaDeviceSynchronize());
    int h[4] = {0, 0, 0, 0};
    CU(cudaMemcpy(h, p->d_lim_stats, sizeof h, cudaMemcpyDeviceToHost));
    CU(cudaMemset(p->d_lim_stats, 0, sizeof h));
    for (int i = 0; i < 3; ++i) open_tiles[i] = h[i];
    return AME_OK;
}

int ame_plan_set_limiter_guess(ame_plan *p, int32_t frames) {
    if (!p) return fail(AME_E_INVALID, "NULL plan");
    if (frames < -1) return fail(AME_E_INVALID, "limiter guess of %d frames (-1 = the default 2 G, or >= 0)", frames);
    p->lim_guess = frames;
    return AME_OK;
}

int ame_plan_set_timing(ame_plan *p, int enable) {
    if (!p) return fail(AME_E_INVALID, "NULL plan");
    GUARD(p->device);
    if (enable && p->t_ev.empty()) {
        p->t_ev.resize((size_t)kMaxTimedSteps * kTimedSlots * 2);
        for (auto &e : p->t_ev) CU(cudaEventCreate(&e));
    }
    p->t_used.assign((size_t)kMaxTimedSteps * kTimedSlots, 0);
    p->t_step = -1;
    p->timing = enable != 0;
    return AME_OK;
}

int ame_plan_kernel_times(ame_plan *p, double *ms_sum, int64_t *launches, int *n_steps) {
    if (!p || !ms_sum || !launches) return fail(AME_E_INVALID, "NULL argument");
    GUARD(p->device);
    CU(cudaDeviceSynchronize());
    const int steps = std::min(p->t_step + 1, kMaxTimedSteps);
    for (int k = 0; k < AME_N_KERNELS; ++k) { ms_sum[k] = 0; launches[k] = 0; }
    for (size_t i = 0; i < (size_t)steps * kTimedSlots && !p->t_used.empty(); ++i)
        if (p->t_used[i]) {
            float ms = 0;
            CU(cudaEventElapsedTime(&ms, p->t_ev[i * 2], p->t_ev[i * 2 + 1]));
            ms_sum[i % AME_N_KERNELS] += ms;
            ++launches[i % AME_N_KERNELS];
        }
    if (n_steps) *n_steps = steps;
    return AME_OK;
}

int ame_plan_kernel_timeline(ame_plan *p, int step, float *ms, int max_waves) {
    if (!p || !ms) return fail(AME_E_INVALID, "NULL argument");
    GUARD(p->device);
    CU(cudaDeviceSynchronize());
    if (p->t_used.empty() || step < 0 || step > p->t_step || step >= kMaxTimedSteps) return fail(AME_E_INVALID, "step %d was not timed", step);
    const size_t base = (size_t)step * kMaxTimedWaves * AME_N_KERNELS;
    const int n = std::min(std::min((int)p->waves.size(), kMaxTimedWaves), max_waves);
    cudaEvent_t t0 = nullptr;                              // the first kernel of wave 0 opens the step
    for (int k = 0; k < AME_N_KERNELS && !t0; ++k)
        if (p->t_used[base + k]) t0 = p->t_ev[(base + k) * 2];
    if (!t0) return fail(AME_E_INVALID, "step %d was not timed", step);
    for (int w = 0; w < n; ++w)
        for (int k = 0; k < AME_N_KERNELS; ++k) {
            const size_t i = base + (size_t)w * AME_N_KERNELS + k;
            float *o = ms + ((size_t)w * AME_N_KERNELS + k) * 2;
            o[0] = o[1] = NAN;
            if (!p->t_used[i]) continue;
            CU(cudaEventElapsedTime(&o[0], t0, p->t_ev[i * 2]));
            CU(cudaEventElapsedTime(&o[1], t0, p->t_ev[i * 2 + 1]));
        }
    return n;
}

int ame_plan_wave_timeline(ame_plan *p, float *ms, int max_waves) {
    if (!p || !ms) return fail(AME_E_INVALID, "NULL argument");
    GUARD(p->device);
    CU(cudaDeviceSynchronize());
    const int n = std::min(p->tl_waves, max_waves);
    for (int w = 0; w < n; ++w)
        for (int k = 0; k < 4; ++k) CU(cudaEventElapsedTime(&ms[4 * w + k], p->tl_ev[0], p->tl_ev[1 + 4 * w + k]));
    return n;
}

// ---- stage entry points (one launch over the whole batch; plans with ONE wave) ----------------------
#define SINGLE_WAVE(p)                                                                             \
    if ((p)->waves.size() != 1) return fail(AME_E_INVALID, "the stage entry points need a plan with one wave (n_waves <= 1)")

int ame_stage_eq(ame_plan *p, const int16_t *d_in, int16_t *d_pre, void *stream) {
    if (!p || !d_in || !d_pre) return fail(AME_E_INVALID, "NULL argument");
    SINGLE_WAVE(p);
    GUARD(p->device);
    int rc = check_warmth(p);
    if (rc) return rc;
    return run_eq(p, p->waves[0], d_in, d_pre, (cudaStream_t)stream);
}

int ame_stage_band_split(ame_plan *p, const int16_t *d_pre, int16_t *d_bands, void *stream) {
    if (!p || !d_pre) return fail(AME_E_INVALID, "NULL argument");
    SINGLE_WAVE(p);
    GUARD(p->device);
    if (p->waves[0].split.n && !d_bands) return fail(AME_E_INVALID, "NULL bands buffer");
    return run_split(p, p->waves[0], d_pre, d_bands, (cudaStream_t)stream);
}

int ame_stage_compress(ame_plan *p, int16_t *d_bands, int16_t *d_pre, void *stream) {
    if (!p || !d_pre) return fail(AME_E_INVALID, "NULL argument");
    SINGLE_WAVE(p);
    GUARD(p->device);
    if (p->waves[0].chain.n && !d_bands) return fail(AME_E_INVALID, "NULL bands buffer");
    Bufs b = slot_bufs(p, p->waves[0], nullptr, nullptr);
    b.bands = d_bands;
    b.pre = d_pre;
    return run_compress(p, p->waves[0], b, (cudaStream_t)stream);
}

int ame_stage_loudness_hist(ame_plan *p, const int16_t *d_pre, int64_t *d_hist, void *stream) {
    if (!p || !d_pre || !d_hist) return fail(AME_E_INVALID, "NULL argument");
    SINGLE_WAVE(p);
    GUARD(p->device);
    return run_hist(p, p->waves[0], d_pre, d_hist, (cudaStream_t)stream);
}

int ame_stage_apply_gain(ame_plan *p, const int16_t *d_pre, const int64_t *d_hist, int16_t *d_out,
                         ame_track_result *results, void *stream) {
    if (!p || !d_pre || !d_hist || !d_out) return fail(AME_E_INVALID, "NULL argument");
    SINGLE_WAVE(p);
    GUARD(p->device);
    cudaStream_t s = (cudaStream_t)stream;
    const Bufs sb = slot_bufs(p, p->waves[0], nullptr, d_out);
    int rc = run_gain(p, p->waves[0], d_pre, d_hist, d_out, sb, s);
    if (rc) return rc;
    if (results) {
        CU(cudaMemcpyAsync(results, p->d_results, (size_t)p->n_tracks * sizeof(ame_track_result), cudaMemcpyDeviceToHost, s));
        CU(cudaStreamSynchronize(s));
    }
    return AME_OK;
}

// ffmpeg alimiter alone (:223) on an int16 signal that is already normalised: the results are cleared, so that
// k_apply_gain passes the samples through unchanged on its way to the limiter's input buffer
int ame_stage_limiter(ame_plan *p, const int16_t *d_norm, int16_t *d_out, void *stream) {
    if (!p || !d_norm || !d_out) return fail(AME_E_INVALID, "NULL argument");
    SINGLE_WAVE(p);
    GUARD(p->device);
    for (int t = 0; t < p->n_tracks; ++t)
        if (!(p->tracks[t].flags & AME_F_LIMITER)) return fail(AME_E_INVALID, "track %d has no limiter stage (AME_F_LIMITER)", t);
    cudaStream_t s = (cudaStream_t)stream;
    CU(cudaMemsetAsync(p->d_results, 0, (size_t)p->n_tracks * sizeof(ame_track_result), s));
    const Bufs sb = slot_bufs(p, p->waves[0], nullptr, d_out);
    return run_apply(p, p->waves[0], d_norm, d_out, sb, s);
}

// two-phase form: every wave must keep its pre-normalisation signal between the two calls (n_slots == n_waves)
int ame_measure_device(ame_plan *p, const int16_t *d_in, int64_t *d_hist, void *stream) {
    if (!p || !d_in || !d_hist) return fail(AME_E_INVALID, "NULL argument");
    if (p->slots.size() != p->waves.size()) return fail(AME_E_INVALID, "the two-phase calls need n_slots == n_waves");
    GUARD(p->device);
    int rc = check_warmth(p);
    if (rc) return rc;
    p->launches = 0;
    if (p->timing) ++p->t_step;
    for (size_t w = 0; w < p->waves.size(); ++w) {
        p->t_wave = (int)std::min<size_t>(w, kMaxTimedWaves - 1);
        Bufs b = slot_bufs(p, p->waves[w], d_in, nullptr);
        b.hist = d_hist;
        if ((rc = run_measure(p, p->waves[w], b, (cudaStream_t)stream))) return rc;
    }
    return AME_OK;
}

int ame_normalize_device(ame_plan *p, const int64_t *d_hist, int16_t *d_out, ame_track_result *results, void *stream) {
    if (!p || !d_hist || !d_out) return fail(AME_E_INVALID, "NULL argument");
    if (p->slots.size() != p->waves.size()) return fail(AME_E_INVALID, "the two-phase calls need n_slots == n_waves");
    GUARD(p->device);
    cudaStream_t s = (cudaStream_t)stream;
    int rc;
    for (size_t w = 0; w < p->waves.size(); ++w) {
        p->t_wave = (int)std::min<size_t>(w, kMaxTimedWaves - 1);
        const Bufs b = slot_bufs(p, p->waves[w], nullptr, d_out);
        if ((rc = run_gain(p, p->waves[w], b.pre, d_hist, d_out, b, s))) return rc;
        if ((rc = run_meter(p, p->waves[w], d_out, p->d_loud_out, s))) return rc;
    }
    if (results) {
        CU(cudaMemcpyAsync(results, p->d_results, (size_t)p->n_tracks * sizeof(ame_track_result), cudaMemcpyDeviceToHost, s));
        CU(cudaStreamSynchronize(s));
    }
    return AME_OK;
}

// ---- by-time sharding without Python: the two messages of the path over NCCL -------------------------------------
// libame does not link NCCL: the entry points are resolved at run time from the libnccl the host process already
// uses (dlopen with RTLD_NOLOAD first), so the library still loads where there is no NCCL at all.
namespace {
typedef int (*nccl_allreduce_t)(const void *, void *, size_t, int, int, void *, cudaStream_t);
typedef int (*nccl_sendrecv_t)(void *, size_t, int, int, void *, cudaStream_t);
typedef int (*nccl_group_t)(void);
typedef const char *(*nccl_errstr_t)(int);
struct NcclApi {
    nccl_allreduce_t all_reduce = nullptr;
    nccl_sendrecv_t send = nullptr, recv = nullptr;
    nccl_group_t group_start = nullptr, group_end = nullptr;
    nccl_errstr_t err = nullptr;
    bool tried = false, ok = false;
};
NcclApi g_nccl;
std::mutex g_nccl_mutex;
constexpr int kNcclInt8 = 0, kNcclInt64 = 4, kNcclSum = 0;     // ncclDataType_t / ncclRedOp_t values (nccl.h, stable since 2.0)

const NcclApi *nccl_api() {
    std::lock_guard<std::mutex> lock(g_nccl_mutex);
    if (!g_nccl.tried) {
        g_nccl.tried = true;
        void *h = nullptr;
        for (const char *name : {"libnccl.so.2", "libnccl.so"}) {
            h = dlopen(name, RTLD_NOW | RTLD_NOLOAD);
            if (!h) h = dlopen(name, RTLD_NOW | RTLD_GLOBAL);
            if (h) break;
        }
        if (h) {
            g_nccl.all_reduce = (nccl_allreduce_t)dlsym(h, "ncclAllReduce");
            g_nccl.send = (nccl_sendrecv_t)dlsym(h, "ncclSend");
            g_nccl.recv = (nccl_sendrecv_t)dlsym(h, "ncclRecv");
            g_nccl.group_start = (nccl_group_t)dlsym(h, "ncclGroupStart");
            g_nccl.group_end = (nccl_group_t)dlsym(h, "ncclGroupEnd");
            g_nccl.err = (nccl_errstr_t)dlsym(h, "ncclGetErrorString");
            g_nccl.ok = g_nccl.all_reduce && g_nccl.send && g_nccl.recv && g_nccl.group_start && g_nccl.group_end;
        }
    }
    return g_nccl.ok ? &g_nccl : nullptr;
}
#define NCCL(api, call)                                                                            \
    do {                                                                                           \
        int r_ = (call);                                                                           \
        if (r_ != 0) return fail(AME_E_CUDA, "%s failed: %s", #call, (api)->err ? (api)->err(r_) : "NCCL error"); \
    } while (0)
}  // namespace

int ame_hist_allreduce(ame_plan *p, int64_t *d_hist, void *nccl_comm, void *stream) {
    if (!p || !d_hist || !nccl_comm) return fail(AME_E_INVALID, "NULL argument");
    const NcclApi *api = nccl_api();
    if (!api) return fail(AME_E_UNSUPPORTED, "libnccl.so.2 not found in this process");
    GUARD(p->device);
    NCCL(api, api->all_reduce(d_hist, d_hist, (size_t)p->n_tracks * 1000, kNcclInt64, kNcclSum, nccl_comm, (cudaStream_t)stream));
    return AME_OK;
}

int ame_shard_halo_exchange(ame_plan *p, int16_t *d_pre, void *nccl_comm, int prev_rank, int next_rank, int64_t send_frames,
                            void *stream) {
    if (!p || !d_pre || !nccl_comm) return fail(AME_E_INVALID, "NULL argument");
    if (p->n_tracks != 1) return fail(AME_E_INVALID, "a time shard is a plan over one track");
    const ame_track_params &tp = p->tracks[0];
    const int64_t have = tp.halo_frames + tp.n_frames;
    if (next_rank >= 0 && (send_frames <= 0 || send_frames > have))
        return fail(AME_E_UNSUPPORTED, "the shard holds %lld frames, fewer than the %lld the next shard's halo needs", (long long)have,
                    (long long)send_frames);
    const NcclApi *api = nccl_api();
    if (!api) return fail(AME_E_UNSUPPORTED, "libnccl.so.2 not found in this process");
    GUARD(p->device);
    int16_t *base = d_pre + 2 * tp.offset_frames;
    NCCL(api, api->group_start());
    if (next_rank >= 0)
        NCCL(api, api->send(base + 2 * (have - send_frames), (size_t)send_frames * 4, kNcclInt8, next_rank, nccl_comm, (cudaStream_t)stream));
    if (prev_rank >= 0 && tp.halo_frames > 0)
        NCCL(api, api->recv(base, (size_t)tp.halo_frames * 4, kNcclInt8, prev_rank, nccl_comm, (cudaStream_t)stream));
    NCCL(api, api->group_end());
    return AME_OK;
}

int ame_master_device(ame_plan *p, const int16_t *d_in, int16_t *d_out, ame_track_result *results, void *stream) {
    if (!p) return fail(AME_E_INVALID, "NULL plan");
    if (!d_in || !d_out) return fail(AME_E_INVALID, "NULL argument");
    GUARD(p->device);
    int rc = check_warmth(p);
    if (rc) return rc;
    cudaStream_t s = (cudaStream_t)stream;
    const int nw = (int)p->waves.size();
    p->launches = 0;
    if (p->timing) ++p->t_step;
    if (nw <= 1) {
        p->t_wave = 0;
        if ((rc = run_chain_of_stages(p, p->waves[0], slot_bufs(p, p->waves[0], d_in, d_out), s))) return rc;
        if ((rc = run_meter(p, p->waves[0], d_out, p->d_loud_out, s))) return rc;
    } else {
        // several waves: fork the caller's stream into the slots' streams and join again.  Waves of different slots
        // overlap (the latency-bound compressor kernels of one under the FP64-bound filters of another); waves of
        // one slot follow each other in stream order, which is what recycles the slot.
        CU(cudaEventRecord(p->ev_in[0], s));
        const int ns = (int)p->slots.size();
        for (int w = 0; w < nw; ++w) {
            cudaStream_t ws = p->slots[p->waves[w].slot].stream;
            if (w < ns) CU(cudaStreamWaitEvent(ws, p->ev_in[0], 0));
            p->t_wave = std::min(w, kMaxTimedWaves - 1);
            if ((rc = run_chain_of_stages(p, p->waves[w], slot_bufs(p, p->waves[w], d_in, d_out), ws))) return drain(p, rc);
            if ((rc = run_meter(p, p->waves[w], d_out, p->d_loud_out, ws))) return drain(p, rc);
        }
        for (int k = 0; k < ns; ++k) {
            CU(cudaEventRecord(p->ev_run[k], p->slots[k].stream));
            CU(cudaStreamWaitEvent(s, p->ev_run[k], 0));
        }
    }
    if (results) {
        CU(cudaMemcpyAsync(results, p->d_results, (size_t)p->n_tracks * sizeof(ame_track_result), cudaMemcpyDeviceToHost, s));
        CU(cudaStreamSynchronize(s));
    }
    return AME_OK;
}

// Host buffers: wave w's H2D copy (stream s_in), kernels (its slot's stream) and D2H copy (s_out) are chained by
// events, so the copy engines (PCIe is full duplex) and the SMs work on different waves at the same time.  Pinned host
// memory makes the copies truly asynchronous; pageable memory still works, the copies then serialise.
static int master_host_impl(ame_plan *p, const int16_t *h_in, int16_t *h_out, ame_track_result *results) {
    int rc = check_warmth(p);
    if (rc) return rc;
    p->launches = 0;
    if (p->timing) ++p->t_step;
    const int nw = (int)p->waves.size();
    const bool tl = p->timing;
    if (tl) {
        while ((int)p->tl_ev.size() < 1 + 4 * nw) {
            cudaEvent_t e;
            CU(cudaEventCreate(&e));
            p->tl_ev.push_back(e);
        }
        p->tl_waves = nw;
        CU(cudaEventRecord(p->tl_ev[0], p->s_in));
    }
    for (int w = 0; w < nw; ++w) {
        const Wave &wv = p->waves[w];
        const size_t off = (size_t)wv.frame_lo * 4, bytes = (size_t)(wv.frame_hi - wv.frame_lo) * 4;
        CU(cudaMemcpyAsync((char *)p->d_in + off, (const char *)h_in + off, bytes, cudaMemcpyHostToDevice, p->s_in));
        CU(cudaEventRecord(p->ev_in[w], p->s_in));
        if (tl) CU(cudaEventRecord(p->tl_ev[1 + 4 * w], p->s_in));
    }
    for (int w = 0; w < nw; ++w) {
        cudaStream_t ws = p->slots[p->waves[w].slot].stream;
        CU(cudaStreamWaitEvent(ws, p->ev_in[w], 0));
        if (tl) CU(cudaEventRecord(p->tl_ev[2 + 4 * w], ws));
        p->t_wave = std::min(w, kMaxTimedWaves - 1);
        if ((rc = run_chain_of_stages(p, p->waves[w], slot_bufs(p, p->waves[w], p->d_in, p->d_out), ws))) return rc;
        CU(cudaEventRecord(p->ev_run[w], ws));
        if (tl) CU(cudaEventRecord(p->tl_ev[3 + 4 * w], ws));
        // the meter reads d_out after ev_run[w]: the wave's D2H copy waits for its kernels, not for its meter
        if ((rc = run_meter(p, p->waves[w], p->d_out, p->d_loud_out, ws))) return rc;
    }
    for (int w = 0; w < nw; ++w) {
        const Wave &wv = p->waves[w];
        const size_t off = (size_t)wv.frame_lo * 4, bytes = (size_t)(wv.frame_hi - wv.frame_lo) * 4;
        CU(cudaStreamWaitEvent(p->s_out, p->ev_run[w], 0));
        CU(cudaMemcpyAsync((char *)h_out + off, (const char *)p->d_out + off, bytes, cudaMemcpyDeviceToHost, p->s_out));
        if (tl) CU(cudaEventRecord(p->tl_ev[4 + 4 * w], p->s_out));
    }
    if (results)
        CU(cudaMemcpyAsync(results, p->d_results, (size_t)p->n_tracks * sizeof(ame_track_result), cudaMemcpyDeviceToHost, p->s_out));
    // only now, behind every copy, s_out waits for the meters of all slots: the synchronisation below covers them
    if (p->any_meter)
        for (size_t k = 0; k < p->slots.size(); ++k) {
            CU(cudaEventRecord(p->ev_meter[k], p->slots[k].stream));
            CU(cudaStreamWaitEvent(p->s_out, p->ev_meter[k], 0));
        }
    CU(cudaStreamSynchronize(p->s_out));
    return AME_OK;
}

int ame_plan_output_loudness(ame_plan *p, ame_loudness *out, void *stream) {
    if (!p || !out) return fail(AME_E_INVALID, "NULL argument");
    GUARD(p->device);
    if (!p->any_meter) {                               // nothing is ever measured
        std::memset(out, 0, (size_t)p->n_tracks * sizeof(ame_loudness));
        return AME_OK;
    }
    cudaStream_t s = (cudaStream_t)stream;
    CU(cudaMemcpyAsync(out, p->d_loud_out, (size_t)p->n_tracks * sizeof(ame_loudness), cudaMemcpyDeviceToHost, s));
    CU(cudaStreamSynchronize(s));
    return AME_OK;
}

int ame_measure_loudness(ame_plan *p, const int16_t *d_buf, ame_loudness *out, void *stream) {
    if (!p || !d_buf) return fail(AME_E_INVALID, "NULL argument");
    if (!p->any_meter) return fail(AME_E_INVALID, "no track carries AME_F_MEASURE_OUTPUT");
    GUARD(p->device);
    cudaStream_t s = (cudaStream_t)stream;
    p->launches = 0;
    CU(cudaMemsetAsync(p->d_loud_any, 0, (size_t)p->n_tracks * sizeof(ame_loudness), s));
    int rc;
    for (const Wave &w : p->waves)
        if ((rc = run_meter(p, w, d_buf, p->d_loud_any, s))) return rc;
    if (out) {
        CU(cudaMemcpyAsync(out, p->d_loud_any, (size_t)p->n_tracks * sizeof(ame_loudness), cudaMemcpyDeviceToHost, s));
        CU(cudaStreamSynchronize(s));
    }
    return AME_OK;
}

int ame_master_host(ame_plan *p, const int16_t *h_in, int16_t *h_out, ame_track_result *results) {
    if (!p || !h_in || !h_out) return fail(AME_E_INVALID, "NULL argument");
    if (!p->d_in || !p->d_out) return fail(AME_E_INVALID, "plan was created without host_io");
    GUARD(p->device);
    // whatever fails in the middle: no copy or kernel may still touch h_in / h_out once we have returned
    return drain(p, master_host_impl(p, h_in, h_out, results));
}

}  // extern "C"
