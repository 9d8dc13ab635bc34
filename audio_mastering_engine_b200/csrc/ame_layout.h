// Plan layout of libame: how a batch of tracks is packed, split into waves and cut into the job tables of every kernel.
// Plain host arithmetic on the track parameters, the plan options and the shape of the device - no CUDA here, so the
// layout builds and is tested without a GPU (tests/test_plan_layout.py).  The job structs are shared with the kernels.
#pragma once
#include <stdint.h>

#include <algorithm>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <map>
#include <string>
#include <tuple>
#include <utility>
#include <vector>

#include "../../include/ame.h"

namespace ame {

constexpr int kGainTile = 32768;   // frames per CTA in k_apply_gain / k_band_sum

struct TileJob {           // one lane pair of k_eq / k_band_split
    int64_t chunk_begin;   // absolute frame index (packed buffer) where filter state is reset
    int64_t tile_begin;    // first frame this job writes (absolute, multiple of 4 unless == chunk_begin)
    int64_t tile_end;      // one past the last frame it writes
    int32_t track;
    int32_t variant;       // EQ stage mask (bit s = stage s active)
};

struct ChainJob {          // one warp of k_compress: one band of one chunk of a multiband track
    int64_t mb_begin;      // of the chunk, in the multiband-only packing (bands planes)
    int64_t n;             // frames
    int64_t grp_begin;     // first slot of this chain in the per-group record array
    int32_t band;
    int32_t table;
    uint32_t thr_i;        // rms > thresh_rms  <=>  rms >= thr_i
    int32_t look;          // look_frames
    int32_t tile0;         // index (within the wave's launch) of the chain's first k_window_flag / k_compact tile
    int32_t pad;
};

struct KwJob { int32_t track; int32_t sb_begin; int32_t sb_end; int32_t pad; };

struct GainJob { int64_t begin; int64_t end; int32_t track; int32_t pad; };

// indexed by integer rms 0..32768.  tau = the smallest attenuation a with fl(a + inc) >= m, so that
// (att + inc < m) <=> (att < tau) exactly and the branch predicates depend on the OLD attenuation only.
struct AttEntry { double m, inc, dec, tau; };

struct TrackDev {          // device-side per-track bookkeeping
    int64_t sb_offset;     // start of this track's 100 ms energies in the energy array
    int32_t n_sb;          // number of complete 100 ms sub-blocks (halo included)
    int32_t s100;          // frames per 100 ms = (fs + 5) / 10   (ebur128.c)
    int32_t first_block;   // time shards: 400 ms blocks before this one belong to the previous shard / the warm-up
    int32_t lim_tile0;     // limiter: index (within the wave's launch) of the track's first limiter tile
    int64_t n_total;       // halo + span frames
    int32_t lim_shift;     // limiter: log2 of the track's limiter tile length (a power of two >= G)
    int32_t pad;
};

struct XoverCfg { double lb0, la10, la20, la11, la21, hb0, ha10, ha20, ha11, ha21; };

constexpr int kWfThreads = 256;
constexpr int kWfTile = 2048;      // frames per CTA of k_window_flag / k_compact (8 per thread)
constexpr int kSeg = 256;          // frames per k_att_chain iteration / per k_compress_apply warp (8 groups)

// One tile of a chain for k_window_flag / k_compact.  It carries what the kernels need of its chain, so a CTA (which
// lives for a few microseconds) starts with ONE dependent load instead of job -> chain -> data.
struct WfJob {
    int64_t tile_begin;    // relative to the chunk
    int64_t plane_off;     // band * mb_frames + mb_begin: offset of the chain in the bands / rms / list planes (frames)
    int64_t n;             // frames of the chain
    int64_t grp_begin;     // first group record of the chain
    int32_t chain;         // index into the plan's chain table
    int32_t look;          // look_frames
    uint32_t thr_i;        // rms > thresh_rms  <=>  rms >= thr_i
    int32_t tile0;         // index (within the launch) of the chain's first tile
};

struct MbChunk {           // one chunk of a multiband track (k_compress_apply)
    int64_t abs_begin;     // absolute frame index in the packed pre buffer
    int64_t mb_begin;      // frame index in the multiband-only packing
    int64_t n;             // frames
    int64_t seg_prefix;    // kSeg-segments in all earlier chunks
    int64_t grp_begin[3];  // first group record of each band's chain
    int32_t track;
    int32_t pad;
};

struct GrpRec { uint32_t mask, base; };   // per 32-frame group of a chain: flagged frames, flagged frames before the group

constexpr int kChainMaxThreads = 256;

struct KwCfg { double b0, b1, b2, a1, a2, ra1, ra2; };   // pre-filter biquad; RLB denominators (numerator 1 -2 1)

constexpr int kLimQueue = 1024;     // largest queue capacity (look-ahead B <= 1000 frames is validated by the host)
constexpr int kLimMaxTile = 1 << 20;     // longest limiter tile (look-ahead + release of the slowest setting must fit one)

// ---- layout -----------------------------------------------------------------------------------------------------

inline int64_t align_up(int64_t v, int64_t a) { return (v + a - 1) / a * a; }

// formats a message into `err` and returns `code`
inline int layout_fail(std::string &err, int code, const char *fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    err = buf;
    return code;
}

struct JobRange { int lo = 0, n = 0; };   // jobs [lo, lo + n) of one job table

// A wave = a contiguous range of tracks whose jobs are contiguous in every job table.  The device path
// launches each kernel ONCE over all waves; the host path (ame_master_host) launches wave by wave so the
// H2D copy of wave w+1 and the D2H copy of wave w-1 overlap the kernels of wave w.
struct Wave {
    int track_lo = 0, track_hi = 0;
    int64_t frame_lo = 0, frame_hi = 0;            // packed-buffer range (multiples of 8 frames)
    JobRange eq, split, chain, wf, mb_chunks, kw, gain, lim;   // of the job table of the same name
    JobRange meter_kw, meter_peak, meter_tracks;   // the output meter's tables (tracks with AME_F_MEASURE_OUTPUT only)
    int64_t seg_lo = 0, seg_hi = 0;
    int slot = 0;                                  // workspace slot (and stream) this wave runs in
    bool limiter = false;                          // a track of the wave has the limiter stage
    bool true_peak = false;                        // a track of the wave wants its oversampled peak
    bool xover_uni = false, kw_uni = false;        // all multiband tracks share the crossover / all k_kweight_energy tracks the K filter
    XoverCfg xover{};
    KwCfg kw_cfg{};
};

// What a plan keeps of its layout.
struct Layout {
    std::vector<ame_track_params> tracks;   // the caller's, with comp[b].table filled in
    std::vector<int64_t> mb_offset;         // per track, -1 if not multiband
    std::vector<TrackDev> tdev;
    std::vector<Wave> waves;
    int n_slots = 0;
    int64_t total_frames = 0;               // padded
    int64_t mb_frames = 0;                  // padded; the largest wave's multiband packing = plane stride of every slot
    int64_t slot_frames = 0, slot_groups = 0;
    int slot_tiles = 0, slot_chains = 0, slot_lim_jobs = 0;
    int64_t n_sb_total = 0;
    int split_tile = 0, kw_tile_sb = 0;
    int lim_keep = 2;                       // queue entries a recorded limiter state holds: look-ahead frames + 2
    bool any_limiter = false, any_tp = false;
    bool any_meter = false;                 // a track carries AME_F_MEASURE_OUTPUT
    std::vector<TrackDev> meter_tdev;       // tdev with sb_offset into the meter's own sub-block energies (flagged tracks)
    int64_t meter_sb_total = 0;             // sub-blocks of the flagged tracks
};

// The tables a plan uploads once.  Every job table is ordered by track, hence contiguous per wave.
struct JobTables {
    std::vector<int64_t> mb_delta;          // per track: multiband packing offset - packed-buffer offset
    std::vector<TileJob> eq, split;
    std::vector<ChainJob> chain;
    std::vector<WfJob> wf;
    std::vector<MbChunk> mb_chunks;
    std::vector<KwJob> kw;
    std::vector<GainJob> gain, lim;         // limiter tiles: the same (begin, end, track) records, shorter tiles
    std::vector<AttEntry> att;              // 32769 entries per distinct compressor band
    // output meter, flagged tracks only: K-weighting tiles (kw_tile_sb sub-blocks, as kw), peak tiles (the gain tiles)
    // and the list of flagged tracks
    std::vector<KwJob> meter_kw;
    std::vector<GainJob> meter_peak;
    std::vector<int32_t> meter_tracks;
};

struct DeviceShape {
    int n_sm;                               // multiprocessors
    int occ_eq, occ_split;                  // resident 128-thread CTAs per SM of k_eq and of k_band_split
};

// split chunk [cb, ce) into ceil(n / T) near-equal tiles whose interior boundaries are multiples of 8
inline void tile_jobs(std::vector<TileJob> &out, int track, int variant, int64_t cb, int64_t ce, int64_t T) {
    const int64_t n = ce - cb;
    if (n <= 0) return;
    const int64_t k = (n + T - 1) / T;
    const int64_t t = align_up((n + k - 1) / k, 8);
    int64_t b = cb;
    while (b < ce) {
        int64_t e = (b + t) & ~(int64_t)7;
        if (e <= b) e = b + t;
        if (e > ce) e = ce;
        out.push_back(TileJob{cb, b, e, track, variant});
        b = e;
    }
}

// smallest tile (multiple of 8, >= min_tile) whose job count fits `slots` threads
inline int64_t pick_tile(const std::vector<int64_t> &chunks, int64_t slots, int64_t min_tile) {
    auto count = [&](int64_t T) {
        int64_t jobs = 0;
        for (int64_t n : chunks) jobs += (n + T - 1) / T;
        return jobs;
    };
    int64_t lo = min_tile, hi = min_tile;
    for (int64_t n : chunks) hi = std::max(hi, align_up(n, 8));
    if (count(lo) <= slots) return lo;
    while (lo < hi) {                    // count() is non-increasing in T
        const int64_t mid = align_up((lo + hi) / 2, 8);
        if (mid >= hi) break;
        if (count(mid) <= slots) hi = mid; else lo = mid + 8;
    }
    return hi;
}

// k_eq tiles are cost-balanced: a thread's work is about (tile + warm-up) * cost-per-frame, and the cost per
// frame differs a lot between tracks (no EQ at all ... 4 stages + warmth).  Give every track the tile length
// that makes (T + warm) * cost equal to one common budget, the smallest budget whose job count fits `slots`.
inline double eq_cost_per_frame(const ame_track_params &t) {
    // relative cost of one frame in each k_eq variant, fitted to launches of 96 identical tracks per variant
    // (profiles/r02/eq_variant_cost.txt, warm-up overlap taken out): 4 stages = 128, 2 shelves + 1 peak = 91, one peak 57,
    // two shelves 58, no EQ 47 (bound by its loads, not by arithmetic); warmth + 26 (+ 20 without EQ); width is free
    double c = 24.0;                                    // unpack, convert, pack, store
    if (t.eq[0].kind != AME_EQ_BYPASS) c += 16.0;       // one section + blend, two channels
    if (t.eq[1].kind != AME_EQ_BYPASS) c += 36.0;       // four sections + blend, two channels
    if (t.eq[2].kind != AME_EQ_BYPASS) c += 36.0;
    if (t.eq[3].kind != AME_EQ_BYPASS) c += 16.0;
    const bool warm = (t.flags & AME_F_WARMTH) != 0;
    if (c == 24.0) return warm ? 67.0 : 47.0;
    return c + (warm ? 26.0 : 0.0);                     // two table look-ups + the 2x2 mix in explicit FP64 ops
}

// k_eq runs one thread per tile and switches on the track's variant, so a warp that mixes VARIANTS would run
// both one after the other; tracks of the same variant can share a warp (coefficients are per-thread registers).
// Every track gets a number of jobs (threads) in proportion to its cost (frames x cost per frame); the jobs of a
// wave are then laid out variant by variant and only the end of each variant's run is padded to a whole warp.
// (Until late in round 2 every track got whole WARPS: with ~9 warps per track the rounding left the cheapest
// tracks of a 128-track launch with 14 % more work per thread than the mean, and the launch ended with them.)
inline int eq_variant_of(const ame_track_params &t) {
    int variant = 0;
    for (int s = 0; s < 4; ++s)
        if (t.eq[s].kind != AME_EQ_BYPASS) variant |= 1 << s;
    if (t.flags & AME_F_WARMTH) variant |= 16;
    return variant;
}

// Threads handed out = the resident set minus the padding at the end of every variant's run (a warp).  Padding the runs to
// whole 8-warp CTAs (no CTA would mix two variants) was measured too: 9.84 ms against 9.69 ms on the 128-track launch -
// the ~4 % of idle threads cost more than the ~12 mixed CTAs.
inline std::vector<int64_t> eq_jobs_per_track(const ame_track_params *tracks, const std::vector<std::vector<int64_t>> &chunks,
                                              const std::vector<double> &cost, int t_lo, int t_hi, int64_t slots, int64_t min_tile) {
    const int n = (int)chunks.size();
    std::vector<int64_t> jobs(n, 0), cap(n, 0), floor_jobs(n, 0);
    std::vector<double> weight(n, 0.0);
    double wsum = 0;
    unsigned variants = 0;
    int n_variants = 0;
    for (int t = t_lo; t < t_hi; ++t) {
        int64_t frames = 0, max_jobs = 0;
        for (int64_t c : chunks[t]) { frames += c; max_jobs += std::max<int64_t>(1, c / min_tile); }
        weight[t] = (double)frames * cost[t];
        cap[t] = std::max<int64_t>(1, max_jobs);
        floor_jobs[t] = std::max<int64_t>(1, (int64_t)chunks[t].size());      // tile_jobs makes one job per chunk at least
        wsum += weight[t];
        const unsigned bit = 1u << eq_variant_of(tracks[t]);
        if (!(variants & bit)) { variants |= bit; ++n_variants; }
    }
    const int64_t avail = std::max<int64_t>(32 * (int64_t)(t_hi - t_lo), slots) - 31 * (int64_t)n_variants;
    std::vector<std::pair<double, int>> rem;
    int64_t used = 0;
    for (int t = t_lo; t < t_hi; ++t) {
        const double share = wsum > 0 ? (double)avail * weight[t] / wsum : 32.0;
        jobs[t] = std::min(cap[t], std::max(floor_jobs[t], (int64_t)share));
        used += jobs[t];
        rem.emplace_back(share - (double)jobs[t], t);
    }
    std::sort(rem.begin(), rem.end(), [](const std::pair<double, int> &a, const std::pair<double, int> &b) { return a.first > b.first; });
    for (size_t i = 0; i < rem.size() && used < avail; ++i)
        if (jobs[rem[i].second] < cap[rem[i].second]) { ++jobs[rem[i].second]; ++used; }
    return jobs;
}

inline int validate(const ame_track_params &t, int idx, std::string &err) {
    if (t.n_frames < 0 || t.offset_frames < 0 || (t.offset_frames & 7))
        return layout_fail(err, AME_E_INVALID, "track %d: offset_frames must be a non-negative multiple of 8", idx);
    if (t.sample_rate < 8000 || t.sample_rate > 384000)
        return layout_fail(err, AME_E_INVALID, "track %d: unsupported sample rate %d", idx, t.sample_rate);
    if (t.halo_frames < 0 || (t.halo_frames & 7) || t.halo_frames % ((t.sample_rate + 5) / 10))
        return layout_fail(err, AME_E_INVALID, "track %d: halo_frames must be a multiple of 8 and of the 100 ms sub-block", idx);
    if (t.warm_eq < 0 || t.warm_xover < 0 || t.warm_kw < 0)
        return layout_fail(err, AME_E_INVALID, "track %d: negative warm-up", idx);
    if (t.flags & AME_F_LIMITER) {
        if (t.halo_frames)
            return layout_fail(err, AME_E_UNSUPPORTED, "track %d: the limiter is one sequential state machine over the whole track "
                                                       "and cannot run on a time shard; limit the gathered output instead", idx);
        if (t.lim_frames < 1 || t.lim_frames > kLimQueue - 24 || !(t.lim_limit > 0.0 && t.lim_limit <= 1.0) || !(t.lim_fs_release > 0.0) ||
            t.lim_release_frames < 1 || t.lim_frames + t.lim_release_frames + 8 > kLimMaxTile || t.lim_thr_i < 1)
            return layout_fail(err, AME_E_INVALID, "track %d: bad limiter parameters (look-ahead %d frames, release %d frames)", idx,
                               t.lim_frames, t.lim_release_frames);
    }
    if ((t.flags & AME_F_MEASURE_OUTPUT) && t.halo_frames)
        return layout_fail(err, AME_E_UNSUPPORTED, "track %d: the output meter measures a whole track and cannot run on a time "
                                                   "shard; measure the gathered output instead", idx);
    for (int s = 0; s < 4; ++s) {
        const int k = t.eq[s].kind;
        const bool shelf = (s == 0 || s == 3);
        if (k == AME_EQ_BYPASS) continue;
        if (shelf ? (k != AME_EQ_SHELF_BOOST && k != AME_EQ_SHELF_CUT) : (k != AME_EQ_PEAK))
            return layout_fail(err, AME_E_INVALID, "track %d: eq stage %d has kind %d", idx, s, k);
    }
    // the kernels rely on the Butterworth numerator shape b0 * (1 +- 2 z^-1 + z^-2) that scipy.signal.butter
    // produces for every filter of the reference (sign pattern and unit-gain sections are fixed by design)
    auto shape = [&](const ame_biquad &q, double sgn, bool unit) {
        return q.b1 == sgn * 2.0 * q.b0 && q.b2 == q.b0 && (!unit || q.b0 == 1.0);
    };
    bool ok = true;
    if (t.eq[0].kind != AME_EQ_BYPASS) ok = ok && shape(t.eq[0].s[0], 1, false);
    if (t.eq[3].kind != AME_EQ_BYPASS) ok = ok && shape(t.eq[3].s[0], -1, false);
    for (int s = 1; s <= 2; ++s)
        if (t.eq[s].kind != AME_EQ_BYPASS)
            ok = ok && shape(t.eq[s].s[0], 1, false) && shape(t.eq[s].s[1], 1, true) && shape(t.eq[s].s[2], -1, true) &&
                 shape(t.eq[s].s[3], -1, true);
    if (t.flags & AME_F_MULTIBAND)
        ok = ok && shape(t.xlp[0], 1, false) && shape(t.xlp[1], 1, true) && shape(t.xhp[0], -1, false) && shape(t.xhp[1], -1, true);
    if (!ok) return layout_fail(err, AME_E_UNSUPPORTED, "track %d: a filter section is not of Butterworth shape b0*(1 +- 2z^-1 + z^-2)", idx);
    if (t.flags & AME_F_MULTIBAND)
        for (int b = 0; b < 3; ++b) {
            const ame_comp_band &c = t.comp[b];
            if (!(c.thresh_rms >= 0) || !(c.attack_frames > 0) || !(c.release_frames > 0) || c.look_frames < 0 ||
                c.look_frames > 4096)
                return layout_fail(err, AME_E_INVALID, "track %d: bad compressor band %d", idx, b);
            // ratio < 1 makes max_attenuation negative: k_att_chain orders attenuations by their bit patterns and shifts
            // parked segments by whole ulps, which holds for non-negative operands only
            if (!(c.coef >= 0))
                return layout_fail(err, AME_E_UNSUPPORTED, "track %d: compressor band %d has a ratio below 1 (1 - 1/ratio = %g)",
                                   idx, b, c.coef);
        }
    return AME_OK;
}

// pydub: (1 - 1/ratio) * max(20 * math.log(rms / thresh_rms, 10), 0); CPython's two-argument log is
// log(x) / log(base) on the platform libm.  tau: smallest a >= 0 with fl(a + inc) >= m.
inline void build_att_table(AttEntry *e, const ame_comp_band &c) {
    const double ln10 = std::log(10.0);
    for (int r = 0; r <= 32768; ++r) {
        double over = 0.0;
        if (r != 0) {
            const double ratio = (double)r / c.thresh_rms;
            if (ratio != 0.0) {
                const double db = 20 * (std::log(ratio) / ln10);
                over = db > 0 ? db : 0.0;
            }
        }
        const double m = c.coef * over;
        const double inc = m / c.attack_frames;
        double tau = m - inc;
        if (!(tau > 0)) tau = 0.0;
        while (tau > 0 && tau + inc >= m) tau = std::nextafter(tau, -1.0);
        while (tau + inc < m) tau = std::nextafter(tau, 1e300);
        e[r] = AttEntry{m, inc, m / c.release_frames, tau};
    }
}

// Validates the tracks and lays the batch out: packing, waves and workspace slots, tile sizes and every job table.  On
// failure returns the status and leaves its message in `err`.
inline int build_layout(const ame_track_params *tracks, int n_tracks, const ame_plan_options &o, const DeviceShape &dev,
                        Layout &lay, JobTables &jobs, std::string &err) {
    lay.tracks.assign(tracks, tracks + n_tracks);
    std::vector<std::pair<int64_t, int64_t>> spans;
    lay.mb_offset.assign(n_tracks, -1);
    lay.tdev.resize(n_tracks);
    int64_t sum_frames = 0;
    for (int t = 0; t < n_tracks; ++t) {
        const ame_track_params &tp = lay.tracks[t];
        if (int rc = validate(tp, t, err)) return rc;
        const int64_t n_total = tp.halo_frames + tp.n_frames;
        if (t && tp.offset_frames < lay.tracks[t - 1].offset_frames)
            return layout_fail(err, AME_E_INVALID, "tracks must be ordered by offset_frames");
        spans.emplace_back(tp.offset_frames, tp.offset_frames + n_total);
        lay.total_frames = std::max(lay.total_frames, align_up(tp.offset_frames + n_total, 8));
        sum_frames += tp.n_frames;
        const int s100 = (tp.sample_rate + 5) / 10;
        TrackDev &td = lay.tdev[t];
        td.s100 = s100;
        td.n_sb = (int)(n_total / s100);
        td.n_total = n_total;
        // blocks whose last sub-block lies in the halo were counted by the previous shard
        td.first_block = tp.halo_frames ? std::max<int>(0, (int)(tp.halo_frames / s100) - 3) : 0;
        td.sb_offset = lay.n_sb_total;
        lay.n_sb_total += td.n_sb;
        td.pad = 0;
        td.lim_tile0 = 0;
        td.lim_shift = 15;
        lay.any_limiter = lay.any_limiter || (tp.flags & AME_F_LIMITER);
        if (tp.flags & AME_F_LIMITER) lay.lim_keep = std::max(lay.lim_keep, tp.lim_frames + 2);
        lay.any_tp = lay.any_tp || (tp.flags & AME_F_TRUE_PEAK);
        lay.any_meter = lay.any_meter || (tp.flags & AME_F_MEASURE_OUTPUT);
    }
    if (lay.any_meter) {
        lay.meter_tdev = lay.tdev;
        for (int t = 0; t < n_tracks; ++t) {
            lay.meter_tdev[t].sb_offset = lay.meter_sb_total;
            if (lay.tracks[t].flags & AME_F_MEASURE_OUTPUT) lay.meter_sb_total += lay.tdev[t].n_sb;
        }
    }
    for (size_t i = 1; i < spans.size(); ++i)
        if (spans[i].first < align_up(spans[i - 1].second, 8))
            return layout_fail(err, AME_E_INVALID, "tracks overlap in the packed buffer");
    if (lay.total_frames == 0) lay.total_frames = 8;

    // ---- waves: contiguous track ranges with about equal frames ----------------------------------
    int n_waves = o.n_waves > 0 ? o.n_waves : 1;
    n_waves = std::max(1, std::min(n_waves, n_tracks));
    {
        // With many waves the FIRST wave is a single track: in the host path nothing can be copied back before the
        // first wave has been copied in and mastered, so a small first wave starts the D2H stream early.
        lay.waves.resize(n_waves);
        const bool small_first = o.host_io && n_waves >= 4 && n_tracks >= 2 * n_waves;
        int t = 0;
        int64_t acc = 0;
        const int64_t first_frames = small_first ? lay.tracks[0].n_frames : 0;
        for (int w = 0; w < n_waves; ++w) {
            Wave &wv = lay.waves[w];
            wv.track_lo = t;
            const int must_leave = n_waves - 1 - w;                 // at least one track for every later wave
            if (small_first && w == 0) {
                acc += lay.tracks[t++].n_frames;
            } else {
                const int64_t share = small_first ? w : w + 1;
                const int64_t parts = small_first ? n_waves - 1 : n_waves;
                const int64_t target = first_frames + (sum_frames - first_frames) * share / parts;
                while (t < n_tracks - must_leave && (t == wv.track_lo || acc + lay.tracks[t].n_frames / 2 <= target)) acc += lay.tracks[t++].n_frames;
            }
            if (w == n_waves - 1) t = n_tracks;
            wv.track_hi = t;
            wv.frame_lo = lay.tracks[wv.track_lo].offset_frames;
            wv.frame_hi = (wv.track_hi < n_tracks) ? lay.tracks[wv.track_hi].offset_frames : lay.total_frames;
        }
    }
    // Slots: a wave's intermediate buffers (pre-normalisation signal, bands, rms, attenuations) live in slot
    // w % n_slots and are recycled in stream order, so a batch far larger than the workspace can be planned.
    int n_slots = o.n_slots > 0 ? o.n_slots : std::min(n_waves, 4);
    n_slots = std::max(1, std::min(n_slots, n_waves));
    lay.n_slots = n_slots;
    for (int w = 0; w < n_waves; ++w) {
        Wave &wv = lay.waves[w];
        wv.slot = w % n_slots;
        int64_t mb = 0;
        for (int t = wv.track_lo; t < wv.track_hi; ++t)
            if (lay.tracks[t].flags & AME_F_MULTIBAND) {
                lay.mb_offset[t] = mb;                              // within the wave's own multiband packing
                mb += align_up(lay.tdev[t].n_total, 8);
            }
        lay.mb_frames = std::max(lay.mb_frames, mb);
        lay.slot_frames = std::max(lay.slot_frames, wv.frame_hi - wv.frame_lo);
    }

    // ---- chunk geometry, tile sizes -----------------------------------------------------------------
    // Tiles are sized so that ONE launch fills its share of the machine with one wave of resident threads (no tail
    // wave).  Waves in different slots run concurrently, so a launch gets 1 / min(n_slots, 4) of the resident threads.
    std::vector<std::vector<int64_t>> chunks_all(n_tracks);
    for (int t = 0; t < n_tracks; ++t) {
        const ame_track_params &tp = lay.tracks[t];
        const int64_t cf = tp.chunk_frames > 0 ? tp.chunk_frames : std::max<int64_t>(tp.n_frames, 1);
        for (int64_t c0 = 0; c0 < tp.n_frames; c0 += cf) chunks_all[t].push_back(std::min(cf, tp.n_frames - c0));
    }
    const int share = std::min(n_slots, 4);
    const int64_t eq_slots = (int64_t)dev.n_sm * std::max(dev.occ_eq, 1) * 128 / share;         // one thread per tile
    const int64_t split_slots = (int64_t)dev.n_sm * std::max(dev.occ_split, 1) * 128 / share;
    constexpr int64_t kMinTile = 512;
    int64_t split_tile = kMinTile;
    std::vector<double> eq_cost(n_tracks);
    std::vector<int64_t> eq_want(n_tracks, 32);
    int max_warm_kw = 0, min_s100 = 1 << 30;
    for (int t = 0; t < n_tracks; ++t) {
        eq_cost[t] = eq_cost_per_frame(lay.tracks[t]);
        max_warm_kw = std::max(max_warm_kw, lay.tracks[t].warm_kw);
        min_s100 = std::min(min_s100, lay.tdev[t].s100);
    }
    // One warp per scheduler already gives these FP64-bound kernels ~77 % of the throughput of two (k_eq alone: 13.7 vs
    // 10.6 ms), and every tile pays its warm-up once: when a wave is so small that a full set of resident threads would
    // make the tiles shorter than ~1.2 x the warm-up (one long 192 kHz track), half the threads do the job sooner -
    // (2T + W) / (2T * 0.77) < (T + W) / T  <=>  T < 1.17 W.
    auto fewer_threads = [](int64_t slots, double frames, double warm_weighted) {
        const double tile = frames / (double)slots, warm = frames > 0 ? warm_weighted / frames : 0.0;
        return (tile < 1.17 * warm && slots >= 512) ? slots / 2 : slots;
    };
    for (const Wave &wv : lay.waves) {
        std::vector<int64_t> cm;
        double eq_frames = 0, eq_warm = 0, mb_fr = 0, mb_warm = 0;
        for (int t = wv.track_lo; t < wv.track_hi; ++t) {
            const ame_track_params &tp = lay.tracks[t];
            eq_frames += (double)tp.n_frames;
            eq_warm += (double)tp.n_frames * tp.warm_eq;
            if (tp.flags & AME_F_MULTIBAND) {
                cm.insert(cm.end(), chunks_all[t].begin(), chunks_all[t].end());
                mb_fr += (double)tp.n_frames;
                mb_warm += (double)tp.n_frames * tp.warm_xover;
            }
        }
        split_tile = std::max(split_tile, pick_tile(cm, fewer_threads(split_slots, mb_fr, mb_warm), kMinTile));
        const std::vector<int64_t> tw = eq_jobs_per_track(lay.tracks.data(), chunks_all, eq_cost, wv.track_lo, wv.track_hi,
                                                          fewer_threads(eq_slots, eq_frames, eq_warm), kMinTile);
        for (int t = wv.track_lo; t < wv.track_hi; ++t) eq_want[t] = tw[t];
    }
    lay.split_tile = o.xover_tile_frames > 0 ? (int)align_up(o.xover_tile_frames, 8) : (int)split_tile;
    if (o.kw_tile_subblocks > 0) {
        lay.kw_tile_sb = o.kw_tile_subblocks;
    } else if (lay.n_sb_total > 0) {
        // a tile of sub-blocks costs (tile + warm-up) frames: keep the warm-up below ~15 % when the batch is big
        // enough to still give every SM ~512 threads per launch, else shrink the tile towards one sub-block
        const int64_t want = std::max<int64_t>(1, ((int64_t)max_warm_kw * 6 + min_s100 - 1) / min_s100);
        const int64_t fill = std::max<int64_t>(1, lay.n_sb_total / n_waves * share / ((int64_t)dev.n_sm * 512));
        lay.kw_tile_sb = (int)std::min(want, fill);
    } else {
        lay.kw_tile_sb = 1;
    }

    // ---- job tables (every table is ordered by track, hence contiguous per wave) ---------------------
    jobs.mb_delta.assign(n_tracks, 0);
    std::map<std::tuple<double, double, double, double>, int> table_index;
    int64_t n_seg_total = 0;

    for (Wave &wv : lay.waves) {
        wv.eq.lo = (int)jobs.eq.size(); wv.split.lo = (int)jobs.split.size(); wv.chain.lo = (int)jobs.chain.size();
        wv.mb_chunks.lo = (int)jobs.mb_chunks.size(); wv.kw.lo = (int)jobs.kw.size(); wv.gain.lo = (int)jobs.gain.size();
        wv.lim.lo = (int)jobs.lim.size();
        wv.seg_lo = n_seg_total;
        int64_t n_groups = 0;                          // group records of this wave (slot-local indices)
        std::map<int, std::vector<TileJob>> eq_bucket;   // k_eq jobs of this wave by variant (a warp runs ONE variant)
        for (int t = wv.track_lo; t < wv.track_hi; ++t) {
            ame_track_params &tp = lay.tracks[t];
            const int variant = eq_variant_of(tp);
            const bool mb = (tp.flags & AME_F_MULTIBAND) != 0;
            if (mb) {
                jobs.mb_delta[t] = lay.mb_offset[t] - tp.offset_frames;
                for (int b = 0; b < 3; ++b) {
                    ame_comp_band &c = tp.comp[b];
                    auto key = std::make_tuple(c.thresh_rms, c.coef, c.attack_frames, c.release_frames);
                    auto it = table_index.find(key);
                    if (it == table_index.end()) {
                        const int idx = (int)table_index.size();
                        table_index[key] = idx;
                        jobs.att.resize(jobs.att.size() + 32769);
                        build_att_table(jobs.att.data() + (size_t)idx * 32769, c);
                        c.table = idx;
                    } else {
                        c.table = it->second;
                    }
                }
            }
            // k_eq jobs of this track: eq_want[t] jobs spread over the chunks by length (or the requested tile), collected
            // per variant and laid out at the end of the wave
            {
                std::vector<TileJob> &bucket = eq_bucket[variant];
                int64_t c0e = 0, jobs_before = 0;
                int64_t nf = 0;
                for (int64_t cn : chunks_all[t]) nf += cn;
                nf = std::max<int64_t>(nf, 1);
                const int64_t want = eq_want[t];
                for (int64_t cn : chunks_all[t]) {
                    const int64_t cb = tp.offset_frames + tp.halo_frames + c0e, ce = cb + cn;
                    int64_t T;
                    if (o.eq_tile_frames > 0) {
                        T = align_up(o.eq_tile_frames, 8);
                    } else {
                        // cumulative rounding: the chunks together get exactly `want` jobs (never more)
                        const int64_t upto = (int64_t)((__int128)want * (c0e + cn) / nf);
                        const int64_t jc = std::max<int64_t>(1, upto - jobs_before);
                        jobs_before = upto;
                        T = std::max<int64_t>(kMinTile, align_up((cn + jc - 1) / jc, 8));
                    }
                    tile_jobs(bucket, t, variant, cb, ce, T);
                    c0e += cn;
                }
            }
            int64_t c0 = 0;
            for (int64_t cn : chunks_all[t]) {
                const int64_t cb = tp.offset_frames + tp.halo_frames + c0, ce = cb + cn;
                if (mb) {
                    tile_jobs(jobs.split, t, 0, cb, ce, lay.split_tile);
                    MbChunk ck{cb, lay.mb_offset[t] + tp.halo_frames + c0, cn, n_seg_total, {0, 0, 0}, t, 0};
                    for (int b = 0; b < 3; ++b) {
                        const double thr = tp.comp[b].thresh_rms;
                        const uint32_t thr_i = thr >= 65535.0 ? 0x7fffffffu : (uint32_t)std::floor(thr) + 1u;
                        ck.grp_begin[b] = n_groups;
                        jobs.chain.push_back(ChainJob{ck.mb_begin, cn, n_groups, b, tp.comp[b].table, thr_i, tp.comp[b].look_frames, 0, 0});
                        n_groups += (cn + 31) / 32;
                    }
                    n_seg_total += (cn + kSeg - 1) / kSeg;
                    jobs.mb_chunks.push_back(ck);
                }
                c0 += cn;
            }
            for (int sb = 0; sb < lay.tdev[t].n_sb; sb += lay.kw_tile_sb)
                jobs.kw.push_back(KwJob{t, sb, std::min(sb + lay.kw_tile_sb, lay.tdev[t].n_sb), 0});
            for (int64_t b = 0; b < tp.n_frames; b += kGainTile)
                jobs.gain.push_back(GainJob{tp.offset_frames + tp.halo_frames + b,
                                            tp.offset_frames + tp.halo_frames + std::min<int64_t>(b + kGainTile, tp.n_frames), t, 0});
            if (tp.flags & AME_F_LIMITER) {
                // limiter tiles: a power of two >= G = look-ahead + release + 8 (a tile without an over-limit frame then
                // guarantees the initial state at its end), as short as that allows: more tiles = more warps in flight
                const int64_t G = (int64_t)tp.lim_frames + tp.lim_release_frames + 8;
                int shift = 13;
                while ((1LL << shift) < G) ++shift;
                lay.tdev[t].lim_shift = shift;
                lay.tdev[t].lim_tile0 = (int)jobs.lim.size() - wv.lim.lo;
                for (int64_t b = 0; b < tp.n_frames; b += 1LL << shift)
                    jobs.lim.push_back(GainJob{tp.offset_frames + tp.halo_frames + b,
                                               tp.offset_frames + tp.halo_frames + std::min<int64_t>(b + (1LL << shift), tp.n_frames), t, 0});
            }
        }
        {
            bool have_x = false, have_k = false;
            wv.xover_uni = wv.kw_uni = true;
            for (int t = wv.track_lo; t < wv.track_hi; ++t) {
                const ame_track_params &tp = lay.tracks[t];
                if (tp.flags & AME_F_MULTIBAND) {
                    const XoverCfg x{tp.xlp[0].b0, tp.xlp[0].a1, tp.xlp[0].a2, tp.xlp[1].a1, tp.xlp[1].a2,
                                     tp.xhp[0].b0, tp.xhp[0].a1, tp.xhp[0].a2, tp.xhp[1].a1, tp.xhp[1].a2};
                    if (!have_x) { wv.xover = x; have_x = true; }
                    else if (std::memcmp(&x, &wv.xover, sizeof x)) wv.xover_uni = false;
                }
                {
                    const KwCfg k{tp.kw[0].b0, tp.kw[0].b1, tp.kw[0].b2, tp.kw[0].a1, tp.kw[0].a2, tp.kw[1].a1, tp.kw[1].a2};
                    const bool rlb = tp.kw[1].b0 == 1.0 && tp.kw[1].b1 == -2.0 && tp.kw[1].b2 == 1.0;
                    if (!have_k) { wv.kw_cfg = k; have_k = true; }
                    else if (std::memcmp(&k, &wv.kw_cfg, sizeof k)) wv.kw_uni = false;
                    if (!rlb) wv.kw_uni = false;
                }
            }
        }
        lay.slot_groups = std::max(lay.slot_groups, n_groups);
        // longest chains first inside the wave: the launch ends with its slowest CTA
        std::stable_sort(jobs.chain.begin() + wv.chain.lo, jobs.chain.end(), [](const ChainJob &a, const ChainJob &b) { return a.n > b.n; });
        wv.wf.lo = (int)jobs.wf.size();
        for (int c = wv.chain.lo; c < (int)jobs.chain.size(); ++c) {
            jobs.chain[c].tile0 = (int)jobs.wf.size() - wv.wf.lo;
            const ChainJob &cj = jobs.chain[c];
            for (int64_t tb = 0; tb < cj.n; tb += kWfTile)
                jobs.wf.push_back(WfJob{tb, (int64_t)cj.band * lay.mb_frames + cj.mb_begin, cj.n, cj.grp_begin, c, cj.look, cj.thr_i, cj.tile0});
        }
        // every variant's run is padded to whole warps (a warp runs ONE variant) and the runs follow one another in
        // variant order; with one 8-warp CTA per SM nearly every SM then executes ONE variant - each variant is its own
        // ~19 KB unrolled loop in the instruction cache (two 4-warp CTAs of different variants per SM: 10.5 ms on the
        // 128-track launch, one 8-warp CTA: 9.7 ms).  Interleaving the variants' warps in proportion (every SM gets the
        // wave's mix of FP64-heavy and load-bound warps) gave 18.0 ms: four loops per CTA (profiles/r02/summary.md).
        for (auto &kv : eq_bucket) {
            std::vector<TileJob> &b = kv.second;
            if (b.empty()) continue;
            TileJob d = b.back();
            d.tile_begin = d.tile_end;
            while (b.size() % 32) b.push_back(d);
            jobs.eq.insert(jobs.eq.end(), b.begin(), b.end());
        }
        wv.eq.n = (int)jobs.eq.size() - wv.eq.lo; wv.split.n = (int)jobs.split.size() - wv.split.lo;
        wv.chain.n = (int)jobs.chain.size() - wv.chain.lo; wv.wf.n = (int)jobs.wf.size() - wv.wf.lo;
        wv.mb_chunks.n = (int)jobs.mb_chunks.size() - wv.mb_chunks.lo; wv.kw.n = (int)jobs.kw.size() - wv.kw.lo;
        wv.gain.n = (int)jobs.gain.size() - wv.gain.lo; wv.seg_hi = n_seg_total;
        wv.lim.n = (int)jobs.lim.size() - wv.lim.lo;
        for (int t = wv.track_lo; t < wv.track_hi; ++t) {
            wv.limiter = wv.limiter || (lay.tracks[t].flags & AME_F_LIMITER);
            wv.true_peak = wv.true_peak || (lay.tracks[t].flags & AME_F_TRUE_PEAK);
        }
        // the output meter: the same K-weighting and gain tiles as the input side, for the flagged tracks only
        wv.meter_kw.lo = (int)jobs.meter_kw.size(); wv.meter_peak.lo = (int)jobs.meter_peak.size();
        wv.meter_tracks.lo = (int)jobs.meter_tracks.size();
        for (int t = wv.track_lo; t < wv.track_hi; ++t) {
            const ame_track_params &tp = lay.tracks[t];
            if (!(tp.flags & AME_F_MEASURE_OUTPUT)) continue;
            jobs.meter_tracks.push_back(t);
            for (int sb = 0; sb < lay.tdev[t].n_sb; sb += lay.kw_tile_sb)
                jobs.meter_kw.push_back(KwJob{t, sb, std::min(sb + lay.kw_tile_sb, lay.tdev[t].n_sb), 0});
            for (int64_t b = 0; b < tp.n_frames; b += kGainTile)
                jobs.meter_peak.push_back(GainJob{tp.offset_frames + b, tp.offset_frames + std::min<int64_t>(b + kGainTile, tp.n_frames), t, 0});
        }
        wv.meter_kw.n = (int)jobs.meter_kw.size() - wv.meter_kw.lo; wv.meter_peak.n = (int)jobs.meter_peak.size() - wv.meter_peak.lo;
        wv.meter_tracks.n = (int)jobs.meter_tracks.size() - wv.meter_tracks.lo;
        lay.slot_lim_jobs = std::max(lay.slot_lim_jobs, wv.lim.n);
        lay.slot_tiles = std::max(lay.slot_tiles, wv.wf.n);
        lay.slot_chains = std::max(lay.slot_chains, wv.chain.n);
    }
    return AME_OK;
}

}  // namespace ame
