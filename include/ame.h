/* libame - C ABI of the B200 (sm_100a) mastering DSP chain.
 *
 * This is the drop-in boundary for ONE path of theouterlimitz/Audio-Mastering-Engine: the per-chunk
 * DSP loop plus loudness normalisation of process_audio_with_ffmpeg_pipeline()
 * (audio_mastering_engine.py:171-246 and the ops at :250-309).  The reference has no FFI layer of its
 * own (pure Python); each entry point below names the reference function(s) it replaces.
 *
 * Conventions
 *   - extern "C", plain pointers and sizes, no torch / C++ types.
 *   - every function returns 0 on success or a negative ame_status; ame_last_error() gives the text.
 *   - audio is interleaved stereo int16 ("frames" = L,R pairs).  A batch is ONE packed buffer;
 *     track t occupies frames [offset_frames, offset_frames + n_frames); offsets are multiples of 8
 *     frames and the buffer is padded to a multiple of 8 frames.
 *   - the caller owns audio buffers; a plan owns its workspace (allocated in ame_plan_create, never on
 *     the processing path).  A plan is bound to one device and one stream at a time (not thread safe);
 *     distinct plans are independent (one per GPU / per concurrent batch).
 *   - there is NO CPU fallback: without a CUDA device every processing call fails with AME_E_CUDA.
 *
 * Filter design stays on the host exactly as the reference does it (scipy.signal.butter at
 * audio_mastering_engine.py:285,296,301,302): the host fills ame_track_params with the designed
 * coefficients; see audio_mastering_engine_b200/design.py.
 */
#ifndef AME_H
#define AME_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define AME_ABI_VERSION 5
#define AME_N_KERNELS 12   /* timed kernel slots of the path, in launch order (ame_kernel_name) */

typedef enum {
    AME_OK = 0,
    AME_E_INVALID = -1,   /* bad argument / inconsistent params */
    AME_E_CUDA = -2,      /* CUDA runtime error (message has the CUDA text) */
    AME_E_NOMEM = -3,     /* workspace allocation failed */
    AME_E_UNSUPPORTED = -4
} ame_status;

/* flags in ame_track_params.flags */
#define AME_F_WARMTH    1u  /* analog_character > 0            (audio_mastering_engine.py:192) */
#define AME_F_WIDTH     2u  /* width != 1.0                    (:195) */
#define AME_F_MULTIBAND 4u  /* settings["multiband"] truthy    (:197) */
#define AME_F_NORMALIZE 8u  /* settings["lufs"] is not None    (:216) */
#define AME_F_LIMITER   16u /* the final ffmpeg alimiter       (:223); not for time shards (global sequential state) */
#define AME_F_TRUE_PEAK 32u /* also measure the BS.1770 Annex 2 true peak of the pre-normalisation signal */
#define AME_F_MEASURE_OUTPUT 64u /* meter the track's final output (ame_loudness); not for time shards (a shard's output is
                                    not the track's output) */

/* EQ stage kinds (apply_shelf_filter :283-289, apply_peak_filter :290-298) */
#define AME_EQ_BYPASS      0  /* gain == 0: stage returns its input untouched */
#define AME_EQ_SHELF_BOOST 1  /* y = x + (H(x) - x) * (g - 1)   one biquad */
#define AME_EQ_SHELF_CUT   2  /* y = x*g + (H(x) - x*g)         one biquad (== bare H(x)) */
#define AME_EQ_PEAK        3  /* y = x + BP4(x) * (g - 1)       four biquads */

/* One second-order section, a0 == 1:  y = b0 x + z0 ; z0 = b1 x - a1 y + z1 ; z1 = b2 x - a2 y
 * (direct form II transposed, the form scipy lfilter/sosfilt evaluate). */
typedef struct { double b0, b1, b2, a1, a2; } ame_biquad;

typedef struct {
    int32_t kind;        /* AME_EQ_* */
    int32_t n_sections;  /* 1 (shelf) or 4 (peak) */
    double g;            /* 10^(gain_db/20) */
    double gm1;          /* g - 1 */
    ame_biquad s[4];
} ame_eq_stage;

typedef struct {
    double thresh_rms;      /* 32768 * 10^(threshold/20)                   (pydub effects.py) */
    double coef;            /* 1 - 1/ratio */
    double attack_frames;   /* 5 ms  * fs/1000 (a float, 220.5 at 44.1 kHz) */
    double release_frames;  /* 50 ms * fs/1000 */
    int32_t look_frames;    /* int(attack_frames) */
    int32_t table;          /* index into the plan's attenuation tables (ame_plan_create fills it) */
} ame_comp_band;

/* Everything the kernels need for one track.  Filled by the host from the reference's settings dict. */
typedef struct {
    int64_t offset_frames;   /* start of the track in the packed buffers (multiple of 8) */
    int64_t n_frames;        /* frames this plan masters (for a time shard: the shard's span) */
    int64_t halo_frames;     /* time shards only: frames stored BEFORE the span, [offset, offset + halo), that hold
                                the previous shard's already-mastered pre-normalisation tail; they warm the K filter
                                up and complete the 400 ms blocks that straddle the shard boundary.  A multiple of
                                8 and of the 100 ms sub-block; 0 for whole tracks */
    int32_t sample_rate;
    int32_t chunk_frames;    /* state-reset period: 30 * fs (:178); <= 0 means the whole track */
    uint32_t flags;          /* AME_F_* */
    int32_t warm_lut;        /* index of the tanh table for this drive (ame_plan_set_warm_lut), or -1 */
    /* warmth: per frame, across the two channels (apply_analog_character :258-266) */
    double wl_b0, wl_b1, wl_a1, wl_gm1;   /* butter(2, 120 Hz, low)  and 10^(cf*1.0/20) - 1 */
    double wh_b0, wh_b1, wh_a1, wh_gm1;   /* butter(2, 12 kHz, high) and 10^(cf*1.5/20) - 1 */
    /* EQ cascade: low shelf 250, peak 1k, peak 4k, high shelf 8k (:277-282) */
    ame_eq_stage eq[4];
    float width;             /* stereo width factor as float32 (:267-271) */
    float pad0_;
    /* multiband (:299-309) */
    ame_biquad xlp[2];       /* butter(4, 250 Hz, lowpass)  as 2 sections */
    ame_biquad xhp[2];       /* butter(4, 4 kHz, highpass)  as 2 sections */
    ame_comp_band comp[3];   /* low, mid, high */
    /* loudness (normalize_loudness_on_disk_with_ffmpeg :227-246, ffmpeg ebur128/loudnorm) */
    ame_biquad kw[2];        /* BS.1770 pre-filter shelf, RLB high-pass */
    double target_lufs;
    /* warm-up (frames processed before a tile only to converge filter state; see DESIGN.md) */
    int32_t warm_eq, warm_xover, warm_kw;
    /* ffmpeg alimiter (:223): limit, 1 / limit (auto level), sample_rate * release[s], look-ahead frames
     * B = int(fs * attack[s] * 2) / 2, release in frames (rounded up), and the smallest |s16| whose x / 32768 exceeds
     * the limit */
    int32_t lim_frames;
    double lim_limit, lim_level, lim_fs_release;
    int32_t lim_release_frames, lim_thr_i;
} ame_track_params;

/* Per-track result of the loudness stage (the numbers ffmpeg prints as JSON at :229-237). */
typedef struct {
    double input_i;          /* integrated loudness, LUFS; -inf when no block passes the gate */
    double measured_i_2dp;   /* input_i rounded to 2 decimals (the '%.2f' string fed to pass 2) */
    double gain;             /* linear gain applied (1.0 when not normalised) */
    double rel_threshold;    /* relative-gate threshold as energy */
    int64_t n_blocks;        /* 400 ms blocks above the absolute gate */
    int32_t normalized;      /* 1 iff a gain was applied */
    int32_t sample_peak;     /* max |s16| of the pre-normalisation signal */
    double input_lra;        /* loudness range, LU (ebur128 short-term histogram, 10th..95th percentile) */
    double input_thresh;     /* relative gate threshold, LUFS (ffmpeg's input_thresh) */
    double true_peak;        /* BS.1770 Annex 2 true peak of the pre-normalisation signal, linear (1.0 = full scale);
                                the sample peak / 32768 when AME_F_TRUE_PEAK is not set or fs >= 192 kHz */
} ame_track_result;

/* EBU R128 meter of one track (AME_F_MEASURE_OUTPUT): what ffmpeg's loudnorm prints as output_* in its second pass, plus
 * the maxima of the ungated momentary (400 ms) and short-term (3 s) loudness, both taken every 100 ms.  integrated,
 * thresh, lra, n_blocks, sample_peak and true_peak are computed exactly as the input side of ame_track_result is. */
typedef struct {
    double integrated;      /* LUFS (ebur128 gated); -inf when no block passes the gate */
    double thresh;          /* relative gate threshold, LUFS; -70 when no block passes the absolute gate */
    double lra;             /* loudness range, LU */
    double true_peak;       /* linear; BS.1770 Annex 2 (4x below 96 kHz, 2x below 192 kHz), else sample peak / 32768 */
    double max_momentary;   /* LUFS; -inf when the track has no complete 400 ms window */
    double max_short_term;  /* LUFS; -inf when the track has no complete 3 s window */
    int64_t n_blocks;       /* 400 ms blocks above the absolute gate */
    int32_t sample_peak;    /* max |s16| over every frame of the track */
    int32_t measured;       /* 1 when this entry holds a measurement */
} ame_loudness;

typedef struct {
    int32_t eq_tile_frames;      /* 0 = choose from the batch size */
    int32_t xover_tile_frames;   /* 0 = auto */
    int32_t kw_tile_subblocks;   /* 0 = auto */
    int32_t host_io;             /* 1 = also allocate device in/out buffers for ame_master_host */
    int32_t n_waves;             /* <= 1: one wave.  > 1: split the batch into that many contiguous groups of tracks;
                                    each wave runs on its own stream, so the latency-bound sequential compressor kernel
                                    of one wave overlaps the bulk kernels of the others, and ame_master_host also
                                    overlaps the H2D copy of wave w+1 and the D2H copy of wave w-1 with the kernels of
                                    wave w.  Tiles shrink with the wave, so more waves = more filter warm-up work */
    int32_t chain_warps;         /* compressor recurrence (k_att_chain): 0 = 4..8 warps (x32 speculative time segments)
                                    per chain, chosen per launch; 1..8 = that many warps; -1 = ONE lane per chain, i.e.
                                    the sequential loop of the reference (the baseline the speculation is tested against) */
    int32_t n_slots;             /* workspace slots: wave w runs in slot w % n_slots on that slot's stream, so only
                                    n_slots waves are in flight and the plan's workspace is that of n_slots waves, not
                                    of the batch (1024 tracks fit one GPU).  <= 0: min(n_waves, 4) */
    int32_t precision;           /* 0 = FP64 filters (results equal to the reference's float64 scipy path);
                                    1 = EQ cascade in FP32 (A/B measurement only: +-1 LSB truncation flips, which the
                                    make-up gain of the loudness stage multiplies - DESIGN.md) */
} ame_plan_options;

typedef struct ame_plan ame_plan;

/* library ------------------------------------------------------------------------------------- */
int ame_abi_version(void);
size_t ame_sizeof_track_params(void);
size_t ame_sizeof_track_result(void);
size_t ame_sizeof_plan_options(void);
size_t ame_sizeof_loudness(void);
const char *ame_last_error(void);             /* thread-local text of the last failure */
int ame_device_count(int *count);
/* plan workspaces are taken from a per-device memory pool that keeps the memory of destroyed plans for the next one
 * (creating and destroying a plan per track then costs microseconds instead of ~100 ms); this returns it to the driver */
int ame_release_cached_memory(int device);

/* plan: geometry + coefficients + workspace for one batch on one device ------------------------- */
int ame_plan_create(int device, const ame_track_params *tracks, int32_t n_tracks,
                    const ame_plan_options *opt, ame_plan **plan);
void ame_plan_destroy(ame_plan *plan);
/* tanh tables for the warmth stage: lut[i] = float32 tanh(float32((i-32768)/32768) * drive),
 * 65536 floats each, built on the host with the SAME libm/numpy call the reference makes (:263). */
int ame_plan_set_warm_luts(ame_plan *plan, const float *luts, int32_t n_luts);
int64_t ame_plan_total_frames(const ame_plan *plan);     /* padded length of the packed buffers */
size_t ame_plan_workspace_bytes(const ame_plan *plan);
int64_t ame_plan_launch_count(const ame_plan *plan);      /* kernels launched by the last ame_master_* / ame_measure_device /
                                                             ame_measure_loudness call (the meter's launches included) */
int32_t ame_plan_wave_count(const ame_plan *plan);
int32_t ame_plan_slot_count(const ame_plan *plan);
/* statistics of the compressor recurrence of the last call (benchmarks): chains, flagged steps in total and in the
 * longest chain, passes (1 + repairs) in total and at most */
/* limiter (AME_F_LIMITER): tiles whose guessed start state was not their predecessor's end state after round 0, 1, 2
 * of k_limiter, summed over the calls since the last query (what is open after round 2 is walked sequentially) */
int ame_plan_limiter_stats(ame_plan *plan, int64_t *open_tiles /* [3] */);
int ame_plan_chain_stats(ame_plan *plan, int64_t *n_chains, int64_t *steps, int64_t *max_steps, int64_t *passes,
                         int32_t *max_passes);
/* limiter, diagnostic / test knob: the round-0 guess of a tile's start state runs the machine from the initial state
 * over `frames` frames in front of the tile (clipped at the track start; only a guess that reaches the track start
 * counts as exact).  -1 (the default) = 2 G frames, G = look-ahead + release + 8; 0 = every tile that does not start
 * in the initial state starts from it, a wrong guess on every such tile of a clipping track.  Shorter windows give
 * wrong guesses and so run the repair rounds and the sequential fallback; the output is the same for every value.
 * Applies to the following calls of the plan. */
int ame_plan_set_limiter_guess(ame_plan *plan, int32_t frames);

/* per-kernel device timing with CUDA events on the processing stream(s) (benchmarks): enable, run up to 64
 * ame_master_* / ame_measure_* calls, then read the summed milliseconds and launch counts per kernel (with
 * several waves every wave's launch is timed on its own stream; overlapping launches share the machine, so
 * their durations add up to more than the wall time). */
int ame_plan_set_timing(ame_plan *plan, int enable);
int ame_plan_kernel_times(ame_plan *plan, double *ms_sum, int64_t *launches, int *n_steps);
const char *ame_kernel_name(int slot);
/* timeline of the last ame_master_host call made with timing enabled: for each wave, milliseconds since the call's
 * first copy was queued at which {its H2D copy finished, its kernels could start, its kernels finished, its D2H copy
 * finished}.  ms holds 4 * max_waves floats; returns the number of waves written, or a negative error. */
int ame_plan_wave_timeline(ame_plan *plan, float *ms, int max_waves);
/* where each launch of timed step `step` (0 = the first call after ame_plan_set_timing) sat on the device: ms holds
 * 2 * AME_N_KERNELS * max_waves floats, {begin, end} per (wave, kernel slot) in milliseconds after the step's first
 * event (slightly negative for a wave whose stream started before wave 0's), NaN for kernels the wave did not
 * launch.  "begin" is when the wave's stream reached the launch, so a launch that waited for free SMs shows the wait
 * as duration.  Returns the number of waves written, or a negative error. */
int ame_plan_kernel_timeline(ame_plan *plan, int step, float *ms, int max_waves);

/* the whole path: replaces the chunk loop + concat + loudnorm of
 * process_audio_with_ffmpeg_pipeline (:185-220).  d_in / d_out are DEVICE pointers to packed
 * int16 stereo (ame_plan_total_frames frames); results is a HOST array of n_tracks entries
 * (may be NULL).  stream is a cudaStream_t (NULL = default stream). */
int ame_master_device(ame_plan *plan, const int16_t *d_in, int16_t *d_out,
                      ame_track_result *results, void *stream);
/* same with HOST buffers (pinned or pageable): H2D, the chain, D2H - pipelined over the plan's waves -
 * synchronised on return. */
int ame_master_host(ame_plan *plan, const int16_t *h_in, int16_t *h_out, ame_track_result *results);

/* EBU R128 meter.  When tracks carry AME_F_MEASURE_OUTPUT, ame_master_device, ame_master_host and ame_normalize_device
 * also meter the FINAL output of those tracks (after the gain, and after the limiter when the track has one), on the
 * streams the call runs on; ame_plan_output_loudness copies those results on `stream` (which must be ordered after the
 * call) and synchronises it.  Before any such call every entry has measured = 0.  out: HOST array of n_tracks entries;
 * tracks without the flag get measured = 0.  The ame_stage_* entry points do not meter. */
int ame_plan_output_loudness(ame_plan *plan, ame_loudness *out, void *stream);
/* stand-alone meter: every track that carries AME_F_MEASURE_OUTPUT, read from d_buf (any DEVICE buffer in the plan's
 * packed layout; the other flags of the track do not matter), on `stream`.  out (may be NULL) is filled synchronously.
 * AME_E_INVALID when no track carries the flag.  Does not touch what ame_plan_output_loudness reports. */
int ame_measure_loudness(ame_plan *plan, const int16_t *d_buf, ame_loudness *out, void *stream);

/* two-phase form for tracks that are time-sharded across GPUs: phase 1 stops after the gating
 * histograms (d_hist: DEVICE int64[n_tracks][1000], caller-owned so it can be all-reduced with
 * NCCL); phase 2 derives the gain from (possibly all-reduced) histograms and applies it.
 * Every wave must keep its pre-normalisation signal between the two calls: n_slots == n_waves. */
int ame_measure_device(ame_plan *plan, const int16_t *d_in, int64_t *d_hist, void *stream);
int ame_normalize_device(ame_plan *plan, const int64_t *d_hist, int16_t *d_out,
                         ame_track_result *results, void *stream);

/* by-time sharding from a host that is not Python (SURVEY 8(b), 8(e)): one plan over ONE track [halo | span] per
 * rank; between ame_stage_compress and ame_stage_loudness_hist a rank sends the last send_frames of its
 * pre-normalisation signal to the next rank and receives its own halo from the previous one (rank < 0 = none), and
 * between ame_stage_loudness_hist and ame_stage_apply_gain the int64[n_tracks][1000] histograms are all-reduced (sum)
 * so that every rank derives the same integrated loudness and gain.  nccl_comm is the caller's ncclComm_t; NCCL is
 * resolved from the process at run time (AME_E_UNSUPPORTED when there is none).  examples/time_shard_nccl.c. */
int ame_shard_halo_exchange(ame_plan *plan, int16_t *d_pre, void *nccl_comm, int prev_rank, int next_rank,
                            int64_t send_frames, void *stream);
int ame_hist_allreduce(ame_plan *plan, int64_t *d_hist, void *nccl_comm, void *stream);

/* stage entry points (parity taps; each replaces the named reference function; plans with ONE wave) */
/* warmth -> int16 -> EQ -> width -> int16: apply_analog_character, audio_segment_to_float_array,
 * apply_eq_to_samples, apply_stereo_width, float_array_to_audio_segment (:192-196) */
int ame_stage_eq(ame_plan *plan, const int16_t *d_in, int16_t *d_pre, void *stream);
/* crossover + int16 truncation of the three bands (:300-305); d_bands = 3 packed buffers back to back */
int ame_stage_band_split(ame_plan *plan, const int16_t *d_pre, int16_t *d_bands, void *stream);
/* pydub compress_dynamic_range on each band + overlay into d_pre (:306-309); d_bands is not modified */
int ame_stage_compress(ame_plan *plan, int16_t *d_bands, int16_t *d_pre, void *stream);
/* K-weighting + 100 ms energies + 400 ms block histogram (ebur128) */
int ame_stage_loudness_hist(ame_plan *plan, const int16_t *d_pre, int64_t *d_hist, void *stream);
/* static gain + s16 rounding (loudnorm linear mode) */
int ame_stage_apply_gain(ame_plan *plan, const int16_t *d_pre, const int64_t *d_hist,
                         int16_t *d_out, ame_track_result *results, void *stream);
/* ffmpeg alimiter alone (audio_mastering_engine.py:223) over a signal that is already normalised - every track of the
 * plan must carry AME_F_LIMITER.  This is how a time-sharded track (whose shards cannot carry the limiter's sequential
 * state) is limited after its spans have been gathered.  Clears the plan's per-track results. */
int ame_stage_limiter(ame_plan *plan, const int16_t *d_norm, int16_t *d_out, void *stream);

/* workspace taps for tests: device pointers owned by the plan (valid until destroy) */
const int16_t *ame_plan_tap_pre(const ame_plan *plan);       /* pre-normalisation int16 */
const int16_t *ame_plan_tap_bands(const ame_plan *plan);     /* 3 x mb-packed int16 band buffers */
const double *ame_plan_tap_subblock_energy(const ame_plan *plan);
int64_t ame_plan_mb_frames(const ame_plan *plan);            /* padded frames of the multiband-only packing */
int64_t ame_plan_mb_offset(const ame_plan *plan, int32_t track); /* -1 when the track is not multiband */
int64_t ame_plan_subblock_offset(const ame_plan *plan, int32_t track);
/* synchronous device -> host copy of a tap (debug / tests; not on the processing path) */
int ame_plan_read_device(ame_plan *plan, void *h_dst, const void *d_src, size_t bytes);

#ifdef __cplusplus
}
#endif
#endif /* AME_H */
