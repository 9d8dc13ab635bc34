// Runs build_layout on the host and prints the layout as JSON (tests/test_plan_layout.py).  Built with g++ alone: the
// layout must not need CUDA.
//   plan_layout_driver TRACKS OPTIONS N_SM OCC_EQ OCC_SPLIT
// TRACKS holds raw ame_track_params, OPTIONS one raw ame_plan_options.
#include <cstdio>
#include <cstdlib>
#include <fstream>
#include <iterator>
#include <string>
#include <vector>

#include "../audio_mastering_engine_b200/csrc/ame_layout.h"

using namespace ame;

static std::string read_file(const char *path) {
    std::ifstream f(path, std::ios::binary);
    return std::string(std::istreambuf_iterator<char>(f), std::istreambuf_iterator<char>());
}

template <class T, class F>
static void array(const char *name, const std::vector<T> &v, F row) {
    std::printf(",\n\"%s\": [", name);
    for (size_t i = 0; i < v.size(); ++i) {
        std::printf(i ? ",[" : "[");
        row(v[i]);
        std::printf("]");
    }
    std::printf("]");
}

int main(int argc, char **argv) {
    if (argc != 6) {
        std::fprintf(stderr, "usage: %s TRACKS OPTIONS N_SM OCC_EQ OCC_SPLIT\n", argv[0]);
        return 2;
    }
    const std::string tr = read_file(argv[1]), op = read_file(argv[2]);
    if (tr.size() % sizeof(ame_track_params) || op.size() != sizeof(ame_plan_options)) {
        std::fprintf(stderr, "input sizes do not match ame_track_params / ame_plan_options\n");
        return 2;
    }
    std::vector<ame_track_params> tracks(tr.size() / sizeof(ame_track_params));
    std::memcpy(tracks.data(), tr.data(), tr.size());
    ame_plan_options o;
    std::memcpy(&o, op.data(), sizeof o);
    const DeviceShape shape{std::atoi(argv[3]), std::atoi(argv[4]), std::atoi(argv[5])};

    Layout lay;
    JobTables jobs;
    std::string err;
    const int rc = build_layout(tracks.data(), (int)tracks.size(), o, shape, lay, jobs, err);
    std::printf("{\"rc\": %d, \"error\": \"", rc);
    for (char c : err) std::printf(c == '"' || c == '\\' ? "\\%c" : "%c", c);
    std::printf("\"");
    if (rc) {
        std::printf("}\n");
        return 0;
    }
    std::printf(",\n\"scalars\": {\"n_slots\": %d, \"total_frames\": %lld, \"mb_frames\": %lld, \"slot_frames\": %lld, "
                "\"slot_groups\": %lld, \"slot_tiles\": %d, \"slot_chains\": %d, \"slot_lim_jobs\": %d, \"n_sb_total\": %lld, "
                "\"split_tile\": %d, \"kw_tile_sb\": %d, \"lim_keep\": %d, \"any_limiter\": %d, \"any_tp\": %d, \"n_att_tables\": %zu}",
                lay.n_slots, (long long)lay.total_frames, (long long)lay.mb_frames, (long long)lay.slot_frames,
                (long long)lay.slot_groups, lay.slot_tiles, lay.slot_chains, lay.slot_lim_jobs, (long long)lay.n_sb_total,
                lay.split_tile, lay.kw_tile_sb, lay.lim_keep, (int)lay.any_limiter, (int)lay.any_tp, jobs.att.size() / 32769);
    auto range = [](const JobRange &r) { std::printf("[%d,%d]", r.lo, r.n); };
    array("waves", lay.waves, [&](const Wave &w) {
        std::printf("%d,%d,%lld,%lld,%lld,%lld,%d,%d,%d,", w.track_lo, w.track_hi, (long long)w.frame_lo, (long long)w.frame_hi,
                    (long long)w.seg_lo, (long long)w.seg_hi, w.slot, (int)w.limiter, (int)w.true_peak);
        for (const JobRange *r : {&w.eq, &w.split, &w.chain, &w.wf, &w.mb_chunks, &w.kw, &w.gain, &w.lim}) {
            range(*r);
            if (r != &w.lim) std::printf(",");
        }
    });
    array("tracks", lay.tracks, [](const ame_track_params &t) {
        std::printf("%d,%d,%d", t.comp[0].table, t.comp[1].table, t.comp[2].table);
    });
    for (const auto &kv : {std::make_pair("mb_offset", &lay.mb_offset), std::make_pair("mb_delta", &jobs.mb_delta)}) {
        std::printf(",\n\"%s\": [", kv.first);
        for (size_t i = 0; i < kv.second->size(); ++i) std::printf(i ? ",%lld" : "%lld", (long long)(*kv.second)[i]);
        std::printf("]");
    }
    array("tdev", lay.tdev, [](const TrackDev &d) {
        std::printf("%lld,%d,%d,%d,%d,%lld,%d", (long long)d.sb_offset, d.n_sb, d.s100, d.first_block, d.lim_tile0,
                    (long long)d.n_total, d.lim_shift);
    });
    auto tile = [](const TileJob &j) {
        std::printf("%lld,%lld,%lld,%d,%d", (long long)j.chunk_begin, (long long)j.tile_begin, (long long)j.tile_end, j.track, j.variant);
    };
    array("eq", jobs.eq, tile);
    array("split", jobs.split, tile);
    array("chain", jobs.chain, [](const ChainJob &c) {
        std::printf("%lld,%lld,%lld,%d,%d,%u,%d,%d", (long long)c.mb_begin, (long long)c.n, (long long)c.grp_begin, c.band, c.table,
                    c.thr_i, c.look, c.tile0);
    });
    array("wf", jobs.wf, [](const WfJob &j) {
        std::printf("%lld,%lld,%lld,%lld,%d,%d,%u,%d", (long long)j.tile_begin, (long long)j.plane_off, (long long)j.n,
                    (long long)j.grp_begin, j.chain, j.look, j.thr_i, j.tile0);
    });
    array("mb_chunks", jobs.mb_chunks, [](const MbChunk &c) {
        std::printf("%lld,%lld,%lld,%lld,%lld,%lld,%lld,%d", (long long)c.abs_begin, (long long)c.mb_begin, (long long)c.n,
                    (long long)c.seg_prefix, (long long)c.grp_begin[0], (long long)c.grp_begin[1], (long long)c.grp_begin[2], c.track);
    });
    array("kw", jobs.kw, [](const KwJob &j) { std::printf("%d,%d,%d", j.track, j.sb_begin, j.sb_end); });
    auto gain = [](const GainJob &j) { std::printf("%lld,%lld,%d", (long long)j.begin, (long long)j.end, j.track); };
    array("gain", jobs.gain, gain);
    array("lim", jobs.lim, gain);
    std::printf("}\n");
    return 0;
}
