// Runs build_layout on the host and prints the output meter's part of the layout as JSON (tests/test_output_meter.py).
// Built with g++ alone, like plan_layout_driver.cpp.
//   meter_layout_driver TRACKS OPTIONS N_SM OCC_EQ OCC_SPLIT
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
    std::printf(",\n\"scalars\": {\"any_meter\": %d, \"meter_sb_total\": %lld, \"kw_tile_sb\": %d}", (int)lay.any_meter,
                (long long)lay.meter_sb_total, lay.kw_tile_sb);
    array("waves", lay.waves, [](const Wave &w) {
        std::printf("%d,%d,%d,%d,%d,%d,%d,%d,%d,%d", w.track_lo, w.track_hi, w.kw_uni ? 1 : 0, w.kw.n, w.meter_kw.lo, w.meter_kw.n,
                    w.meter_peak.lo, w.meter_peak.n, w.meter_tracks.lo, w.meter_tracks.n);
    });
    array("tdev", lay.tdev, [](const TrackDev &d) { std::printf("%lld,%d,%d", (long long)d.sb_offset, d.n_sb, d.s100); });
    array("meter_tdev", lay.meter_tdev, [](const TrackDev &d) { std::printf("%lld,%d,%d", (long long)d.sb_offset, d.n_sb, d.s100); });
    array("meter_kw", jobs.meter_kw, [](const KwJob &j) { std::printf("%d,%d,%d", j.track, j.sb_begin, j.sb_end); });
    array("meter_peak", jobs.meter_peak, [](const GainJob &j) { std::printf("%lld,%lld,%d", (long long)j.begin, (long long)j.end, j.track); });
    std::printf(",\n\"meter_tracks\": [");
    for (size_t i = 0; i < jobs.meter_tracks.size(); ++i) std::printf(i ? ",%d" : "%d", jobs.meter_tracks[i]);
    std::printf("]}\n");
    return 0;
}
