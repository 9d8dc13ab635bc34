// Writes the compressor attenuation tables that build_layout uploads (build_att_table) as raw AttEntry[32769] records
// (tests/test_compressor_exact.py).  Built with g++ alone, like plan_layout_driver.cpp.
//   att_table_driver OUT THRESH_RMS COEF ATTACK_FRAMES RELEASE_FRAMES [THRESH_RMS COEF ATTACK_FRAMES RELEASE_FRAMES ...]
// Every number is read with strtod, so hexadecimal floats carry the exact doubles of design.track_params.
#include <cstdio>
#include <cstdlib>
#include <vector>

#include "../audio_mastering_engine_b200/csrc/ame_layout.h"

using namespace ame;

int main(int argc, char **argv) {
    if (argc < 6 || (argc - 2) % 4) {
        std::fprintf(stderr, "usage: %s OUT THRESH_RMS COEF ATTACK_FRAMES RELEASE_FRAMES [...]\n", argv[0]);
        return 2;
    }
    FILE *f = std::fopen(argv[1], "wb");
    if (!f) return 2;
    std::vector<AttEntry> e(32769);
    for (int a = 2; a < argc; a += 4) {
        ame_comp_band c{};
        c.thresh_rms = std::strtod(argv[a], nullptr);
        c.coef = std::strtod(argv[a + 1], nullptr);
        c.attack_frames = std::strtod(argv[a + 2], nullptr);
        c.release_frames = std::strtod(argv[a + 3], nullptr);
        build_att_table(e.data(), c);
        if (std::fwrite(e.data(), sizeof(AttEntry), e.size(), f) != e.size()) return 1;
    }
    return std::fclose(f) ? 1 : 0;
}
