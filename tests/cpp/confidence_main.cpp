// A caller of the C++ class that asks for per-pixel confidence with the extension MatchWithConfidence, built against this
// repo's include/ and lib by the test-suite.
//   confidence_main left.bgr right.bgr W H dmax out_prefix
// Writes out_prefix.{disp,origin,best,second} (float32 / uint8 / float32 / float32, W*H each).  The map must equal the one
// Match gives, and the call with all three side-output pointers null must give it too.  Without a device it checks the
// truth table only and prints CONFIDENCE_NO_GPU.
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "ADCensusStereo.h"

static bool read_file(const char* path, std::vector<uint8>& buf) {
    FILE* f = std::fopen(path, "rb");
    if (!f) return false;
    const size_t n = std::fread(buf.data(), 1, buf.size(), f);
    std::fclose(f);
    return n == buf.size();
}

static bool write_file(const std::string& path, const void* p, size_t bytes) {
    FILE* f = std::fopen(path.c_str(), "wb");
    if (!f) return false;
    const bool ok = std::fwrite(p, 1, bytes, f) == bytes;
    std::fclose(f);
    return ok;
}

int main(int argc, char** argv) {
    if (argc < 7) return 2;
    const sint32 width = std::atoi(argv[3]), height = std::atoi(argv[4]);
    const size_t n = (size_t)width * height;
    ADCensusOption option;
    option.max_disparity = std::atoi(argv[5]);
    std::vector<uint8> left(n * 3), right(n * 3), origin(n, 0xee);
    std::vector<float32> disp(n, -1.0f), plain(n, -2.0f), bare(n, -3.0f), best(n, -4.0f), second(n, -5.0f);
    if (!read_file(argv[1], left) || !read_file(argv[2], right)) return 20;
    ADCensusStereo stereo;
    // before Initialize, like Match
    if (stereo.MatchWithConfidence(left.data(), right.data(), disp.data(), origin.data(), best.data(), second.data())) return 10;
    if (!stereo.Initialize(width, height, option)) {
        std::printf("CONFIDENCE_NO_GPU\n");
        return 0;
    }
    if (stereo.MatchWithConfidence(nullptr, right.data(), disp.data(), origin.data(), best.data(), second.data())) return 11;
    if (stereo.MatchWithConfidence(left.data(), right.data(), nullptr, origin.data(), best.data(), second.data())) return 12;
    if (!stereo.MatchWithConfidence(left.data(), right.data(), disp.data(), origin.data(), best.data(), second.data())) return 13;
    if (!stereo.Match(left.data(), right.data(), plain.data())) return 14;
    if (std::memcmp(disp.data(), plain.data(), n * sizeof(float32)) != 0) return 15;
    if (!stereo.MatchWithConfidence(left.data(), right.data(), bare.data(), nullptr, nullptr, nullptr)) return 16;
    if (std::memcmp(bare.data(), plain.data(), n * sizeof(float32)) != 0) return 17;
    const std::string pre = argv[6];
    if (!write_file(pre + ".disp", disp.data(), n * 4) || !write_file(pre + ".origin", origin.data(), n) ||
        !write_file(pre + ".best", best.data(), n * 4) || !write_file(pre + ".second", second.data(), n * 4))
        return 21;
    std::printf("CONFIDENCE_OK\n");
    return 0;
}
