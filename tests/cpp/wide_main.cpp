// A caller of the C++ class that opts into a disparity range above the default limit with the extension overload
// Initialize(width, height, option, max_disparity_range), built against this repo's include/ and lib by the test-suite.
//   wide_main left.bgr right.bgr W H dmin dmax out.f32
// The three-argument Initialize must refuse the range; the overload with a limit of 512 must accept it, Match, and keep
// the limit through Reset (the map after Reset must be the same).  The GPU test checks the written map against the oracle.
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>

#include "ADCensusStereo.h"

static bool read_file(const char* path, std::vector<uint8>& buf) {
    FILE* f = std::fopen(path, "rb");
    if (!f) return false;
    const size_t n = std::fread(buf.data(), 1, buf.size(), f);
    std::fclose(f);
    return n == buf.size();
}

int main(int argc, char** argv) {
    if (argc < 8) return 2;
    const sint32 width = std::atoi(argv[3]), height = std::atoi(argv[4]);
    ADCensusOption option;
    option.min_disparity = std::atoi(argv[5]);
    option.max_disparity = std::atoi(argv[6]);
    std::vector<uint8> left((size_t)width * height * 3), right((size_t)width * height * 3);
    if (!read_file(argv[1], left) || !read_file(argv[2], right)) return 20;
    std::vector<float32> disparity((size_t)width * height, -1.0f), again((size_t)width * height, -2.0f);
    ADCensusStereo stereo;
    if (stereo.Initialize(width, height, option)) return 11;                 // above the default limit: refused
    if (!stereo.Initialize(width, height, option, 512)) return 12;
    if (!stereo.Match(left.data(), right.data(), disparity.data())) return 13;
    if (!stereo.Reset(width, height, option)) return 14;                     // keeps the limit of 512
    if (!stereo.Match(left.data(), right.data(), again.data())) return 15;
    if (std::memcmp(disparity.data(), again.data(), disparity.size() * sizeof(float32)) != 0) return 16;
    FILE* f = std::fopen(argv[7], "wb");
    if (!f || std::fwrite(disparity.data(), sizeof(float32), disparity.size(), f) != disparity.size()) return 21;
    std::fclose(f);
    std::printf("WIDE_OK\n");
    return 0;
}
