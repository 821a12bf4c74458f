// Host harness for tests/test_goal_lidar_cpu.py: the goal_lidar routine the optional-key env kernels call
// (mobrob_b200/csrc/env_point.cuh) compiled for the HOST.
//   in : int64 count | per case: double ex, ey, max_dist (<= 0: None), exp_gain, num_bins, alias
//   out: per case: float block[num_bins]
#include <vector>

#include "../../mobrob_b200/csrc/env_point.cuh"

namespace mr {
void set_error(const char*, ...) {}
void count_launch(uint64_t) {}
}  // namespace mr

int main(int argc, char** argv) {
    if (argc < 3) return 2;
    FILE* fi = fopen(argv[1], "rb");
    FILE* fo = fopen(argv[2], "wb");
    if (!fi || !fo) return 3;
    int64_t count;
    if (fread(&count, 8, 1, fi) != 1) return 4;
    std::vector<float> block;
    for (int64_t c = 0; c < count; ++c) {
        double v[6];
        if (fread(v, 8, 6, fi) != 6) return 4;
        const mr::LidarCfg cfg = mr::make_lidar_cfg((int)v[4], v[2], v[3], (int)v[5]);
        block.assign((size_t)cfg.num_bins, -1.f);   // every entry must be written
        mr::goal_lidar(block.data(), v[0], v[1], cfg);
        fwrite(block.data(), 4, block.size(), fo);
    }
    fclose(fo);
    return 0;
}
