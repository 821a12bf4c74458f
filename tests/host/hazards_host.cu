// Host harness for tests/test_hazards_cpu.py: the hazard routines the env kernels call (mobrob_b200/csrc/env_point.cuh:
// hazard_layout, hazards_lidar, hazard_cost) compiled for the HOST.  Reads float64 records from argv[1], writes float64
// results to argv[2]:
//   0 layout : seed num keepout n_loc loc[n_loc][2]          -> ok heading hazards[num][2]
//   1 lidar  : num hazards[num][2] m[6] px py pz bins max_dist exp_gain alias -> block[bins]
//   2 cost   : num hazards[num][2] x y size cost indicator   -> cost
#include <vector>

#include "../../mobrob_b200/csrc/env_point.cuh"

namespace mr {
void set_error(const char*, ...) {}
void count_launch(uint64_t) {}
}  // namespace mr

static FILE *fi, *fo;
static double rd() { double v = 0; if (fread(&v, 8, 1, fi) != 1) exit(4); return v; }
static void wr(double v) { fwrite(&v, 8, 1, fo); }

int main(int argc, char** argv) {
    if (argc < 3) return 2;
    fi = fopen(argv[1], "rb");
    fo = fopen(argv[2], "wb");
    if (!fi || !fo) return 3;
    double mode;
    while (fread(&mode, 8, 1, fi) == 1) {
        if (mode == 0) {
            const uint32_t seed = (uint32_t)(int64_t)rd();
            const int num = (int)rd();
            const double keepout = rd();
            const int n_loc = (int)rd();
            std::vector<double> box(4 * num);
            for (int h = 0; h < num; ++h) {   // the boxes mr_env_set_hazards forms
                if (h < n_loc) {
                    const double x = rd(), y = rd(), k = keepout + 1e-9;
                    box[4 * h] = (x - k) + keepout; box[4 * h + 1] = (y - k) + keepout;
                    box[4 * h + 2] = (x + k) - keepout; box[4 * h + 3] = (y + k) - keepout;
                } else {
                    box[4 * h] = -2.0 + keepout; box[4 * h + 1] = -2.0 + keepout;
                    box[4 * h + 2] = 2.0 - keepout; box[4 * h + 3] = 2.0 - keepout;
                }
            }
            mr::HazardCfg c{};
            c.num = num; c.keepout = keepout; c.box = box.data();
            std::vector<double2> pos(num > 0 ? num : 1);
            double heading = 0.0;
            const bool ok = mr::hazard_layout(seed, c, pos.data(), heading);
            wr(ok ? 1.0 : 0.0);
            wr(heading);
            for (int h = 0; h < num; ++h) { wr(pos[h].x); wr(pos[h].y); }
        } else if (mode == 1) {
            const int num = (int)rd();
            std::vector<double2> pos(num);
            for (auto& p : pos) { p.x = rd(); p.y = rd(); }
            double m[6];
            for (double& v : m) v = rd();
            const double px = rd(), py = rd(), pz = rd();
            const int bins = (int)rd();
            const double max_dist = rd(), gain = rd();
            const int alias = (int)rd();
            const mr::LidarCfg lc = mr::make_lidar_cfg(bins, max_dist, gain, alias);
            std::vector<float> block(bins, -1.f);
            mr::hazards_lidar(block.data(), pos.data(), num, m, px, py, pz, lc);
            for (float v : block) wr(v);
        } else {
            const int num = (int)rd();
            std::vector<double2> pos(num);
            for (auto& p : pos) { p.x = rd(); p.y = rd(); }
            const double x = rd(), y = rd();
            mr::HazardCfg c{};
            c.num = num; c.size = rd(); c.cost = rd();
            c.flags = mr::HAZ_CONSTRAIN | (rd() != 0 ? mr::HAZ_INDICATOR : 0u);
            wr(mr::hazard_cost(c, pos.data(), x, y));
        }
    }
    fclose(fo);
    return 0;
}
