// Host harness for tests/test_device_perm_host_cpu.py: the keyed Feistel bijection of mr_device_permutations
// (mobrob_b200/csrc/perm.cuh, the functions device_perm_kernel / device_rows_kernel call) evaluated on the CPU.
//   argv: seed stream n out.bin   ->   int64 perm[n]
#include <stdlib.h>

#include <vector>

#include "../../mobrob_b200/csrc/perm.cuh"

namespace mr {
void set_error(const char*, ...) {}
void count_launch(uint64_t) {}
}  // namespace mr

int main(int argc, char** argv) {
    if (argc < 5) return 2;
    const uint64_t seed = strtoull(argv[1], nullptr, 10), stream = strtoull(argv[2], nullptr, 10);
    const int64_t n = strtoll(argv[3], nullptr, 10);
    FILE* fo = fopen(argv[4], "wb");
    if (!fo || n <= 0) return 3;
    const mr::PermKey K = mr::make_perm_key(seed, stream, n);
    std::vector<int64_t> out((size_t)n);
    for (int64_t i = 0; i < n; ++i) out[i] = (int64_t)mr::perm_index((uint32_t)i, n, K);
    fwrite(out.data(), 8, out.size(), fo);
    fclose(fo);
    return 0;
}
