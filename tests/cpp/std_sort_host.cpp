// Host build of the device's restatement of std::sort (dsdtm_b200/csrc/std_sort.cuh) next to g++'s own std::sort, on the corner
// record and the comparator of Feature_detector::detect (ref: src/Feature_detection.cpp:111). Test infrastructure.
#include <algorithm>
#include <cstdint>

#include "../../dsdtm_b200/csrc/std_sort.cuh"

struct Corner { int32_t x, y, level; float score; };     // orc_corner / dsdtm_corner

static bool score_desc(const Corner& a, const Corner& b) { return b.score < a.score; }

extern "C" {
void prod_sort_corners(Corner* c, long n) { dsdtm::std_sort(c, n, score_desc); }
void ref_sort_corners(Corner* c, long n) { std::sort(c, c + n, score_desc); }
}
