// keyframe_chain_oracle.cpp -- TEST INFRASTRUCTURE: the CPU restatement of the key-frame half of the batched chain (dsdtm_batch_run
// flags 15), built from the oracle's primitives and compiled together with oracle/dsdtm_oracle.cpp into tests/cpp/_build
// (tests/keyframe_chain.py). Tracking::CraeteKeyframe (ref: src/Tracking.cpp:412-464) on a tracked frame, per pair:
//   Set_ExistingFeatures (ref: src/Feature_detection.cpp:43-50): byte int(px.y / (float)cell) * grid_cols + int(px.x / (float)cell) per
//     match; an index outside the grid is skipped and counted in occ_skipped;
//   the mask: orc_circle_fill at cvRound(px) with radius cell_size for every match (SearchLocalPoints, ref: src/Feature_alignment.cpp:
//     100-113), then radius min_dist for every match (Frame::Set_Mask, ref: src/Frame.cpp:286-298; skipped without matches);
//   detect(cur, thr) (ref: src/Feature_detection.cpp:69-154): orc_detect_cells on the cur pyramid with the occupancy, nothing when
//     max_fts - n_matches <= 0 (the early return), else orc_detect_select (g++'s std::sort); tied = 1 when two cells above 20 share a score;
//   the new features' lift: orc_undistort_points, orc_feature_normal, orc_feature_depth on the float depth (orc_depth_convert of the
//     16-bit image; none = -1), orc_unproject with the pose after PoseOptimization.
// matches: n_pairs x 200; cur_imgs: n_pairs level-0 images; depth16: n_pairs images or NULL, has_depth: n_pairs flags or NULL;
// want: n_pairs flags or NULL (= all). corners / lifted: n_pairs x max_fts, rows past n_new zero.
#include <cstring>
#include <thread>
#include <vector>

#include "../../oracle/dsdtm_oracle.h"

typedef struct {
    int32_t point;
    float   px[2];
    int32_t level;
} orc_match;

typedef struct {
    float   px[2];
    float   depth;
    int32_t status;          // 1 = OK, 2 = no depth (the values of DSDTM_LIFT_*)
    double  normal[3];
    double  point_w[3];
} orc_lifted;

extern "C" {

int orc_keyframe_chain(const orc_cam* cam, int levels, int cell_size, int min_dist, int max_fts, float thr, const float dist[5],
                       float depth_scale, int n_pairs, const uint8_t* cur_imgs, const orc_match* matches, const int* n_matches,
                       const double* poses, const uint16_t* depth16, const int* has_depth, const uint8_t* want, int n_threads,
                       int* n_new, orc_corner* corners, orc_lifted* lifted, uint8_t* tied, int* occ_skipped)
{
    const int W = cam->width, Hh = cam->height;
    const int rows = (Hh + cell_size - 1) / cell_size, cols = (W + cell_size - 1) / cell_size, n_cells = rows * cols;
    const size_t npx = (size_t)W * Hh;
    std::memset(corners, 0, (size_t)n_pairs * max_fts * sizeof(orc_corner));
    std::memset(lifted, 0, (size_t)n_pairs * max_fts * sizeof(orc_lifted));
    auto work = [&](int t) {
        std::vector<uint8_t> occ(n_cells), mask(npx);
        std::vector<orc_corner> cells(n_cells);
        std::vector<float> depth(npx);
        int ws[16], hs[16], offs[16];
        int total = 0;
        for (int l = 0, w = W, h = Hh; l < levels; ++l, w = (w + 1) / 2, h = (h + 1) / 2) total += w * h;
        std::vector<uint8_t> pyr(total);
        for (int i = t; i < n_pairs; i += n_threads) {
            n_new[i] = 0; tied[i] = 0; occ_skipped[i] = 0;
            if (want && !want[i]) continue;
            const orc_match* M = matches + (size_t)i * 200;
            const int nm = n_matches[i];
            std::fill(occ.begin(), occ.end(), (uint8_t)0);
            for (int m = 0; m < nm; ++m) {
                const long long k = (long long)(int)(M[m].px[1] / (float)cell_size) * cols + (int)(M[m].px[0] / (float)cell_size);
                if (k >= 0 && k < n_cells) occ[k] = 1;
                else ++occ_skipped[i];
            }
            std::fill(mask.begin(), mask.end(), (uint8_t)255);
            for (int m = 0; m < nm; ++m) orc_circle_fill(mask.data(), W, Hh, W, orc_cvround(M[m].px[0]), orc_cvround(M[m].px[1]), cell_size, 0);
            for (int m = 0; m < nm; ++m) orc_circle_fill(mask.data(), W, Hh, W, orc_cvround(M[m].px[0]), orc_cvround(M[m].px[1]), min_dist, 0);
            if (max_fts - nm <= 0) continue;                                        // ref: src/Feature_detection.cpp:71-72
            orc_pyramid(cur_imgs + (size_t)i * npx, W, Hh, levels, pyr.data(), offs, ws, hs);
            orc_detect_cells(pyr.data(), offs, ws, hs, levels, W, Hh, cell_size, occ.data(), (double)thr, cells.data());
            for (int a = 0; a < n_cells && !tied[i]; ++a)
                for (int b = a + 1; b < n_cells; ++b)
                    if (cells[a].score > 20 && cells[a].score == cells[b].score) { tied[i] = 1; break; }
            orc_corner* C = corners + (size_t)i * max_fts;
            const int added = orc_detect_select(cells.data(), n_cells, mask.data(), W, Hh, cell_size, max_fts, nm, C);
            n_new[i] = added;
            const bool hd = depth16 && (!has_depth || has_depth[i]);
            if (hd) orc_depth_convert(depth16 + (size_t)i * npx, (int)npx, depth_scale, depth.data());
            for (int q = 0; q < added; ++q) {
                orc_lifted& o = lifted[(size_t)i * max_fts + q];
                const float px[2] = { (float)C[q].x, (float)C[q].y };
                orc_undistort_points(cam, dist, px, 1, o.px);
                orc_feature_normal(cam, o.px, o.normal);
                o.depth = hd ? orc_feature_depth(depth.data(), W, Hh, o.px) : -1.0f;
                o.status = 2;
                if (!(o.depth < 0.f)) {
                    orc_unproject(cam, poses + 7 * (size_t)i, o.px, o.depth, o.point_w);
                    o.status = 1;
                }
            }
        }
    };
    if (n_threads <= 1) { work(0); return 0; }
    std::vector<std::thread> th;
    for (int t = 0; t < n_threads; ++t) th.emplace_back(work, t);
    for (auto& t : th) t.join();
    return 0;
}

}  // extern "C"
