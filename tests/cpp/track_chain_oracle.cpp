// track_chain_oracle.cpp -- TEST INFRASTRUCTURE: the CPU restatement of the whole tracked-pose chain (dsdtm_batch_run flags 7), built
// from the oracle's primitives and compiled together with oracle/dsdtm_oracle.cpp into tests/cpp/_build (tests/track_select.py).
// Tracking::TrackWithLocalMap behind the batched refinement chain (ref: src/Tracking.cpp:219-236): orc_pair_batch_map, then per pair
// SearchLocalPoints' greedy selection over the records (ref: src/Feature_alignment.cpp:71-121: cells in index order, candidates by found
// count descending, stable; mask test at cvRound of the float projection; gates; the first converged candidate wins and paints a filled
// circle of radius cell_size on a full-size mask; 200 matches end it), Frame::Add_Feature's bearing (orc_feature_normal) and
// orc_pose_optimization from T_c2r * T_ref. found = n_pairs x points_per_pair (NULL = all 1). matches / res_norm: n_pairs x 200.
#include <algorithm>
#include <thread>
#include <vector>

#include "../../oracle/dsdtm_oracle.h"

typedef struct {
    int32_t point;
    float   px[2];
    int32_t level;
} orc_match;

extern "C" {

int orc_pair_batch_track(const orc_cam* cam, int levels, int cell_size, const uint8_t* ref_pyrs, const uint8_t* cur_imgs, int n_pairs,
                         const orc_ref_feat* feats, int feats_per_pair, const int* n_feats, const double* ref_centers,
                         const double* poses_ref, const double* poses_in, int max_level, int min_level, int max_iters,
                         int points_per_pair, int max_search_level, int align_iters, const int* found, int ba_iters, int n_threads,
                         double* poses_out, int* n_tracked, orc_reproj* reproj, double* poses_track, int* n_matches,
                         orc_match* matches, double* res_norm, orc_ba_summary* summaries)
{
    orc_pair_batch_map(cam, levels, cell_size, ref_pyrs, cur_imgs, n_pairs, feats, feats_per_pair, n_feats, ref_centers, poses_ref, poses_in,
                       max_level, min_level, max_iters, points_per_pair, max_search_level, align_iters, n_threads, poses_out, n_tracked, reproj);
    const int W = cam->width, Hh = cam->height, K = 200;
    const int n_cells = ((W + cell_size - 1) / cell_size) * ((Hh + cell_size - 1) / cell_size);
    auto work = [&](int t) {
        std::vector<uint8_t> mask((size_t)W * Hh);
        std::vector<std::vector<int>> cells(n_cells);
        for (int i = t; i < n_pairs; i += n_threads) {
            const orc_reproj* R = reproj + (size_t)i * points_per_pair;
            const int* F = found ? found + (size_t)i * points_per_pair : nullptr;
            for (auto& c : cells) c.clear();
            for (int j = 0; j < points_per_pair; ++j)                                   // ReprojectPoint's insertion order
                if (R[j].cell >= 0) cells[R[j].cell].push_back(j);
            std::fill(mask.begin(), mask.end(), (uint8_t)255);                          // a new Frame's mImgMask
            orc_match* M = matches + (size_t)i * K;
            int n = 0;
            for (int cell = 0; cell < n_cells && n < K; ++cell) {                       // ref: :75-82
                std::vector<int>& c = cells[cell];
                std::stable_sort(c.begin(), c.end(), [&](int a, int b) { return (F ? F[a] : 1) > (F ? F[b] : 1); });   // std::list::sort
                for (int j : c) {
                    const orc_reproj& r = R[j];
                    if (mask[(size_t)orc_cvround((float)r.px_proj[1]) * W + orc_cvround((float)r.px_proj[0])] != 255) continue;   // ref: :92
                    if ((r.flags & 6) != 6 || r.level < 0 || !(r.flags & 8)) continue;  // Get_ClosetObs / IsInImage gate / FindMatchDirect
                    const float p[2] = { (float)r.px[0], (float)r.px[1] };
                    M[n].point = j; M[n].px[0] = p[0]; M[n].px[1] = p[1]; M[n].level = r.level;
                    orc_circle_fill(mask.data(), W, Hh, W, orc_cvround(p[0]), orc_cvround(p[1]), cell_size, 0);
                    ++n;
                    break;
                }
            }
            n_matches[i] = n;
            // Optimizer::PoseOptimization over the new frame's features (ref: src/Optimizer.cpp:46-68), from cur.Get_Pose() after Run
            std::vector<double> nm(3 * (size_t)n), pw(3 * (size_t)n);
            std::vector<int> lv(n);
            const orc_ref_feat* Fe = feats + (size_t)i * feats_per_pair;
            for (int k = 0; k < n; ++k) {
                orc_feature_normal(cam, M[k].px, &nm[3 * (size_t)k]);
                for (int q = 0; q < 3; ++q) pw[3 * (size_t)k + q] = Fe[M[k].point].point_w[q];
                lv[k] = M[k].level;
            }
            double pose_cur[7];
            orc_se3_mul(poses_out + 7 * (size_t)i, poses_ref + 7 * (size_t)i, pose_cur);
            orc_pose_optimization(n, nm.data(), lv.data(), pw.data(), pose_cur, ba_iters, poses_track + 7 * (size_t)i,
                                  res_norm ? res_norm + (size_t)i * K : nullptr, summaries ? summaries + i : nullptr);
        }
    };
    if (n_threads <= 1) { work(0); return 0; }
    std::vector<std::thread> th;
    for (int t = 0; t < n_threads; ++t) th.emplace_back(work, t);
    for (auto& t : th) t.join();
    return 0;
}


}  // extern "C"
