// dsdtm_host.cpp -- bodies of the reference's front-end classes as marshalling + C-ABI calls (see dsdtm_host.h).
#include "dsdtm_host.h"

#if defined(__SSE2__)
#include <emmintrin.h>
#endif
#include <algorithm>
#include <cstdlib>
#include <chrono>
#include <cstring>
#include <unordered_map>
#include <mutex>
#include <fstream>
#include <sstream>
#include <stdexcept>

namespace DSDTM {

// ================================================================================================ value types
int cvRound(double v) { return (int)std::nearbyint(v); }

SE3::SE3() { p[0] = 1; for (int i = 1; i < 7; ++i) p[i] = 0; }
SE3::SE3(const double q[7]) { std::memcpy(p, q, sizeof p); }

static void quat_rot(const double* q, const double* v, double* o)   // Eigen _transformVector
{
    double uv[3] = { q[2] * v[2] - q[3] * v[1], q[3] * v[0] - q[1] * v[2], q[1] * v[1] - q[2] * v[0] };
    uv[0] += uv[0]; uv[1] += uv[1]; uv[2] += uv[2];
    const double c[3] = { q[2] * uv[2] - q[3] * uv[1], q[3] * uv[0] - q[1] * uv[2], q[1] * uv[1] - q[2] * uv[0] };
    for (int i = 0; i < 3; ++i) o[i] = v[i] + q[0] * uv[i] + c[i];
}

SE3 SE3::operator*(const SE3& o) const   // translation_ += so3_*o.translation_; so3_ *= o.so3_ (normalised)
{
    SE3 r;
    double rt[3];
    quat_rot(p, o.p + 4, rt);
    for (int i = 0; i < 3; ++i) r.p[4 + i] = p[4 + i] + rt[i];
    const double aw = p[0], ax = p[1], ay = p[2], az = p[3], bw = o.p[0], bx = o.p[1], by = o.p[2], bz = o.p[3];
    double q[4] = { aw * bw - ax * bx - ay * by - az * bz, aw * bx + ax * bw + ay * bz - az * by,
                    aw * by + ay * bw + az * bx - ax * bz, aw * bz + az * bw + ax * by - ay * bx };
    const double n = std::sqrt(q[1] * q[1] + q[2] * q[2] + q[3] * q[3] + q[0] * q[0]);
    for (int i = 0; i < 4; ++i) r.p[i] = q[i] / n;
    return r;
}

SE3 SE3::inverse() const
{
    SE3 r;
    r.p[0] = p[0]; r.p[1] = -p[1]; r.p[2] = -p[2]; r.p[3] = -p[3];
    const double nt[3] = { p[4] * -1., p[5] * -1., p[6] * -1. };
    quat_rot(r.p, nt, r.p + 4);
    return r;
}

Vector3d SE3::operator*(const Vector3d& v) const
{
    double o[3];
    quat_rot(p, v.v, o);
    return Vector3d(o[0] + p[4], o[1] + p[5], o[2] + p[6]);
}

SE3 SE3::exp(const double x[6])
{
    const double* om = x + 3;
    const double theta = std::sqrt(om[0] * om[0] + om[1] * om[1] + om[2] * om[2]);
    SE3 r;
    double imag;
    if (theta < 1e-10) { const double t2 = theta * theta; imag = 0.5 - 0.0208333 * t2 + 0.000260417 * t2 * t2; }
    else imag = std::sin(0.5 * theta) / theta;
    double q[4] = { std::cos(0.5 * theta), imag * om[0], imag * om[1], imag * om[2] };
    const double n = std::sqrt(q[0] * q[0] + q[1] * q[1] + q[2] * q[2] + q[3] * q[3]);
    for (int i = 0; i < 4; ++i) r.p[i] = q[i] / n;
    const double O[9] = { 0, -om[2], om[1], om[2], 0, -om[0], -om[1], om[0], 0 };
    double V[9];
    if (theta < 1e-10) {
        const double w = r.p[0], a = r.p[1], b = r.p[2], c = r.p[3];
        const double R[9] = { 1 - 2 * (b * b + c * c), 2 * (a * b - w * c), 2 * (a * c + w * b), 2 * (a * b + w * c), 1 - 2 * (a * a + c * c),
                              2 * (b * c - w * a), 2 * (a * c - w * b), 2 * (b * c + w * a), 1 - 2 * (a * a + b * b) };
        std::memcpy(V, R, sizeof V);
    } else {
        double O2[9];
        for (int i = 0; i < 3; ++i) for (int j = 0; j < 3; ++j) { double s = 0; for (int k = 0; k < 3; ++k) s += O[3 * i + k] * O[3 * k + j]; O2[3 * i + j] = s; }
        const double t2 = theta * theta, a = (1 - std::cos(theta)) / t2, b = (theta - std::sin(theta)) / (t2 * theta);
        for (int i = 0; i < 9; ++i) V[i] = ((i % 4 == 0) ? 1.0 : 0.0) + a * O[i] + b * O2[i];
    }
    for (int i = 0; i < 3; ++i) r.p[4 + i] = V[3 * i] * x[0] + V[3 * i + 1] * x[1] + V[3 * i + 2] * x[2];
    return r;
}

// Image-sized buffers are recycled: a fresh 300 KB allocation per mask per frame is an mmap plus ~75 page faults (about 20 us each
// time), which the per-frame constructors would pay three times over.
namespace {
struct BufPool {
    std::mutex m;
    std::unordered_map<size_t, std::vector<std::vector<uchar>*>> idle;
    static BufPool& get() { static BufPool* p = new BufPool; return *p; }     // never destroyed: buffers may outlive static teardown
    std::shared_ptr<std::vector<uchar>> take(size_t n)
    {
        std::vector<uchar>* v = nullptr;
        if (n >= 4096) {
            std::lock_guard<std::mutex> g(m);
            auto& l = idle[n];
            if (!l.empty()) { v = l.back(); l.pop_back(); }
        }
        if (!v) v = new std::vector<uchar>(n);
        return std::shared_ptr<std::vector<uchar>>(v, [n](std::vector<uchar>* q) {
            BufPool& p = BufPool::get();
            std::lock_guard<std::mutex> g(p.m);
            auto& l = p.idle[n];
            if (n >= 4096 && l.size() < 16) l.push_back(q); else delete q;
        });
    }
};
}  // namespace

Mat8::Mat8(int rows_, int cols_, uchar fill) : rows(rows_), cols(cols_), step(cols_)
{
    store = BufPool::get().take((size_t)rows * cols);
    data = store->data();
    std::memset(data, fill, (size_t)rows * cols);
}

Mat8::Mat8(int rows_, int cols_, const uchar* src, int src_step) : rows(rows_), cols(cols_), step(cols_)
{
    store = BufPool::get().take((size_t)rows * cols);
    data = store->data();
    for (int y = 0; y < rows; ++y) std::memcpy(data + (size_t)y * cols, src + (size_t)y * src_step, cols);
}

// cv::circle(img, center, radius, color, -1): OpenCV's filled midpoint circle (checked against cv2 goldens in tests/)
void circle(Mat8& img, Point2f center, int radius, uchar color)
{
    const int cx = cvRound(center.x), cy = cvRound(center.y), w = img.cols, h = img.rows;
    auto span = [&](int y, int x0, int x1) {
        if (y < 0 || y >= h) return;
        x0 = std::max(x0, 0); x1 = std::min(x1, w - 1);
        if (x0 <= x1) std::memset(img.data + (size_t)y * img.step + x0, color, (size_t)(x1 - x0 + 1));
    };
    int err = 0, dx = radius, dy = 0, plus = 1, minus = (radius << 1) - 1;
    while (dx >= dy) {
        span(cy - dy, cx - dx, cx + dx); span(cy + dy, cx - dx, cx + dx);
        span(cy - dx, cx - dy, cx + dy); span(cy + dx, cx - dy, cx + dy);
        dy++; err += plus; plus += 2;
        const int mask = (err <= 0) - 1;
        err -= minus & mask; dx += mask; minus -= mask & 2;
    }
}

// ================================================================================================ Config
std::map<std::string, std::string>& Config::table() { static std::map<std::string, std::string> t; return t; }
void Config::Clear() { table().clear(); }
void Config::Set(const std::string& k, const std::string& v) { table()[k] = v; }
bool Config::Has(const std::string& k) { return table().count(k) != 0; }

void Config::setParameterFile(const std::string& path)
{
    std::ifstream f(path);
    if (!f) throw std::runtime_error("Config: parameter file " + path + " does not exist");   // ref: src/Config.cpp:17-21
    std::string line;
    while (std::getline(f, line)) {
        const size_t hash = line.find('#');
        if (hash != std::string::npos) line = line.substr(0, hash);
        if (line.empty() || line[0] == '%' || line.compare(0, 3, "---") == 0) continue;
        // unresolved merge-conflict markers of the shipped kinect.yaml (SURVEY D5) are skipped; the later block wins
        if (line.compare(0, 7, "<<<<<<<") == 0 || line.compare(0, 7, "=======") == 0 || line.compare(0, 7, ">>>>>>>") == 0) continue;
        const size_t colon = line.find(':');
        if (colon == std::string::npos) continue;
        auto trim = [](std::string s) { const char* ws = " \t\r\n\""; s.erase(0, s.find_first_not_of(ws)); s.erase(s.find_last_not_of(ws) + 1); return s; };
        const std::string k = trim(line.substr(0, colon)), v = trim(line.substr(colon + 1));
        if (!k.empty() && !v.empty()) table()[k] = v;
    }
}

template <> int Config::Get<int>(const std::string& k)
{
    auto it = table().find(k);
    if (it == table().end()) return 0;   // cv::FileStorage yields 0 for a missing node
    return (int)std::strtod(it->second.c_str(), nullptr);
}
template <> float Config::Get<float>(const std::string& k) { auto it = table().find(k); return it == table().end() ? 0.f : (float)std::strtod(it->second.c_str(), nullptr); }
template <> double Config::Get<double>(const std::string& k) { auto it = table().find(k); return it == table().end() ? 0.0 : std::strtod(it->second.c_str(), nullptr); }
template <> std::string Config::Get<std::string>(const std::string& k) { auto it = table().find(k); return it == table().end() ? std::string() : it->second; }

// ================================================================================================ Camera
Camera::Camera()
{
    mf = Config::Get<float>("Camera.f");
    mfx = Config::Get<float>("Camera.fx"); mfy = Config::Get<float>("Camera.fy");
    mcx = Config::Get<float>("Camera.cx"); mcy = Config::Get<float>("Camera.cy");
    mwidth = Config::Get<int>("Camera.width"); mheight = Config::Get<int>("Camera.height");
    mk1 = Config::Has("Camera.k1") ? Config::Get<float>("Camera.k1") : 0.f; mk2 = Config::Has("Camera.k2") ? Config::Get<float>("Camera.k2") : 0.f;
    mp1 = Config::Has("Camera.p1") ? Config::Get<float>("Camera.p1") : 0.f; mp2 = Config::Has("Camera.p2") ? Config::Get<float>("Camera.p2") : 0.f;
    mk3 = Config::Has("Camera.k3") ? Config::Get<float>("Camera.k3") : 0.f;
}

Vector2d Camera::Camera2Pixel(const Vector3d& P) const { return Vector2d(mfx * P[0] / P[2] + mcx, mfy * P[1] / P[2] + mcy); }
Vector3d Camera::Pixel2Camera(const Point2f& pt, const float& depth) const
{
    return Vector3d(depth * (pt.x - mcx) / mfx, depth * (pt.y - mcy) / mfy, depth);   // float arithmetic, then widened (Q8)
}
Vector3d Camera::Pixel2Camera(const Vector2d& pt, const float& depth) const
{
    return Vector3d(depth * (pt(0) - mcx) / mfx, depth * (pt(1) - mcy) / mfy, depth);
}
bool Camera::IsInImage(const Point2f p, int b, int level) const
{
    return cvRound(p.x) >= b && cvRound(p.x) < mwidth / (1 << level) - b && cvRound(p.y) >= b && cvRound(p.y) < mheight / (1 << level) - b;
}

// ================================================================================================ GPU runtime
static GpuRuntime* g_runtime = nullptr;

GpuRuntime& GpuRuntime::Instance()
{
    if (!g_runtime) g_runtime = new GpuRuntime();
    return *g_runtime;
}
void GpuRuntime::Shutdown() { delete g_runtime; g_runtime = nullptr; }

GpuRuntime::GpuRuntime()
{
    dsdtm_cam cam;
    cam.width = Config::Get<int>("Camera.width"); cam.height = Config::Get<int>("Camera.height");
    cam.fx = Config::Get<float>("Camera.fx"); cam.fy = Config::Get<float>("Camera.fy");
    cam.cx = Config::Get<float>("Camera.cx"); cam.cy = Config::Get<float>("Camera.cy");
    cam.f = Config::Get<float>("Camera.f");
    dsdtm_params prm;
    prm.levels = mLevels = Config::Get<int>("Camera.MaxPyraLevels");
    prm.cell_size = Config::Get<int>("Camera.CellSize");
    const int max_fts = std::max(Config::Get<int>("Camera.Max_fts"), 16);
    prm.max_feats = std::min(std::max(max_fts, 64), DSDTM_MAX_FEATS_LIMIT);
    const int rows = (cam.height + prm.cell_size - 1) / std::max(prm.cell_size, 1), cols = (cam.width + prm.cell_size - 1) / std::max(prm.cell_size, 1);
    prm.max_patches = std::max(4 * rows * cols, 1024);      // speculative batch of every reprojected candidate
    prm.max_frames = mMaxFrames = Config::Has("Gpu.MaxFrames") ? Config::Get<int>("Gpu.MaxFrames") : 32;
    prm.max_batch = 1;
    mCtx = dsdtm_create(Config::Has("Gpu.Device") ? Config::Get<int>("Gpu.Device") : 0, &cam, &prm);
    if (!mCtx) throw std::runtime_error(std::string("DSDTM GPU front end unavailable (no CPU fallback): ") + dsdtm_create_error());
    mOwner.assign(mMaxFrames, nullptr);
    mStamp.assign(mMaxFrames, 0);
}

GpuRuntime::~GpuRuntime()
{
    for (auto* o : mOwner) if (o) o->slot = -1;
    if (mCtx) dsdtm_destroy(mCtx);
}

int GpuRuntime::Acquire(GpuSlot* owner)
{
    int best = -1;
    for (int i = 0; i < mMaxFrames; ++i) if (!mOwner[i]) { best = i; break; }
    if (best < 0) {   // evict the least recently used pyramid; its owner re-uploads on next use
        for (int i = 0; i < mMaxFrames; ++i) if (best < 0 || mStamp[i] < mStamp[best]) best = i;
        if (mStamp[best] > mEpochStart) mEpochEvicted = true;      // a slot handed out inside the current epoch was recycled
        mOwner[best]->slot = -1;
    }
    mOwner[best] = owner;
    mStamp[best] = ++mClock;
    return best;
}

void GpuRuntime::Release(int slot) { if (slot >= 0 && slot < mMaxFrames) mOwner[slot] = nullptr; }

std::shared_ptr<GpuSlot> GpuRuntime::Upload(const Mat8& img, uint8_t* levels_out)
{
    auto s = std::make_shared<GpuSlot>(img);
    s->slot = Acquire(s.get());
    // no host copies wanted: queue the copy + pyramid and return; every later call on the context is ordered after them
    const int rc = levels_out ? dsdtm_frame_upload_pyramid_host(mCtx, s->slot, s->host.data, s->host.step, levels_out)
                              : dsdtm_frame_upload_pyramid_async(mCtx, s->slot, s->host.data, s->host.step);
    if (rc != 0) throw std::runtime_error(std::string("dsdtm_frame_upload_pyramid: ") + dsdtm_last_error(mCtx));
    return s;
}

std::shared_ptr<GpuSlot> GpuRuntime::UploadLevel(const Mat8& img, int level)
{
    auto s = std::make_shared<GpuSlot>(Mat8());                   // no host copy: the handle lives for one call and is never re-uploaded
    s->slot = Acquire(s.get());
    if (dsdtm_frame_upload_level(mCtx, s->slot, level, img.data, img.step) != 0)
        throw std::runtime_error(std::string("dsdtm_frame_upload_level: ") + dsdtm_last_error(mCtx));
    return s;
}

int GpuRuntime::Resident(const std::shared_ptr<GpuSlot>& s)
{
    if (s->slot >= 0) { mStamp[s->slot] = ++mClock; return s->slot; }
    s->slot = Acquire(s.get());
    if (dsdtm_frame_upload_pyramid(mCtx, s->slot, s->host.data, s->host.step) != 0)
        throw std::runtime_error(std::string("dsdtm_frame_upload_pyramid: ") + dsdtm_last_error(mCtx));
    return s->slot;
}

GpuSlot::~GpuSlot() { if (g_runtime && slot >= 0) g_runtime->Release(slot); }

// ================================================================================================ Frame / KeyFrame / MapPoint
unsigned long Frame::mlNextId = 0;

Frame::Frame(CameraPtr cam, const Mat8& gray, double ts) : mCamera(cam), mdCloTimestamp(ts), mColorImg(gray)
{
    mlId = mlNextId++;                                            // ref: src/Frame.cpp:30,39
    mPyra_levels = Config::Get<int>("Camera.MaxPyraLevels");      // ref: src/Frame.cpp:51-52
    mMin_Dist = Config::Get<int>("Camera.Min_dist");
    mvImg_Pyr.resize(mPyra_levels);
    ComputeImagePyramid(mColorImg, mvImg_Pyr);                    // ref: :55
    mImgMask = Mat8(mCamera->mheight, mCamera->mwidth, 255);      // ref: :64-65
    mDynamicMask = Mat8(mCamera->mheight, mCamera->mwidth, 0);
}

Frame::~Frame() { if (g_runtime && g_runtime->DepthOwner() == this) g_runtime->SetDepthOwner(nullptr); }

void Frame::ComputeImagePyramid(const Mat8 image, PyrLevels& pyr)   // ref: src/Frame.cpp:74-81
{
    GpuRuntime& rt = GpuRuntime::Instance();
    pyr.Set(0, image);                                            // level 0 aliases the caller's image
    // H2D + pyrDown chain on the device. The GPU stages never read host copies of levels 1..; mvImg_Pyr[l] fetches one on first use.
    mGpu = rt.Upload(image);
    pyr.Bind(mGpu);
}

void PyrLevels::Bind(const std::shared_ptr<GpuSlot>& g)
{
    gpu = g;
    for (size_t l = 1; l < m.size(); ++l) pending[l] = 1;
}

void PyrLevels::Fetch(size_t l) const
{
    GpuRuntime& rt = GpuRuntime::Instance();
    int w = 0, h = 0; size_t off = 0;
    dsdtm_level_info(rt.ctx(), (int)l, &w, &h, &off);
    Mat8 img(h, w, 0);
    const int slot = rt.Resident(gpu);                            // re-uploads and rebuilds the pyramid if the slot was recycled
    if (dsdtm_frame_download_level(rt.ctx(), slot, (int)l, img.data) != 0)
        throw std::runtime_error(std::string("dsdtm_frame_download_level: ") + dsdtm_last_error(rt.ctx()));
    m[l] = img; pending[l] = 0;
}

void Frame::Add_Feature(Feature* f, bool normal)                  // ref: src/Frame.cpp:83-92
{
    if (normal) { f->mNormal = mCamera->Pixel2Camera(f->mpx, 1.0f); f->mNormal.normalize(); }
    mvFeatures.push_back(f);
}

void Frame::Set_Pose(const SE3& pose)                             // ref: src/Frame.cpp:167-174
{
    mT_c2w = pose;
    mOw = mT_c2w.inverse().translation();
}

Vector2d Frame::World2Pixel(const Vector3d& p) const { return mCamera->Camera2Pixel(mT_c2w * p); }   // ref: :318-323

// ---- RGB-D keyframe path. One depth slot is enough: only the frame that is becoming a keyframe needs its depth on the device.
void Frame::SetDepth(const uint16_t* depth, int stride_bytes, float depth_scale)
{
    GpuRuntime& rt = GpuRuntime::Instance();
    if (dsdtm_depth_upload(rt.ctx(), 0, depth, stride_bytes) != 0)
        throw std::runtime_error(std::string("dsdtm_depth_upload: ") + dsdtm_last_error(rt.ctx()));
    rt.SetDepthOwner(this);
    mHasDepth = true; mDepthScale = depth_scale;
}

void Frame::UndistortFeatures()                                   // ref: src/Frame.cpp:94-150 (+ :152-157, :200-224 for the cache)
{
    GpuRuntime& rt = GpuRuntime::Instance();
    const int n = (int)mvFeatures.size();
    mvMapPoints.resize(n);
    if (n == 0) { mLifted.clear(); return; }
    if (mHasDepth && rt.DepthOwner() != this)
        throw std::runtime_error("Frame::UndistortFeatures: the depth slot now holds another frame's depth (call SetDepth again)");
    std::vector<float> px((size_t)2 * n);
    std::vector<uint8_t> initial(n);
    for (int i = 0; i < n; ++i) { px[2 * i] = mvFeatures[i]->mpx.x; px[2 * i + 1] = mvFeatures[i]->mpx.y; initial[i] = mvFeatures[i]->mbInitial; }
    const float dist[5] = { mCamera->mk1, mCamera->mk2, mCamera->mp1, mCamera->mp2, mCamera->mk3 };
    mLifted.assign(n, dsdtm_lifted{});
    if (dsdtm_keyframe_lift(rt.ctx(), mHasDepth ? 0 : -1, mT_c2w.data(), dist, mDepthScale, px.data(), initial.data(), n, mLifted.data()) != 0)
        throw std::runtime_error(std::string("dsdtm_keyframe_lift: ") + dsdtm_last_error(rt.ctx()));
    for (int i = 0; i < n; ++i) {
        if (mvFeatures[i]->mbInitial) continue;                  // ref: :140-141
        mvFeatures[i]->mpx = Point2f(mLifted[i].px[0], mLifted[i].px[1]);
        mvFeatures[i]->mNormal = Vector3d(mLifted[i].normal[0], mLifted[i].normal[1], mLifted[i].normal[2]);
    }
}

float Frame::Get_FeatureDetph(const Feature* feature)             // ref: src/Frame.cpp:176-198
{
    for (size_t i = 0; i < mvFeatures.size() && i < mLifted.size(); ++i)
        if (mvFeatures[i] == feature) {
            if (mLifted[i].status == DSDTM_LIFT_SKIPPED) break;
            return mLifted[i].depth;
        }
    throw std::runtime_error("Frame::Get_FeatureDetph: feature was not lifted (call UndistortFeatures after SetDepth; mbInitial features are skipped as in the reference)");
}

Vector3d Frame::UnProject(const Point2f px, const float d) { return mT_c2w.inverse() * mCamera->Pixel2Camera(px, d); }   // ref: :152-157

void Frame::Set_Mask()                                            // ref: src/Frame.cpp:286-298
{
    for (size_t k = 0; k < mvFeatures.size(); ++k)
        if (k < mvMapPoints.size() && mvMapPoints[k]) circle(mImgMask, mvFeatures[k]->mpx, mMin_Dist, 0);
    // cv::threshold(mDynamicMask, 200, 255, THRESH_BINARY) and the saturating mImgMask - mDynamicMask as ONE pass over the two images
    // (16 pixels per step; the per-pixel scalar form cost 380 us per key frame at 640x480)
    const size_t n = (size_t)std::min(mDynamicMask.rows * mDynamicMask.cols, mImgMask.rows * mImgMask.cols);
    uchar* d = mDynamicMask.data;
    uchar* m = mImgMask.data;
    size_t i = 0;
#if defined(__SSE2__)
    const __m128i bias = _mm_set1_epi8((char)0x80), thr = _mm_set1_epi8((char)(200 ^ 0x80));
    for (; i + 16 <= n; i += 16) {
        const __m128i dv = _mm_loadu_si128(reinterpret_cast<const __m128i*>(d + i));
        const __m128i bin = _mm_cmpgt_epi8(_mm_xor_si128(dv, bias), thr);               // unsigned d > 200 ? 0xFF : 0
        _mm_storeu_si128(reinterpret_cast<__m128i*>(d + i), bin);
        const __m128i mv = _mm_loadu_si128(reinterpret_cast<const __m128i*>(m + i));
        _mm_storeu_si128(reinterpret_cast<__m128i*>(m + i), _mm_subs_epu8(mv, bin));
    }
#endif
    for (; i < n; ++i) {
        d[i] = d[i] > 200 ? 255 : 0;
        m[i] = (uchar)std::max((int)m[i] - (int)d[i], 0);         // saturating subtraction
    }
}

KeyFrame::KeyFrame(Frame* f) : mvImg_Pyr(f->mvImg_Pyr), mvFeatures(f->mvFeatures), mGpu(f->mGpu) { Set_Pose(f->Get_Pose()); }
void KeyFrame::Set_Pose(const SE3& p) { mT_c2w = p; mOw = mT_c2w.inverse().translation(); }

// change queue of the device-resident map store: positions (bundle adjustment) and bad flags (PoseOptimization's EraseFound) reach
// the device at the next Map::Sync(); a mutex because LocalMapping may move points from its own thread
MapPoint::DenseState* MapPoint::sDense = nullptr;
static std::mutex g_touched_mutex;
static std::vector<MapPoint*> g_touched;
void MapPoint::Touch()
{
    if (mStoreId < 0) return;
    std::unique_lock<std::mutex> l(g_touched_mutex);
    if (!mTouched) { mTouched = true; g_touched.push_back(this); }
}
void MapPoint::DrainTouched(std::vector<MapPoint*>& out)
{
    std::unique_lock<std::mutex> l(g_touched_mutex);
    out.swap(g_touched);
    g_touched.clear();
    for (MapPoint* m : out) m->mTouched = false;
}

bool MapPoint::Get_ClosetObs(const Frame* frame, Feature*& feature, KeyFrame*& kf) const   // ref: src/MapPoint.cpp:133-174
{
    if (mObservations.empty()) return false;
    const Vector3d pose = Get_Pose();
    Vector3d dir = frame->Get_CameraCnt() - pose;
    dir.normalize();
    double best = 0;
    auto best_it = mObservations.begin();
    for (auto it = mObservations.begin(); it != mObservations.end(); ++it) {
        Vector3d d = it->first->Get_CameraCnt() - pose;
        d.normalize();
        const double c = d.dot(dir);
        if (c > best) { best = c; best_it = it; }
    }
    feature = best_it->first->mvFeatures[best_it->second];
    kf = best_it->first;
    return !(best < 0.5);
}

// ================================================================================================ Feature_detector
Feature_detector::Feature_detector()                              // ref: src/Feature_detection.cpp:10-21
{
    mCell_size = Config::Get<int>("Camera.CellSize");
    mPyr_levels = Config::Get<int>("Camera.MaxPyraLevels");
    mMax_fts = Config::Get<int>("Camera.Max_fts");
    mImg_width = Config::Get<int>("Camera.width");
    mImg_height = Config::Get<int>("Camera.height");
    mGrid_rows = (int)std::ceil(1.0 * mImg_height / mCell_size);
    mGrid_cols = (int)std::ceil(1.0 * mImg_width / mCell_size);
    mvGrid_occupy.resize((size_t)mGrid_rows * mGrid_cols, false);
}

void Feature_detector::Set_ExistingFeatures(const Features& features)      // ref: :43-50
{
    mvGrid_occupy.assign((size_t)mGrid_rows * mGrid_cols, false);
    for (Feature* f : features)
        mvGrid_occupy[(size_t)static_cast<int>(f->mpx.y / mCell_size) * mGrid_cols + static_cast<int>(f->mpx.x / mCell_size)] = true;
}

void Feature_detector::Set_ExistingFeatures(const std::vector<Point2f>& features)   // ref: :52-62 (note the cast placement)
{
    mvGrid_occupy.assign((size_t)mGrid_rows * mGrid_cols, false);
    for (const Point2f& f : features)
        mvGrid_occupy.at((size_t)(static_cast<int>((f.y / mCell_size) * mGrid_cols) + static_cast<int>(f.x / mCell_size))) = true;
}

void Feature_detector::ResetGrid() { std::fill(mvGrid_occupy.begin(), mvGrid_occupy.end(), false); }

void Feature_detector::detect(Frame* frame, const double detection_threshold, const bool)   // ref: :69-154
{
    if ((int)frame->mvFeatures.size() >= mMax_fts) return;
    const bool timing = getenv("DSDTM_HOST_TIMING") != nullptr;
    const auto T0 = std::chrono::steady_clock::now();
    if (frame->mvFeatures.size() > 0) frame->Set_Mask();          // ref: :120-123
    const auto T1 = std::chrono::steady_clock::now();
    GpuRuntime& rt = GpuRuntime::Instance();
    const int slot = rt.Resident(frame->mGpu);
    const int n = mGrid_rows * mGrid_cols;
    std::vector<uint8_t> occ(n);
    for (int i = 0; i < n; ++i) occ[i] = mvGrid_occupy[i] ? 1 : 0;
    // mImgMask as Set_Mask and SearchLocalPoints left it (an empty Mat = nothing painted; rows are copied dense if strided)
    const Mat8& m = frame->mImgMask;
    std::vector<uint8_t> dense;
    const uint8_t* mask = nullptr;
    if (!m.empty()) {
        mask = m.data;
        if (m.step != m.cols) {
            dense.resize((size_t)m.rows * m.cols);
            for (int y = 0; y < m.rows; ++y) std::memcpy(dense.data() + (size_t)y * m.cols, m.data + (size_t)y * m.step, m.cols);
            mask = dense.data();
        }
    }
    const int max_new = mMax_fts - (int)frame->mvFeatures.size();
    std::vector<dsdtm_corner> sel(max_new);
    int n_sel = 0;
    // levels loop + FAST + non-max + Shi-Tomasi + per-cell best, the unstable std::sort and the mask-circle walk on the device (ref: :76-150)
    if (dsdtm_detect(rt.ctx(), slot, (float)detection_threshold, occ.data(), mask, nullptr, 0, max_new, sel.data(), &n_sel, nullptr) != 0)
        throw std::runtime_error(std::string("dsdtm_detect: ") + dsdtm_last_error(rt.ctx()));
    const auto T2 = std::chrono::steady_clock::now();
    for (int i = 0; i < n_sel; ++i)                               // ref: :145
        frame->Add_Feature(new Feature(frame, Point2f((float)sel[i].x, (float)sel[i].y), sel[i].level), 0);
    ResetGrid();
    frame->mImgMask.release();                                    // ref: :152-153
    if (timing) {
        const auto T3 = std::chrono::steady_clock::now();
        auto us = [](std::chrono::steady_clock::time_point a, std::chrono::steady_clock::time_point b) { return std::chrono::duration<double, std::micro>(b - a).count(); };
        fprintf(stderr, "detect: Set_Mask %.1f us, device detect %.1f us, Add_Feature %.1f us\n", us(T0, T1), us(T1, T2), us(T2, T3));
    }
}

// ================================================================================================ Map / Tracking (local-map selection)
void Map::Pack(KeyFrame* kf, dsdtm_map_kf& row, std::vector<double>& pts) const
{
    const Vector3d t = kf->Get_Pose().translation();
    for (int k = 0; k < 3; ++k) row.t[k] = t[k];
    for (Feature* f : kf->mvFeatures) {                          // KeyFrame::mvMapPoints is parallel to the features (ref: src/Keyframe.cpp:11-19)
        Vector3d P(0, 0, 0);                                     // null map point: the zero row the kernel skips (ref: src/Tracking.cpp:324-328)
        if (f->Mpt) P = f->Mpt->Get_Pose();
        pts.push_back(P[0]); pts.push_back(P[1]); pts.push_back(P[2]);
    }
}

Map::~Map()
{
    for (MapPoint* m : mStorePoints) m->mStoreId = -1;
    if (MapPoint::sDense == &mDense) MapPoint::sDense = nullptr;
    for (KeyFrame* k : mvKeyFrames) { k->mStoreRow = -1; k->mStoreSlot = -1; }
    if (g_runtime && (mStoreKfs > 0 || !mStorePoints.empty())) dsdtm_store_clear(g_runtime->ctx());
    if (g_runtime && g_runtime->TrackingMap() == this) g_runtime->SetTrackingMap(nullptr);
}

void Map::AddKeyFrame(KeyFrame* kf)
{
    if (mIndex.count(kf)) return;
    mIndex[kf] = (int)mvKeyFrames.size();
    mvKeyFrames.push_back(kf);
    mRows.push_back(Rows{ mPoints, (int)kf->mvFeatures.size() });
    mPoints += (int)kf->mvFeatures.size();
}

void Map::MarkMoved(KeyFrame* kf)
{
    auto it = mIndex.find(kf);
    if (it != mIndex.end() && it->second < mUploadedKfs) mPending.push_back(it->second);
    if (kf->mStoreRow >= 0) mStoreMoved.push_back(kf);
}

// The device-resident map store (dsdtm_store_*): new key frames append their rows (their map points first), touched map points and
// moved key frames are rewritten, and a key frame whose pyramid was evicted from the frame pool is re-uploaded (the store holds slots).
void Map::SyncStore()
{
    GpuRuntime& rt = GpuRuntime::Instance();
    dsdtm_ctx* ctx = rt.ctx();
    auto check = [&](int rc, const char* what) { if (rc != 0) throw std::runtime_error(std::string(what) + ": " + dsdtm_last_error(ctx)); };
    rt.BeginEpoch();
    for (int i = mStoreKfs; i < (int)mvKeyFrames.size(); ++i) {
        KeyFrame* kf = mvKeyFrames[i];
        std::vector<double> pos; std::vector<int32_t> bad;
        const int first = (int)mStorePoints.size();
        for (Feature* f : kf->mvFeatures)
            if (f->Mpt && f->Mpt->mStoreId < 0) {
                f->Mpt->mStoreId = (int)mStorePoints.size();
                mStorePoints.push_back(f->Mpt);
                mDense.found.push_back(f->Mpt->Get_FoundNums()); mDense.bad.push_back(f->Mpt->IsBad() ? 1 : 0);
                MapPoint::sDense = &mDense;
                const Vector3d P = f->Mpt->Get_Pose();
                pos.push_back(P[0]); pos.push_back(P[1]); pos.push_back(P[2]);
                bad.push_back(f->Mpt->IsBad() ? 1 : 0);
            }
        if (!bad.empty()) check(dsdtm_store_set_points(ctx, first, (int)bad.size(), pos.data(), bad.data()), "dsdtm_store_set_points");
        dsdtm_store_kf row{};
        row.slot = rt.Resident(kf->mGpu);
        const SE3 T = kf->Get_Pose();
        const Vector3d O = kf->Get_CameraCnt();
        for (int k = 0; k < 7; ++k) row.pose_c2w[k] = T.data()[k];
        for (int k = 0; k < 3; ++k) row.center[k] = O[k];
        std::vector<dsdtm_store_feat> feats(kf->mvFeatures.size());
        for (size_t j = 0; j < feats.size(); ++j) {
            const Feature* f = kf->mvFeatures[j];
            dsdtm_store_feat& o = feats[j];
            o.mp = f->Mpt ? f->Mpt->mStoreId : -1;
            o.level = f->mlevel; o.px[0] = f->mpx.x; o.px[1] = f->mpx.y;
            for (int k = 0; k < 3; ++k) o.normal[k] = f->mNormal[k];
            o.is_obs = (f->Mpt && f->Mpt->HasObservation(kf, j)) ? 1 : 0;
            o.next_obs = -1;
        }
        int32_t r = -1;
        check(dsdtm_store_append_keyframe(ctx, &row, feats.data(), (int)feats.size(), &r), "dsdtm_store_append_keyframe");
        kf->mStoreRow = r; kf->mStoreSlot = row.slot;
        ++mVersion;
    }
    mStoreKfs = (int)mvKeyFrames.size();
    std::vector<MapPoint*> touched;
    MapPoint::DrainTouched(touched);
    if (!touched.empty()) {
        std::vector<int32_t> ids, bad; std::vector<double> pos;
        for (MapPoint* m : touched) {
            if (m->mStoreId < 0) continue;
            const Vector3d P = m->Get_Pose();
            ids.push_back(m->mStoreId); bad.push_back(m->IsBad() ? 1 : 0);
            pos.push_back(P[0]); pos.push_back(P[1]); pos.push_back(P[2]);
        }
        if (!ids.empty()) { check(dsdtm_store_update_points(ctx, ids.data(), (int)ids.size(), pos.data(), bad.data()), "dsdtm_store_update_points"); ++mVersion; }
    }
    // every key frame's pyramid must be resident under the slot the store names (touching it also keeps it young in the LRU pool)
    for (KeyFrame* kf : mvKeyFrames) {
        const int slot = rt.Resident(kf->mGpu);
        const bool moved = std::find(mStoreMoved.begin(), mStoreMoved.end(), kf) != mStoreMoved.end();
        if (slot != kf->mStoreSlot || moved) {
            const SE3 T = kf->Get_Pose();
            const Vector3d O = kf->Get_CameraCnt();
            double c3[3] = { O[0], O[1], O[2] };
            check(dsdtm_store_set_keyframe(ctx, kf->mStoreRow, slot, T.data(), c3), "dsdtm_store_set_keyframe");
            kf->mStoreSlot = slot;
            ++mVersion;
        }
    }
    mStoreMoved.clear();
    if (!rt.SlotsStillValid())
        throw std::runtime_error("Map::SyncStore: frame pool too small for the key frames of the map (raise Gpu.MaxFrames)");
}

void Map::Sync()
{
    dsdtm_ctx* ctx = GpuRuntime::Instance().ctx();
    std::vector<double> pts;
    auto check = [&](int rc) { if (rc != 0) throw std::runtime_error(std::string("dsdtm_map_table_upload: ") + dsdtm_last_error(ctx)); };
    for (int i : mPending) {                                     // rewritten rows: one key frame at a time (its rows are contiguous)
        dsdtm_map_kf row{ mRows[i].pt_begin, mRows[i].pt_count, { 0, 0, 0 } };
        pts.clear();
        Pack(mvKeyFrames[i], row, pts);
        check(dsdtm_map_table_upload(ctx, i, 1, &row, row.pt_begin, row.pt_count, pts.data()));
    }
    mPending.clear();
    const int n = (int)mvKeyFrames.size();
    if (mUploadedKfs < n) {                                      // appended key frames: one call for all of them
        std::vector<dsdtm_map_kf> rows;
        pts.clear();
        for (int i = mUploadedKfs; i < n; ++i) {
            dsdtm_map_kf row{ mRows[i].pt_begin, mRows[i].pt_count, { 0, 0, 0 } };
            Pack(mvKeyFrames[i], row, pts);
            rows.push_back(row);
        }
        check(dsdtm_map_table_upload(ctx, mUploadedKfs, n - mUploadedKfs, rows.data(), mRows[mUploadedKfs].pt_begin, (int)(pts.size() / 3), pts.data()));
        mUploadedKfs = n;
    }
}

Tracking::Tracking(CameraPtr cam, Map* map) : mMap(map), mFeature_Alignment(new Feature_Alignment(cam)), mCam(cam) { GpuRuntime::Instance().SetTrackingMap(map); }
Tracking::~Tracking() { if (g_runtime && g_runtime->TrackingMap() == mMap) g_runtime->SetTrackingMap(nullptr); delete mFeature_Alignment; }

void Tracking::GetCloseKeyFrames(const Frame* tFrame, std::list<std::pair<KeyFrame*, double>>& tClose_kfs) const   // ref: src/Tracking.cpp:315-345
{
    mMap->Sync();
    const int n = mMap->ReturnKeyFramesSize();
    if (n == 0) return;
    dsdtm_ctx* ctx = GpuRuntime::Instance().ctx();
    static thread_local std::vector<uint8_t> visible;
    static thread_local std::vector<double> dist;
    visible.resize(n); dist.resize(n);
    int32_t n_local = 0;
    if (dsdtm_close_keyframes(ctx, tFrame->Get_Pose().data(), n, 0, visible.data(), dist.data(), nullptr, &n_local) != 0)
        throw std::runtime_error(std::string("dsdtm_close_keyframes: ") + dsdtm_last_error(ctx));
    for (int i = 0; i < n; ++i)
        if (visible[i]) tClose_kfs.push_back(std::make_pair(mMap->Row(i), dist[i]));      // ref: :331-333, in GetAllKeyFrames order
}

bool Tracking::sUseStore = true;
bool Tracking::sSpeculate = true;

// UpdateLocalMap on the device-resident map store: ONE call selects the close key frames, ranks them, visits every map point of the
// ten nearest once, reprojects it and -- for the points that land in the image -- runs Get_ClosetObs, the IsInImage gate,
// SolveAffineMatrix, WarpAffine and Align2D. What comes back is one record per candidate; SearchLocalPoints orders its cells and
// replays the mask-dependent greedy selection. Same candidates, same order, same arithmetic as the host loop below
// (tests: test_update_local_map_device_path_equals_the_host_loop).
void Tracking::UpdateLocalMapOnDevice()
{
    GpuRuntime& rt = GpuRuntime::Instance();
    const auto T0 = std::chrono::steady_clock::now();
    mMap->Sync();
    mMap->SyncStore();
    const auto T1 = std::chrono::steady_clock::now();
    mFeature_Alignment->ResetGrid();
    mvpLocalKeyFrames.clear();
    mvpLocalMapPoints.clear();
    mLastReprojected = 0;
    if (mMap->ReturnKeyFramesSize() == 0) return;
    const SE3 Tc = mCurrentFrame->Get_Pose();
    {   // Run already did this frame's local-map stage with exactly this pose on exactly this map: take its records
        GpuRuntime::Speculation& sp = rt.Spec();
        if (sp.frame == mCurrentFrame.get() && sp.map_version == mMap->Version() && std::memcmp(sp.pose, Tc.data(), sizeof sp.pose) == 0) {
            for (int i = 0; i < sp.n_local; ++i) mvpLocalKeyFrames.push_back(mMap->Row(sp.rows[i]));
            mLastReprojected = sp.n_out;
            sp.frame = nullptr;
            mFeature_Alignment->SetFused(mCurrentFrame.get(), std::move(sp.cands), &mMap->StorePoints(), &mMap->Dense());
            if (getenv("DSDTM_HOST_TIMING")) fprintf(stderr, "UpdateLocalMap(device): records of Run's submission taken (n=%d)\n", mLastReprojected);
            return;
        }
        sp.frame = nullptr;
    }
    const int cur_slot = rt.Resident(mCurrentFrame->mGpu);
    const Vector3d Oc = mCurrentFrame->Get_CameraCnt();
    const double center[3] = { Oc[0], Oc[1], Oc[2] };
    static thread_local std::vector<dsdtm_store_cand> cands;
    const int cap = 4096;
    cands.resize(cap);
    int32_t rows[16], n_local = 0, n_out = 0;
    if (dsdtm_store_track(rt.ctx(), cur_slot, Tc.data(), center, 10, Config::Get<int>("Camera.MaxPyraLevels") - 3, 10, rows, &n_local,
                          cands.data(), cap, &n_out) != 0)
        throw std::runtime_error(std::string("dsdtm_store_track: ") + dsdtm_last_error(rt.ctx()));
    for (int i = 0; i < n_local; ++i) mvpLocalKeyFrames.push_back(mMap->Row(rows[i]));
    cands.resize((size_t)n_out);
    mLastReprojected = n_out;
    std::vector<dsdtm_store_cand> mine(cands.begin(), cands.end());
    mFeature_Alignment->SetFused(mCurrentFrame.get(), std::move(mine), &mMap->StorePoints(), &mMap->Dense());
    if (getenv("DSDTM_HOST_TIMING")) {
        const auto T2 = std::chrono::steady_clock::now();
        auto us = [](std::chrono::steady_clock::time_point a, std::chrono::steady_clock::time_point b) { return std::chrono::duration<double, std::micro>(b - a).count(); };
        fprintf(stderr, "UpdateLocalMap(device): sync %.1f us, dsdtm_store_track %.1f us (n=%d)\n", us(T0, T1), us(T1, T2), n_out);
    }
    // mvpLocalMapPoints (the viewer's list, ref: :299,308-312) is not rebuilt per frame here: nothing on the path reads it
}

void Tracking::UpdateLocalMap()                                   // ref: src/Tracking.cpp:257-313
{
    if (sUseStore) { UpdateLocalMapOnDevice(); return; }
    mFeature_Alignment->ResetGrid();
    std::list<std::pair<KeyFrame*, double>> tClose_kfs;
    GetCloseKeyFrames(mCurrentFrame.get(), tClose_kfs);
    tClose_kfs.sort([](const std::pair<KeyFrame*, double>& a, const std::pair<KeyFrame*, double>& b) { return a.second < b.second; });   // ref: :266-267
    mvpLocalKeyFrames.clear();
    mvpLocalKeyFrames.reserve(10);
    mvpLocalMapPoints.clear();
    mLastReprojected = 0;
    int tNum = 0;
    for (auto iter = tClose_kfs.begin(); iter != tClose_kfs.end() && tNum < 10; iter++, tNum++) {   // ref: :276
        KeyFrame* tKFrame = iter->first;
        mvpLocalKeyFrames.push_back(tKFrame);
        for (Feature* f : tKFrame->mvFeatures) {                  // KeyFrame::GetMapPoints()
            MapPoint* tMp = f->Mpt;
            if (tMp == nullptr) continue;
            if (tMp->IsBad()) continue;
            if (tMp->mLastProjectedFrameId == mCurrentFrame->mlId) continue;
            tMp->mLastProjectedFrameId = mCurrentFrame->mlId;
            if (mFeature_Alignment->ReprojectPoint(mCurrentFrame, tMp)) {
                mvpLocalMapPoints[tMp] = tKFrame;
                mLastReprojected++;
                // ref: :299-300 IsinFrustum + IncreaseVisible feed MapPoint::Get_FoundRatio, which only LocalMapping's culling reads
            }
        }
    }
    // ref: :308-312 SetReferenceMapPoints is the viewer's copy
}

// ================================================================================================ Optimizer
static dsdtm_ba_summary g_last_ba_summary = {};
static std::vector<double> g_last_ba_residuals;
const dsdtm_ba_summary& Optimizer::LastSummary() { return g_last_ba_summary; }
const std::vector<double>& Optimizer::LastResiduals() { return g_last_ba_residuals; }

void Optimizer::PoseOptimization(FramePtr tCurFrame, int /*tIterations: the reference ignores it and sets max_num_iterations = 100*/)
{
    double tReprojectThresh = Config::Get<float>("Optimization.LocalBAthreshhold");   // ref: src/Optimizer.cpp:22-24
    tReprojectThresh = tReprojectThresh / tCurFrame->mCamera->mf;
    const double tOutlineThres = tReprojectThresh;

    // ref: :41-68 -- one residual block per feature with a good, initialised map point, in mvFeatures order; tvMpts is keyed by
    // the FEATURE index (tNum advances on skipped features too)
    // (std::map<int, MapPoint*> in the reference; a vector indexed by the feature number answers tvMpts[i] identically --
    //  a missing key reads as null -- without 200 node allocations per frame)
    static thread_local std::vector<dsdtm_ba_obs> obs;
    static thread_local std::vector<MapPoint*> tvMpts;
    obs.clear(); obs.reserve(tCurFrame->mvFeatures.size());
    tvMpts.assign(tCurFrame->mvFeatures.size(), nullptr);
    int tNum = 0;
    for (auto iter = tCurFrame->mvFeatures.begin(); iter != tCurFrame->mvFeatures.end(); ++iter, ++tNum) {
        if (!(*iter)->Mpt) continue;
        if ((*iter)->Mpt->IsBad()) continue;
        if (!((*iter)->mbInitial)) continue;
        const Vector3d P = (*iter)->Mpt->Get_Pose();             // snapshot under the point's mutex (LocalMapping may move it)
        tvMpts[tNum] = (*iter)->Mpt;
        dsdtm_ba_obs o;
        for (int k = 0; k < 3; ++k) { o.normal[k] = (*iter)->mNormal[k]; o.point_w[k] = P[k]; }
        o.level = (*iter)->mlevel; o.reserved = 0;
        obs.push_back(o);
    }

    dsdtm_ctx* ctx = GpuRuntime::Instance().ctx();
    double pose_out[7];
    g_last_ba_residuals.assign(obs.size(), 0.0);
    const int rc = dsdtm_pose_optimize(ctx, obs.data(), (int)obs.size(), tCurFrame->Get_Pose().data(), 100, pose_out,
                                       g_last_ba_residuals.data(), &g_last_ba_summary);
    if (rc != 0) throw std::runtime_error(std::string("Optimizer::PoseOptimization: ") + dsdtm_last_error(ctx));
    tCurFrame->Set_Pose(SE3(pose_out));                          // ref: :79

    // ref: :81-94, literally: residual i is the i-th residual BLOCK, tvMpts[i] the map point of FEATURE i (std::map::operator[]
    // inserts a null entry for a feature that was skipped) -- the two numberings agree only while no feature is skipped
    const std::vector<double>& tvdResidual = g_last_ba_residuals;
    for (int i = 0; i < (int)tvdResidual.size(); ++i) {
        if (tvdResidual[i] > tOutlineThres) {
            if (!tvMpts[i]) continue;
            if (tvMpts[i]->IsBad()) continue;
            tvMpts[i]->EraseFound();
        }
    }
}

// ================================================================================================ Sprase_ImgAlign
Sprase_ImgAlign::Sprase_ImgAlign(int tMaxLevel, int tMinLevel, int tMaxIterators)
    : mnMaxLevel(tMaxLevel), mnMinLevel(tMinLevel), mnMaxIterators(tMaxIterators)
{
    mnMinfts = Config::Get<int>("Camera.Min_fts");                // ref: src/Sprase_ImageAlign.cpp:14
}

void Sprase_ImgAlign::Reset() { mT_c2r = SE3(); mLog.clear(); }   // ref: src/Sprase_ImageAlign.cpp:22-27 (the device holds no per-run state)

void Sprase_ImgAlign::GetJocabianBA(const Vector3d& p, double J[12]) const   // ref: :169-193
{
    const double x = p[0], y = p[1], z_inv = 1.0 / p[2], z_inv2 = z_inv * z_inv;
    J[0] = -z_inv; J[1] = 0.0; J[2] = x * z_inv2; J[3] = y * J[2]; J[4] = -(1.0 + x * J[2]); J[5] = y * z_inv;
    J[6] = 0.0; J[7] = -z_inv; J[8] = y * z_inv2; J[9] = 1.0 + y * J[8]; J[10] = -x * J[8]; J[11] = -x * z_inv;
}

int Sprase_ImgAlign::Run(FramePtr cur, FramePtr ref)              // ref: src/Sprase_ImageAlign.cpp:29-60
{
    mLog.clear();
    if ((int)ref->mvFeatures.size() < mnMinfts) return 0;         // ref: :34-38 "Too few features to track"
    GpuRuntime& rt = GpuRuntime::Instance();
    // snapshot every map point ONCE on the tracking thread (the mapper moves them under mutex, SURVEY 7 "thread-safety at the seam")
    std::vector<dsdtm_ref_feat>& feats = mFeats;
    feats.clear();
    feats.reserve(ref->mvFeatures.size());
    for (Feature* f : ref->mvFeatures) {
        dsdtm_ref_feat r;
        r.px[0] = f->mpx.x; r.px[1] = f->mpx.y; r.level = f->mlevel; r.initial = f->mbInitial ? 1 : 0;
        for (int k = 0; k < 3; ++k) r.normal[k] = f->mNormal[k];
        const Vector3d P = (f->mbInitial && f->Mpt) ? f->Mpt->Get_Pose() : Vector3d();
        for (int k = 0; k < 3; ++k) r.point_w[k] = P[k];
        feats.push_back(r);
    }
    const SE3 T_c2r = cur->Get_Pose() * ref->Get_Pose().inverse();   // ref: :43
    const Vector3d cen = ref->Get_CameraCnt();
    double pose_out[7];
    int n_tracked = 0, n_log = 0;
    if (mWantLog) mLog.resize(256);
    Map* tmap = (Tracking::sUseStore && Tracking::sSpeculate && !mWantLog) ? rt.TrackingMap() : nullptr;
    if (tmap && tmap->ReturnKeyFramesSize() > 0) {
        // Run + Tracking::UpdateLocalMap in ONE submission (dsdtm_track_frame_store): the tables are brought up to date first, the
        // device composes cur.Set_Pose(T_c2r * ref) itself and runs the local-map stage with it; the records wait in the runtime
        tmap->Sync();
        tmap->SyncStore();
        const int ref_slot = rt.Resident(ref->mGpu), cur_slot = rt.Resident(cur->mGpu);
        dsdtm_track_store_in in{};
        in.ref_slot = ref_slot; in.cur_slot = cur_slot; in.n_feats = (int)feats.size(); in.feats = feats.data();
        const SE3 Tr = ref->Get_Pose();
        for (int k = 0; k < 3; ++k) in.ref_center[k] = cen[k];
        for (int k = 0; k < 7; ++k) { in.pose_ref_c2w[k] = Tr.data()[k]; in.pose_c2r_in[k] = T_c2r.data()[k]; }
        in.max_level = mnMaxLevel; in.min_level = mnMinLevel; in.max_iters = mnMaxIterators;
        in.max_local = 10; in.max_search_level = Config::Get<int>("Camera.MaxPyraLevels") - 3; in.align_iters = 10;
        dsdtm_track_out to{};
        GpuRuntime::Speculation& sp = rt.Spec();
        sp.frame = nullptr;
        const int cap = 4096;
        sp.cands.resize(cap);
        int32_t nl = 0, no = 0;
        if (dsdtm_track_frame_store(rt.ctx(), &in, &to, sp.rows, &nl, sp.cands.data(), cap, &no) != 0)
            throw std::runtime_error(std::string("dsdtm_track_frame_store: ") + dsdtm_last_error(rt.ctx()));
        mLog.clear();
        mT_c2r = SE3(to.pose_c2r);
        cur->Set_Pose(mT_c2r * ref->Get_Pose());                 // ref: :57
        if (std::memcmp(cur->Get_Pose().data(), to.pose_cur_c2w, 7 * sizeof(double)) == 0) {   // the device composed the same bits
            sp.cands.resize((size_t)no);
            sp.n_local = nl; sp.n_out = no; sp.map_version = tmap->Version();
            std::memcpy(sp.pose, to.pose_cur_c2w, sizeof sp.pose);
            sp.frame = cur.get();
        }
        return to.n_tracked;
    }
    const int ref_slot = rt.Resident(ref->mGpu), cur_slot = rt.Resident(cur->mGpu);
    // chunks of max_feats would change the reference's single linear system; the capacity is sized from Camera.Max_fts instead
    if (dsdtm_sparse_align(rt.ctx(), ref_slot, cur_slot, feats.data(), (int)feats.size(), cen.v, T_c2r.data(), mnMaxLevel, mnMinLevel,
                           mnMaxIterators, pose_out, &n_tracked, mWantLog ? mLog.data() : nullptr, mWantLog ? (int)mLog.size() : 0, &n_log) != 0)
        throw std::runtime_error(std::string("dsdtm_sparse_align: ") + dsdtm_last_error(rt.ctx()));
    mLog.resize(std::min<size_t>(n_log, mLog.size()));
    mT_c2r = SE3(pose_out);
    cur->Set_Pose(mT_c2r * ref->Get_Pose());                     // ref: :57
    return n_tracked;                                             // ref: :59
}

// ================================================================================================ Feature_Alignment
struct Feature_Alignment::Prepared {
    dsdtm_candidate c;     // everything SolveAffineMatrix reads, snapshotted on the tracking thread
};

Feature_Alignment::Feature_Alignment(CameraPtr camera) : mCam(camera)   // ref: src/Feature_alignment.cpp:11-44
{
    mMax_pts = Config::Get<int>("Camera.Max_tkfts");
    mPyr_levels = Config::Get<int>("Camera.MaxPyraLevels");
    mCell_size = Config::Get<int>("Camera.CellSize");
    mGrid_Rows = (int)std::ceil(1.0 * mCam->mheight / mCell_size);
    mGrid_Cols = (int)std::ceil(1.0 * mCam->mwidth / mCell_size);
    mCells.resize((size_t)mGrid_Rows * mGrid_Cols);
    for (auto& c : mCells) c = new Cell;
    // the reference also builds a shuffled mCellOrder that it never uses (Q9): cells are visited in index order
}

Feature_Alignment::~Feature_Alignment() { for (auto* c : mCells) delete c; }
void Feature_Alignment::ResetGrid() { for (auto* c : mCells) c->clear(); mFusedFrame = nullptr; mFusedPoints = nullptr; mFused.clear(); }

void Feature_Alignment::SetFused(const Frame* frame, std::vector<dsdtm_store_cand>&& cands, const std::vector<MapPoint*>* points, const MapPoint::DenseState* dense)
{
    mFused = std::move(cands); mFusedFrame = frame; mFusedPoints = points; mFusedDense = dense;
}

// a caller mixes the two styles (UpdateLocalMap on the device, then its own ReprojectPoint calls): rebuild the reference's cell lists
// from the records, in the reference's insertion order, and continue on the host path
void Feature_Alignment::MaterializeFused()
{
    std::vector<const dsdtm_store_cand*> o;
    for (const auto& c : mFused) o.push_back(&c);
    std::sort(o.begin(), o.end(), [](const dsdtm_store_cand* a, const dsdtm_store_cand* b) { return a->order < b->order; });
    for (const dsdtm_store_cand* c : o)
        mCells[c->r.cell]->push_back(Candidate((*mFusedPoints)[c->mp], Vector2d(c->r.px_proj[0], c->r.px_proj[1])));
    mFusedFrame = nullptr; mFusedPoints = nullptr; mFusedDense = nullptr; mFused.clear();
}

// SearchLocalPoints on the records of dsdtm_store_track (ref: :71-121): cells in index order, candidates of a cell by found count
// (std::list::sort is stable: ties keep the order of the ReprojectPoint calls = `order`), first converged candidate whose projection
// is still unmasked wins the cell, its circle masks later candidates, 200 matches end the search.
void Feature_Alignment::SearchFused(FramePtr frame)
{
    const auto T0 = std::chrono::steady_clock::now();
    // bucket the records by cell (counting sort: 1376 cells), then order each cell's few candidates by (found desc, order asc)
    struct Key { int found, order, idx; };
    static thread_local std::vector<Key> keys;
    static thread_local std::vector<int> begin;
    const int n_cells = (int)mCells.size();
    begin.assign((size_t)n_cells + 1, 0);
    for (const dsdtm_store_cand& c : mFused) begin[(size_t)c.r.cell + 1]++;
    for (int i = 0; i < n_cells; ++i) begin[(size_t)i + 1] += begin[(size_t)i];
    keys.resize(mFused.size());
    {
        static thread_local std::vector<int> fill;
        fill.assign(begin.begin(), begin.end() - 1);
        for (size_t i = 0; i < mFused.size(); ++i) {
            const dsdtm_store_cand& c = mFused[i];
            keys[(size_t)fill[(size_t)c.r.cell]++] = Key{ mFusedDense->found[(size_t)c.mp], c.order, (int)i };
        }
    }
    int matches = 0;
    const int gates = DSDTM_LM_OBS_OK | DSDTM_LM_REF_OK;
    for (int cell = 0; cell < n_cells && matches < 200; ++cell) {   // ref: :75-82, the literal 200
        const int b0 = begin[(size_t)cell], b1 = begin[(size_t)cell + 1];
        if (b0 == b1) continue;
        if (b1 - b0 > 1)
            std::sort(keys.begin() + b0, keys.begin() + b1, [](const Key& a, const Key& b) { return a.found != b.found ? a.found > b.found : a.order < b.order; });
        for (int k = b0; k < b1; ++k) {
            const dsdtm_store_cand& c = mFused[(size_t)keys[(size_t)k].idx];
            if (mFusedDense->bad[(size_t)c.mp]) continue;
            if (frame->mImgMask.at(cvRound((float)c.r.px_proj[1]), cvRound((float)c.r.px_proj[0])) != 255) continue;
            if ((c.r.flags & gates) != gates || c.r.level < 0) continue;
            if (!(c.r.flags & DSDTM_LM_CONVERGED)) continue;
            MapPoint* mp = (*mFusedPoints)[(size_t)c.mp];
            mp->IncreaseFound();
            const Point2f p((float)c.r.px[0], (float)c.r.px[1]);
            Feature* f = new Feature(frame.get(), p, c.r.level);
            f->SetPose(mp);
            circle(frame->mImgMask, p, mCell_size, 0);
            frame->Add_Feature(f);
            frame->Add_MapPoint(mp);
            matches++;
            break;                                               // ReprojectCell returns at the first match
        }
    }
    mLastMatches = matches;
    mFusedFrame = nullptr; mFusedPoints = nullptr; mFused.clear();
    if (getenv("DSDTM_HOST_TIMING")) {
        const auto T1 = std::chrono::steady_clock::now();
        fprintf(stderr, "SearchLocalPoints(records): order + replay %.1f us\n", std::chrono::duration<double, std::micro>(T1 - T0).count());
    }
}

bool Feature_Alignment::ReprojectPoint(FramePtr frame, MapPoint* mp)     // ref: :54-69
{
    if (mFusedPoints) MaterializeFused();
    const Vector2d px = frame->World2Pixel(mp->Get_Pose());
    if (mCam->IsInImage(Point2f((float)px(0), (float)px(1)), 8)) {
        const int index = static_cast<int>(px(1) / mCell_size) * mGrid_Cols + static_cast<int>(px(0) / mCell_size);
        mCells[index]->push_back(Candidate(mp, px));
        return true;
    }
    return false;
}

Matrix2d Feature_Alignment::SolveAffineMatrix(KeyFrame* kf, const FramePtr cur, Feature* rf, const MapPoint*)   // ref: :160-190
{
    Matrix2d A;
    const int HalfLarger = mHalf_PatchSize + 1, level = rf->mlevel;
    const Vector3d P = (kf->Get_CameraCnt() - rf->Mpt->Get_Pose()).norm() * rf->mNormal;
    const Point2f rp = rf->mpx;
    const Vector2d pxU(rp.x + HalfLarger * (1 << level), rp.y), pxV(rp.x, rp.y + HalfLarger * (1 << level));
    Vector3d PU = mCam->Pixel2Camera(pxU, 1.0f), PV = mCam->Pixel2Camera(pxV, 1.0f);
    PU.normalize(); PV.normalize();
    PU = PU * (P(2) / PU(2)); PV = PV * (P(2) / PV(2));
    const SE3 T = cur->Get_Pose() * kf->Get_Pose().inverse();
    const Vector2d c = mCam->Camera2Pixel(T * P), cu = mCam->Camera2Pixel(T * PU), cv = mCam->Camera2Pixel(T * PV);
    A(0, 0) = (cu(0) - c(0)) / HalfLarger; A(1, 0) = (cu(1) - c(1)) / HalfLarger;
    A(0, 1) = (cv(0) - c(0)) / HalfLarger; A(1, 1) = (cv(1) - c(1)) / HalfLarger;
    return A;
}

int Feature_Alignment::GetBestSearchLevel(Matrix2d A, int max_level)      // ref: :192-204
{
    int L = 0;
    double D = A.determinant();
    while (D > 3.0 && L < max_level) { L++; D = D * 0.25; }
    return L;
}

// host-side map walk of FindMatchDirect (ref: :128-140): the observation lookup and the two early-outs. The arithmetic that
// follows (SolveAffineMatrix, GetBestSearchLevel, WarpAffine, Align2D) runs on the device: dsdtm_feature_align_batch.
bool Feature_Alignment::Prepare(const MapPoint* mp, const FramePtr frame, const Vector2d& px, Prepared& out)
{
    Feature* rf = nullptr;
    KeyFrame* kf = nullptr;
    if (!mp->Get_ClosetObs(frame.get(), rf, kf)) return false;
    if (!mCam->IsInImage(Point2f(rf->mpx.x / (1 << rf->mlevel), rf->mpx.y / (1 << rf->mlevel)), mHalf_PatchSize + 1, rf->mlevel)) return false;
    dsdtm_candidate& c = out.c;
    c.ref_slot = GpuRuntime::Instance().Resident(kf->mGpu);
    c.ref_level = rf->mlevel;
    c.ref_px[0] = rf->mpx.x; c.ref_px[1] = rf->mpx.y;
    const Vector3d P = rf->Mpt->Get_Pose(), O = kf->Get_CameraCnt();
    const SE3 T = frame->Get_Pose() * kf->Get_Pose().inverse();          // ref: :181
    for (int k = 0; k < 3; ++k) { c.ref_normal[k] = rf->mNormal[k]; c.ref_point_w[k] = P[k]; c.kf_center[k] = O[k]; }
    for (int k = 0; k < 7; ++k) c.pose_c2r[k] = T.data()[k];
    c.px[0] = px[0]; c.px[1] = px[1];
    return true;
}

void Feature_Alignment::SearchLocalPoints(FramePtr frame)                 // ref: :71-121
{
    if (HasFused(frame.get())) { SearchFused(frame); return; }
    if (mFusedPoints) MaterializeFused();
    const auto T0 = std::chrono::steady_clock::now();
    GpuRuntime::Instance().BeginEpoch();
    // The reference walks cells in index order, candidates by found-count, and stops a cell at the first match; a match
    // paints the mask and thereby only changes which LATER candidates are tried, never their alignment result. So: sort
    // the cells (as the reference does, in place), snapshot the map points of all candidates with their observations into
    // flat tables, let the device do Get_ClosetObs + the IsInImage gate + SolveAffineMatrix + WarpAffine + Align2D for all
    // of them in ONE call (dsdtm_local_map_align_batch), then replay the greedy selection in the reference's order.
    GpuRuntime& rt = GpuRuntime::Instance();
    struct Item { Candidate* cand; int index; };               // index into the point table, -1 = IsBad at snapshot time
    // flat, reused across frames: the items of cell ci are items[cell_begin[ci] .. cell_begin[ci + 1])
    static thread_local std::vector<Item> items;
    static thread_local std::vector<int> cell_begin;
    static thread_local std::vector<dsdtm_kf_view> kfs;
    static thread_local std::vector<dsdtm_obs> obs;
    static thread_local std::vector<dsdtm_map_point> pts;
    static thread_local unsigned long long snap_epoch = 0;
    items.clear(); kfs.clear(); obs.clear(); pts.clear();
    cell_begin.assign(mCells.size() + 1, 0);
    ++snap_epoch;
    const int cur_slot_first = rt.Resident(frame->mGpu);     // touch the current frame first: it must stay resident as well
    for (size_t ci = 0; ci < mCells.size(); ++ci) {
        Cell* cell = mCells[ci];
        cell_begin[ci] = (int)items.size();
        if (cell->empty()) continue;
        if (cell->size() > 1)
            cell->sort([](Candidate& a, Candidate& b) { return a.mMpPoint->Get_FoundNums() > b.mMpPoint->Get_FoundNums(); });   // ref: :88,123-126
        for (Candidate& c : *cell) {
            Item it{ &c, -1 };
            if (!c.mMpPoint->IsBad()) {
                dsdtm_map_point mp;
                const Vector3d P = c.mMpPoint->Get_Pose();
                for (int k = 0; k < 3; ++k) mp.point_w[k] = P[k];
                mp.obs_begin = (int)obs.size();
                c.mMpPoint->ForEachObservation([&](KeyFrame* kf, size_t feat) {   // std::map order = the reference's iteration order
                    if (kf->mSnapEpoch != snap_epoch) {
                        dsdtm_kf_view v{};
                        v.slot = rt.Resident(kf->mGpu);
                        const Vector3d O = kf->Get_CameraCnt();
                        const SE3 T = kf->Get_Pose();
                        for (int k = 0; k < 3; ++k) v.center[k] = O[k];
                        for (int k = 0; k < 7; ++k) v.pose_c2w[k] = T.data()[k];
                        kf->mSnapEpoch = snap_epoch;
                        kf->mSnapIndex = (int)kfs.size();
                        kfs.push_back(v);
                    }
                    const Feature* f = kf->mvFeatures[feat];
                    dsdtm_obs ob{};
                    ob.kf = kf->mSnapIndex; ob.level = f->mlevel; ob.px[0] = f->mpx.x; ob.px[1] = f->mpx.y;
                    const Vector3d Pf = (f->Mpt && f->Mpt != c.mMpPoint) ? f->Mpt->Get_Pose() : P;   // ref: :167 rf->Mpt->Get_Pose()
                    for (int k = 0; k < 3; ++k) { ob.normal[k] = f->mNormal[k]; ob.point_w[k] = Pf[k]; }
                    obs.push_back(ob);
                });
                mp.obs_count = (int)obs.size() - mp.obs_begin;
                it.index = (int)pts.size();
                pts.push_back(mp);
            }
            items.push_back(it);
        }
    }
    cell_begin[mCells.size()] = (int)items.size();
    const int n = (int)pts.size();
    static thread_local std::vector<dsdtm_reproj> res;
    res.resize(n);
    const auto T1 = std::chrono::steady_clock::now();
    if (n > 0) {
        const int cur_slot = rt.Resident(frame->mGpu);
        // Resolving many keyframes can recycle a slot that an earlier table entry already points to when the pool is smaller
        // than the set of keyframes observing the local map (+ the current frame). That would silently sample the wrong image:
        // fail loudly instead. (180 GB of HBM hold ~400 k VGA pyramids: size Gpu.MaxFrames for the whole map.)
        if (cur_slot != cur_slot_first || !rt.SlotsStillValid())
            throw std::runtime_error("Feature_Alignment::SearchLocalPoints: frame pool too small for the local map (raise Gpu.MaxFrames)");
        const SE3 Tc = frame->Get_Pose();
        const Vector3d Oc = frame->Get_CameraCnt();
        double pose[7], center[3];
        for (int k = 0; k < 7; ++k) pose[k] = Tc.data()[k];
        for (int k = 0; k < 3; ++k) center[k] = Oc[k];
        if (dsdtm_local_map_align_batch(rt.ctx(), cur_slot, pose, center, kfs.data(), (int)kfs.size(), obs.data(), (int)obs.size(),
                                        pts.data(), n, mPyr_levels - 3, 10, res.data()) != 0)
            throw std::runtime_error(std::string("dsdtm_local_map_align_batch: ") + dsdtm_last_error(rt.ctx()));
    }
    const auto T2 = std::chrono::steady_clock::now();
    // replay (ref: :75-82, :91-118)
    int matches = 0;
    for (size_t ci = 0; ci < mCells.size(); ++ci) {
        for (int ii = cell_begin[ci]; ii < cell_begin[ci + 1]; ++ii) {
            Item& it = items[ii];
            Candidate& c = *it.cand;
            if (c.mMpPoint->IsBad()) continue;
            if (frame->mImgMask.at(cvRound((float)c.mPx[1]), cvRound((float)c.mPx[0])) != 255) continue;
            if (it.index < 0) continue;
            const dsdtm_reproj& r = res[it.index];
            const int gates = DSDTM_LM_OBS_OK | DSDTM_LM_REF_OK;   // FindMatchDirect's early-outs (:135-140), evaluated on the device
            if ((r.flags & gates) != gates || r.level < 0) continue;
            const int L = r.level;
            c.mPx = Vector2d(r.px[0], r.px[1]);                    // ref: :154 (tPt is updated even on failure; already level-0 scaled)
            if (!(r.flags & DSDTM_LM_CONVERGED)) continue;
            c.mMpPoint->IncreaseFound();
            Feature* f = new Feature(frame.get(), Point2f((float)c.mPx[0], (float)c.mPx[1]), L);
            f->SetPose(c.mMpPoint);
            circle(frame->mImgMask, Point2f((float)c.mPx[0], (float)c.mPx[1]), mCell_size, 0);
            frame->Add_Feature(f);
            frame->Add_MapPoint(c.mMpPoint);
            matches++;
            break;                                               // ReprojectCell returns at the first match
        }
        if (matches >= 200) break;                               // ref: :80 literal
    }
    if (getenv("DSDTM_HOST_TIMING")) {
        const auto T3 = std::chrono::steady_clock::now();
        auto us = [](std::chrono::steady_clock::time_point a, std::chrono::steady_clock::time_point b) { return std::chrono::duration<double, std::micro>(b - a).count(); };
        fprintf(stderr, "SearchLocalPoints: snapshot %.1f us, gpu %.1f us, replay %.1f us (n=%d)\n", us(T0, T1), us(T1, T2), us(T2, T3), n);
    }
    mLastMatches = matches;
}

bool Feature_Alignment::FindMatchDirect(const MapPoint* mp, const FramePtr frame, Vector2d& pt, int& level)   // ref: :128-158
{
    Prepared p;
    if (!Prepare(mp, frame, pt, p)) return false;
    GpuRuntime& rt = GpuRuntime::Instance();
    uint8_t conv = 0;
    double px[2];
    int L = 0;
    if (dsdtm_feature_align_batch(rt.ctx(), rt.Resident(frame->mGpu), &p.c, 1, mPyr_levels - 3, 10, px, &L, &conv, nullptr) != 0)
        throw std::runtime_error(std::string("FindMatchDirect: ") + dsdtm_last_error(rt.ctx()));
    pt = Vector2d(px[0], px[1]);
    level = L;
    return conv != 0;
}

bool Feature_Alignment::CellComparator(Candidate& c1, Candidate& c2) { return c1.mMpPoint->Get_FoundNums() > c2.mMpPoint->Get_FoundNums(); }

void Feature_Alignment::WarpAffine(const Matrix2d A, KeyFrame* kf, Feature* rf, const int search_level, uchar* patch10)   // ref: :206-259
{
    GpuRuntime& rt = GpuRuntime::Instance();
    const int slot = rt.Resident(kf->mGpu), rl = rf->mlevel, sl = search_level;
    const double a[4] = { A(0, 0), A(0, 1), A(1, 0), A(1, 1) };
    const float px[2] = { rf->mpx.x, rf->mpx.y };
    if (dsdtm_warp_affine_batch(rt.ctx(), &slot, a, px, &rl, &sl, 1, patch10) != 0)
        throw std::runtime_error(std::string("dsdtm_warp_affine_batch: ") + dsdtm_last_error(rt.ctx()));
}

void Feature_Alignment::GetPatchNoBoarder()                      // ref: :261-275 (inner 8 x 8 of the 10 x 10 patch)
{
    for (int y = 1; y < 9; ++y)
        for (int x = 1; x < 9; ++x) mPatch[(y - 1) * 8 + (x - 1)] = mPatch_WithBoarder[y * 10 + x];
}

bool Feature_Alignment::Align2DGaussNewton(const FramePtr cur, int level, uchar* patch10, uchar*, int MaxIters, Vector2d& px)   // ref: :318-417
{
    GpuRuntime& rt = GpuRuntime::Instance();
    uint8_t conv = 0;
    double p[2] = { px[0], px[1] };
    if (dsdtm_align2d_batch(rt.ctx(), rt.Resident(cur->mGpu), &level, patch10, p, 1, MaxIters, &conv) != 0)
        throw std::runtime_error(std::string("dsdtm_align2d_batch: ") + dsdtm_last_error(rt.ctx()));
    px = Vector2d(p[0], p[1]);
    return conv != 0;
}

bool Feature_Alignment::Align2DGaussNewton(const Mat8& img, uchar* patch10, uchar*, int MaxIters, Vector2d& px)   // ref: include/Feature_alignment.h:85
{
    GpuRuntime& rt = GpuRuntime::Instance();
    int level = -1;
    for (int l = 0; l < rt.levels() && level < 0; ++l) {
        int w = 0, h = 0; size_t off = 0;
        if (dsdtm_level_info(rt.ctx(), l, &w, &h, &off) == 0 && w == img.cols && h == img.rows) level = l;
    }
    if (level < 0 || img.empty())
        throw std::invalid_argument("Feature_Alignment::Align2DGaussNewton(image, ...): the image must have the size of a pyramid level of the configured camera");
    const std::shared_ptr<GpuSlot> slot = rt.UploadLevel(img, level);
    uint8_t conv = 0;
    double p[2] = { px[0], px[1] };
    if (dsdtm_align2d_batch(rt.ctx(), slot->slot, &level, patch10, p, 1, MaxIters, &conv) != 0)
        throw std::runtime_error(std::string("dsdtm_align2d_batch: ") + dsdtm_last_error(rt.ctx()));
    px = Vector2d(p[0], p[1]);
    return conv != 0;
}

}  // namespace DSDTM
