// optflow_b200 -- job driver: the reference's `optflow <job.json[.gz]>` CLI on top of the C ABI.
//
// Mirrors main / from_file / get_rois / solve_rois / solve_wrapper / move_pm / upload_points of
// the reference (src/optflow.cpp:29-178, 228-261, 302-392, 395-497, 574-641), both the plain and the
// feature pre-alignment path (N4: find_alignment of src/features.cpp:46-167 through tvl1_find_alignment):
//   * same job JSON (comments tolerated, .gz transparently inflated), same key precedence
//     im_args.get(key, args.get(key, default));
//   * same pair loop incl. re-use of the previous pair's decoded frame (:97-103);
//   * same ROI keys ("top", "bottom", "custom", "custom" with "0"/"1") walked in jsoncpp's
//     alphabetical member order; same output naming
//     <output_dir>/<output_name>_<scale %0.2f>[_top|_bottom]_{x,y}.tiff (:155-157, :345, :480-481);
//   * output_type "map" | "flow" -> float TIFF planes, "random_points" -> match records.
//   * "features" / no roi / frames of different size: frame1 is aligned to frame0 by keypoints and an
//     affine warp before the solve, the map is warped by the same affine afterwards (:366-377, :411-444),
//     and random_points takes its `features` branch (:544-550).  The descriptor is this library's own
//     ORB-style one for either feature type (SURF is non-free): see tvl1_b200.h.
// Differences, all because the dependency is out of scope or absent here:
//   * match batches are written to <output_dir>/point_matches_<n>.json with exactly the payload
//     upload_points would PUT to the Render service (:620-634) -- there is no network here;
// N2, the I/O path: frames are decoded on host threads into PINNED buffers `prefetch` pairs ahead; a
// decoded frame goes up once on a copy stream, is prescaled by `scale` there (tvl1_prescale_u8: the
// 8-bit cv::resize of :111,124, bit for bit, any factor) and stays on the device in one of three frame
// slots, so the slice two adjacent pairs share is neither decoded nor uploaded twice (:97-103) and the
// next pair's new frame arrives while the current pair is solved.  The coordinate grid of "map" and the
// frame1 <= 1 mask are applied on the device (tvl1_finish_flow_u8); flow planes come down into pinned
// buffers and are written to TIFF on a host thread while the next pair is solved.
// All arithmetic runs in libtvl1_b200.so; this file only moves bytes and JSON.
#include <zlib.h>

#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <ctime>
#include <future>
#include <iostream>
#include <map>
#include <mutex>
#include <stdexcept>
#include <string>
#include <vector>

#include "../../include/tvl1_b200.h"
#include "imageio.h"
#include "minijson.h"

using mj::Value;

namespace {

struct Rect { int x, y, w, h; };

struct DeviceBuf {
    void* ptr = nullptr;
    size_t bytes = 0;
};

// pinned host buffers, recycled: taken by the decode threads and the flow downloads, returned when the
// copy / the TIFF writer is done with them
struct PinnedPool {
    int device = 0;
    std::mutex m;
    std::vector<std::pair<void*, size_t>> free_;
    void* get(size_t bytes, size_t* cap)
    {
        {
            std::lock_guard<std::mutex> l(m);
            for (size_t k = 0; k < free_.size(); k++)
                if (free_[k].second >= bytes) {
                    void* p = free_[k].first;
                    *cap = free_[k].second;
                    free_.erase(free_.begin() + (long)k);
                    return p;
                }
        }
        void* p = nullptr;
        tvl1_set_device(device);   // the calling thread may be a decode thread: same device, same context
        if (tvl1_host_alloc_pinned(bytes, &p) < 0) return nullptr;
        *cap = bytes;
        return p;
    }
    void put(void* p, size_t cap)
    {
        std::lock_guard<std::mutex> l(m);
        free_.emplace_back(p, cap);
    }
    ~PinnedPool()
    {
        for (auto& f : free_) tvl1_host_free_pinned(f.first);
    }
};

// a prescaled frame resident on the device
struct FrameSlot {
    std::string name;
    float scale = -1.f;
    DeviceBuf buf;
    int w = 0, h = 0;
    long long last_use = -1;   // pair index
};

struct Driver {
    int device = 0;
    int prefetch = 8;       // pairs whose frames are decoded ahead on host threads
    tvl1_handle* solver = nullptr;
    tvl1_params cur{};
    bool have_params = false;
    void *s_solve = nullptr, *s_copy = nullptr;   // streams
    FrameSlot slot[3];
    DeviceBuf raw, du, dv;
    DeviceBuf mx, my;          // warped map planes of the features path
    DeviceBuf aligned[2];      // frame1 after the affine pre-alignment (ping-pong: a second roi key re-aligns it)
    PinnedPool pool;
    std::vector<std::pair<void*, size_t>> in_copy;   // pinned buffers the copy stream may still read
    std::vector<std::future<bool>> writers;          // TIFF writers in flight
    long long rand_skip = 0;   // debug mode: one rand() stream for the whole process
    int uploads = 0;
    int shard = 0, nshards = 1, skipped = 0;
    // --timing: where the wall time of a job goes (seconds): waiting for a frame's decode, staging, solving + outputs
    bool timing = false;
    double t_decode_wait = 0, t_stage = 0, t_solve = 0, t_lookahead = 0, t_points = 0, t_tail = 0, t_setup = 0;
    mj::Value all_matches = mj::Value::array();   // every batch so far, for the "matches_file" key

    ~Driver()
    {
        for (auto& w : writers) w.get();
        if (s_copy) { tvl1_stream_sync(s_copy); tvl1_stream_destroy(s_copy); }
        if (s_solve) { tvl1_stream_sync(s_solve); tvl1_stream_destroy(s_solve); }
        for (auto& b : in_copy) pool.put(b.first, b.second);
        if (solver) tvl1_destroy(solver);
        for (DeviceBuf* f : {&slot[0].buf, &slot[1].buf, &slot[2].buf, &raw, &du, &dv, &mx, &my, &aligned[0], &aligned[1]})
            if (f->ptr) tvl1_dev_free(device, f->ptr);
    }
};

[[noreturn]] void die(const std::string& m)
{
    std::cerr << "optflow_b200: " << m << "\n";
    std::exit(2);
}

// A problem with ONE pair (roi outside the frame, frames of different size, a solver status): the pair
// is logged and skipped and the job goes on, as the reference does for an unreadable image
// (src/optflow.cpp:108-112, 120-124); matches already batched are still flushed at the end.
struct PairError : std::runtime_error { using std::runtime_error::runtime_error; };
[[noreturn]] void pair_fail(const std::string& m) { throw PairError(m); }

void ck(int rc, const char* what)
{
    if (rc < 0) pair_fail(std::string(what) + ": " + tvl1_last_error());
}

const Value& pick(const Value& im, const Value& args, const char* key, const Value& dflt)
{
    // im_args.get(key, args.get(key, default))
    return im.get(key, args.get(key, dflt));
}

std::string slurp(const std::string& path)
{
    gzFile g = gzopen(path.c_str(), "rb");   // reads plain files too
    if (!g) die("cannot open " + path);
    std::string s;
    char buf[1 << 16];
    int n;
    while ((n = gzread(g, buf, sizeof(buf))) > 0) s.append(buf, (size_t)n);
    gzclose(g);
    return s;
}

void reserve(Driver& D, DeviceBuf& f, size_t bytes)
{
    if (f.bytes >= bytes) return;
    if (f.ptr) tvl1_dev_free(D.device, f.ptr);
    f.ptr = nullptr;
    ck(tvl1_dev_alloc(D.device, bytes, &f.ptr), "device allocation");
    f.bytes = bytes;
}

// generate_TV_args (src/optflow.cpp:500-514) + the optional CPU-class keys
tvl1_params tv_params(const Value& im, const Value& args)
{
    tvl1_params p;
    tvl1_default_params(&p);
    p.tau = pick(im, args, "tau", Value(0.25)).asDouble();
    p.lambda = pick(im, args, "lambda", Value(0.05)).asDouble();
    p.theta = pick(im, args, "theta", Value(0.3)).asDouble();
    p.nscales = (int)pick(im, args, "nscales", Value(10)).asInt();
    p.warps = (int)pick(im, args, "warps", Value(5)).asInt();
    p.epsilon = pick(im, args, "epsilon", Value(0.01)).asDouble();
    p.iterations = (int)pick(im, args, "iterations", Value(300)).asInt();
    p.scale_step = pick(im, args, "scaleStep", Value(0.8)).asDouble();
    p.gamma = pick(im, args, "gamma", Value(0.0)).asDouble();
    p.use_initial_flow = 0;   // read but never forwarded by the reference (:512, :518)
    p.inner_iterations = (int)pick(im, args, "innerIterations", Value(0)).asInt();
    p.outer_iterations = (int)pick(im, args, "outerIterations", Value(0)).asInt();
    p.median_filtering = (int)pick(im, args, "medianFiltering", Value(5)).asInt();
    // "cpu" (default): cv::DualTVL1OpticalFlow; "cuda": cv::cuda::OpticalFlowDual_TVL1's algorithm, whose flat
    // loop has no inner / outer iterations and no median -- those keys are refused rather than ignored
    const std::string sem = pick(im, args, "semantics", Value("cpu")).asString();
    if (sem == "cuda") {
        p.semantics = TVL1_SEMANTICS_CUDA;
        for (const char* k : {"innerIterations", "outerIterations", "medianFiltering"})
            if (im.isMember(k) || args.isMember(k))
                pair_fail(std::string("\"") + k + "\" has no meaning with \"semantics\": \"cuda\"");
        p.median_filtering = 1;
    } else if (sem != "cpu") {
        pair_fail("\"semantics\" must be \"cpu\" or \"cuda\", not \"" + sem + "\"");
    }
    return p;
}

void ensure_solver(Driver& D, const tvl1_params& p)
{
    if (!D.solver) {
        ck(tvl1_create(&p, D.device, &D.solver), "tvl1_create");
    } else if (!D.have_params || std::memcmp(&p, &D.cur, sizeof(p)) != 0) {
        ck(tvl1_set_params(D.solver, &p), "tvl1_set_params");
    }
    D.cur = p;
    D.have_params = true;
}

Rect roi_from_array(const Value& a)
{
    if (!a.isArray() || a.size() < 4) pair_fail("an roi must be [x, y, width, height]");
    return Rect{(int)a[0].asInt(), (int)a[1].asInt(), (int)a[2].asInt(), (int)a[3].asInt()};
}

// get_rois (src/optflow.cpp:228-261)
void get_rois(Value& rois, const Value& spec, int rows, int cols)
{
    auto rect = [](int x, int y, int w, int h) {
        Value v = Value::array();
        v.append(Value(x)); v.append(Value(y)); v.append(Value(w)); v.append(Value(h));
        return v;
    };
    if (spec.isMember("top")) rois["top"] = rect(0, 0, cols, (int)spec.get("top", Value(300)).asInt());
    if (spec.isMember("bottom")) {
        const int b = (int)spec.get("bottom", Value(300)).asInt();
        rois["bottom"] = rect(0, rows - b, cols, b);
    }
    if (spec.isMember("custom")) {
        const Value& c = spec.at("custom");
        if (c.isMember("0")) {
            if (!c.isMember("1")) pair_fail("rois.custom with \"0\" needs \"1\" as well");
            rois["custom_diff"]["0"] = c.at("0");
            rois["custom_diff"]["1"] = c.at("1");
        } else {
            rois["custom"] = c;
        }
    }
}

void check_roi(const Rect& r, int w, int h, const char* which)
{
    if (r.w <= 0 || r.h <= 0 || r.x < 0 || r.y < 0 || r.x + r.w > w || r.y + r.h > h)
        pair_fail(std::string("roi outside the frame (") + which + ")");
}

// solve_wrapper (src/optflow.cpp:395-497).  f0 / f1: the pair's frames on the device (f1 already moved by
// `affine` when `features`).
void solve_wrapper(Driver& D, const FrameSlot& f0, const FrameSlot& f1, const Rect& r0, const Rect& r1,
                   Value& im, const Value& args, const float* affine, bool features)
{
    if (r0.w != r1.w || r0.h != r1.h) pair_fail("the two rois of a pair must have the same size");
    const int w = r0.w, h = r0.h;
    ensure_solver(D, tv_params(im, args));
    reserve(D, D.du, (size_t)w * h * 4);
    reserve(D, D.dv, (size_t)w * h * 4);
    const uint8_t* p0 = (const uint8_t*)f0.buf.ptr + (size_t)r0.y * f0.w + r0.x;   // ROI views: pointer + pitch
    const uint8_t* p1 = (const uint8_t*)f1.buf.ptr + (size_t)r1.y * f1.w + r1.x;
    float *du = (float*)D.du.ptr, *dv = (float*)D.dv.ptr;
    ck(tvl1_calc_u8(D.solver, p0, (size_t)f0.w, p1, (size_t)f1.w, w, h, du, dv, (size_t)w * 4, D.s_solve, nullptr), "tvl1_calc_u8");

    const std::string output_type = pick(im, args, "output_type", Value("map")).asString();
    if (features) {
        // :411-444: map = flow + grid, moved by the SAME affine (cv::cuda::warpAffine, linear, constant 0),
        // back to a displacement for "flow"; then the frame1 <= 1 mask (:471-473).  All on the device.
        reserve(D, D.mx, (size_t)w * h * 4);
        reserve(D, D.my, (size_t)w * h * 4);
        float *mx = (float*)D.mx.ptr, *my = (float*)D.my.ptr;
        ck(tvl1_finish_flow_u8(D.solver, nullptr, 0, w, h, du, dv, (size_t)w * 4, 1, D.s_solve), "map grid");
        ck(tvl1_warp_affine_f32(du, (size_t)w * 4, w, h, affine, mx, (size_t)w * 4, w, h, D.s_solve), "tvl1_warp_affine_f32");
        ck(tvl1_warp_affine_f32(dv, (size_t)w * 4, w, h, affine, my, (size_t)w * 4, w, h, D.s_solve), "tvl1_warp_affine_f32");
        ck(tvl1_finish_flow_u8(D.solver, p1, (size_t)f1.w, w, h, mx, my, (size_t)w * 4, output_type == "flow" ? -1 : 0, D.s_solve),
           "tvl1_finish_flow_u8");
        du = mx; dv = my;
    } else {
        // the coordinate grid of "map" (:445-466) and the frame1 <= 1 mask (:471-473), on the device
        ck(tvl1_finish_flow_u8(D.solver, p1, (size_t)f1.w, w, h, du, dv, (size_t)w * 4, output_type == "map", D.s_solve),
           "tvl1_finish_flow_u8");
    }
    if (output_type == "random_points") {
        const bool debug = args.get("debug", Value(false)).asBool();
        const float scale = pick(im, args, "scale", Value(0.5)).asFloat();
        const int npoints = (int)pick(im, args, "npoints", Value(25)).asInt();
        const int cap = npoints > 0 ? npoints : 1;
        std::vector<double> px(cap), py(cap), qx(cap), qy(cap), wt(cap);
        int n = 0;
        long long used = 0;
        // srand(time(0)) unless debug (:532-535); debug keeps drawing from one unseeded stream
        const long long seed = debug ? -1 : (long long)std::time(nullptr);
        ck(tvl1_sample_matches_ex(D.solver, p0, (size_t)f0.w, p1, (size_t)f1.w, du, dv, (size_t)w * 4, w, h, r0.x, r0.y,
                                  r1.x, r1.y, scale, npoints, seed, debug ? D.rand_skip : 0, features ? 1 : 0, px.data(),
                                  py.data(), qx.data(), qy.data(), wt.data(), nullptr, &n, &used, D.s_solve), "tvl1_sample_matches");
        if (debug) D.rand_skip += used;
        Value& pm = im["point_matches"];
        if (!pm.isMember("p")) {
            pm["p"] = Value::array(); pm["p"].append(Value::array()); pm["p"].append(Value::array());
            pm["q"] = Value::array(); pm["q"].append(Value::array()); pm["q"].append(Value::array());
            pm["w"] = Value::array();
        }
        for (int k = 0; k < n; k++) {
            pm["w"].append(Value((long long)(wt[k] != 0.0 ? 1 : 0)));
            pm["p"][0].append(Value(px[k])); pm["p"][1].append(Value(py[k]));
            pm["q"][0].append(Value(qx[k])); pm["q"][1].append(Value(qy[k]));
        }
        return;
    }
    // "map" | "flow": planes into pinned host buffers, float TIFFs written by a host thread while the
    // next pair is solved (at most two writers in flight)
    const size_t nb = (size_t)w * h * 4;
    size_t capx = 0, capy = 0;
    float* hx = (float*)D.pool.get(nb, &capx);
    float* hy = (float*)D.pool.get(nb, &capy);
    if (!hx || !hy) die("pinned host allocation failed");
    ck(tvl1_dev_d2h_async(hx, du, nb, D.s_solve), "download");
    ck(tvl1_dev_d2h_async(hy, dv, nb, D.s_solve), "download");
    ck(tvl1_stream_sync(D.s_solve), "download");
    while (D.writers.size() >= 2) {
        if (!D.writers.front().get()) die("cannot write a flow TIFF");
        D.writers.erase(D.writers.begin());
    }
    const std::string base = im.at("output").asString() + im.at("output_suffix").asString();
    PinnedPool* pool = &D.pool;
    D.writers.push_back(std::async(std::launch::async, [=]() {
        const bool ok = imio::write_tiff_f32(base + "_x.tiff", hx, w, h) && imio::write_tiff_f32(base + "_y.tiff", hy, w, h);
        if (!ok) std::cerr << "optflow_b200: cannot write " << base << "_{x,y}.tiff\n";
        pool->put(hx, capx);
        pool->put(hy, capy);
        return ok;
    }));
}

// move_pm (src/optflow.cpp:574-593)
void move_pm(Value& im, Value& args)
{
    Value single = Value::object();
    single["pGroupId"] = im.at("pGroupId");
    single["pId"] = im.at("pId");
    single["qGroupId"] = im.at("qGroupId");
    single["qId"] = im.at("qId");
    single["matches"] = im.at("point_matches");
    args["point_matches"].append(single);
    im["point_matches"] = Value::object();
}

// upload_points (src/optflow.cpp:595-641): same payload, written to a file instead of PUT
void upload_points(Driver& D, Value& args)
{
    // One file per batch, named by shard and batch so that the ranks of a sharded job (one process per
    // GPU) never write the same name: point_matches_NNN.json, or point_matches_rRofW_NNN.json under
    // --shard R/W.  The optional "matches_file" key collects EVERY batch of this process in one JSON
    // array (rewritten after each batch; "<file>.rRofW" under --shard).
    const std::string dir = args.get("output_dir", Value(".")).asString();
    char name[96];
    if (D.nshards > 1) std::snprintf(name, sizeof(name), "/point_matches_r%dof%d_%03d.json", D.shard, D.nshards, D.uploads++);
    else std::snprintf(name, sizeof(name), "/point_matches_%03d.json", D.uploads++);
    const std::string payload = mj::dump(args.at("point_matches"));
    auto write_all = [](const std::string& path, const std::string& text) {
        FILE* f = std::fopen(path.c_str(), "wb");
        if (!f) die("cannot write " + path);
        std::fwrite(text.data(), 1, text.size(), f);
        std::fclose(f);
    };
    std::string path = dir + name;
    if (args.isMember("matches_file")) {
        path = args.at("matches_file").asString();
        if (D.nshards > 1) {
            char suf[48];
            std::snprintf(suf, sizeof(suf), ".r%dof%d", D.shard, D.nshards);
            path += suf;
        }
        const Value& batch = args.at("point_matches");
        for (size_t k = 0; k < batch.size(); k++) D.all_matches.append(batch[k]);
        write_all(path, mj::dump(D.all_matches));
    } else {
        write_all(path, payload);
    }
    if (args.get("debug", Value(false)).asBool()) {
        std::cout << payload << "\n";
        std::cout << "http://" << args.get("host", Value("10.40.3.162")).asString() << ":" << args.get("port", Value("8080")).asString()
                  << "/render-ws/v1/owner/" << args.get("owner", Value("flyem")).asString() << "/matchCollection/"
                  << args.get("matchCollection", Value("forgetful_owner")).asString() << "/matches -> " << path << "\n";
    }
}

// cv::imread(..., IMREAD_GRAYSCALE) on a host thread, into a pinned buffer (:106, :119)
struct Decoded { bool ok = false; std::string err; int w = 0, h = 0; uint8_t* px = nullptr; size_t cap = 0; };
Decoded decode_frame(const std::string& path, PinnedPool* pool)
{
    Decoded d;
    imio::Gray8 img;
    if (!imio::read_gray8(path, img, d.err)) return d;
    d.px = (uint8_t*)pool->get(img.px.size(), &d.cap);
    if (!d.px) { d.err = "pinned host allocation failed"; return d; }
    std::memcpy(d.px, img.px.data(), img.px.size());
    d.w = img.w; d.h = img.h; d.ok = true;
    return d;
}

// pinned buffers whose upload has completed go back to the pool
void recycle_uploads(Driver& D, bool wait)
{
    if (D.in_copy.empty()) return;
    if (wait) ck(tvl1_stream_sync(D.s_copy), "copy stream");
    else if (tvl1_stream_query(D.s_copy) != 1) return;
    for (auto& b : D.in_copy) D.pool.put(b.first, b.second);
    D.in_copy.clear();
}

// A decoded frame -> device slot, on the copy stream: upload, then cv::resize(frame, frame, Size(), scale,
// scale) of the reference's loader (:111, :124) on the device.  Nothing here waits for the GPU.
void stage_frame(Driver& D, FrameSlot& sl, const std::string& name, float scale, Decoded& d)
{
    int dw = d.w, dh = d.h;
    if (scale != 1.f) ck(tvl1_prescaled_size(d.w, d.h, (double)scale, &dw, &dh), "prescale");
    sl.name.clear();   // invalid until everything below has been enqueued
    reserve(D, sl.buf, (size_t)dw * dh);
    const size_t raw_bytes = (size_t)d.w * d.h;
    if (scale == 1.f) {
        ck(tvl1_dev_h2d_async(sl.buf.ptr, d.px, raw_bytes, D.s_copy), "upload");
    } else {
        if (D.raw.bytes < raw_bytes) {   // the copy stream may still be reading the old staging buffer
            ck(tvl1_stream_sync(D.s_copy), "copy stream");
            reserve(D, D.raw, raw_bytes);
        }
        ck(tvl1_dev_h2d_async(D.raw.ptr, d.px, raw_bytes, D.s_copy), "upload");
        ck(tvl1_prescale_u8((const uint8_t*)D.raw.ptr, (size_t)d.w, d.w, d.h, (double)scale, (uint8_t*)sl.buf.ptr, (size_t)dw,
                            D.s_copy), "prescale");
    }
    D.in_copy.emplace_back(d.px, d.cap);
    d.px = nullptr;
    sl.name = name; sl.scale = scale; sl.w = dw; sl.h = dh;
}

// orb_defaults (src/features.cpp:19-32) + ratio / ransac / homo (:107, :133), per-pair > global > default
tvl1_feature_params feature_params(const Value& im, const Value& args)
{
    tvl1_feature_params p;
    tvl1_default_feature_params(&p);
    p.nfeatures = (int)pick(im, args, "nfeatures", Value(5000)).asInt();
    p.scale_factor = pick(im, args, "scaleFactor", Value(1.2)).asFloat();
    p.nlevels = (int)pick(im, args, "nlevels", Value(8)).asInt();
    p.edge_threshold = (int)pick(im, args, "edgeThreshold", Value(31)).asInt();
    p.first_level = (int)pick(im, args, "firstLevel", Value(0)).asInt();
    p.patch_size = (int)pick(im, args, "patchSize", Value(31)).asInt();
    p.fast_threshold = (int)pick(im, args, "fastThreshold", Value(20)).asInt();
    p.ratio = pick(im, args, "ratio", Value(0.8)).asFloat();
    p.ransac = pick(im, args, "ransac", Value(5.0)).asDouble();
    p.homo = (int)pick(im, args, "homo", Value(8)).asInt();
    p.debug = args.get("debug", Value(false)).asBool() ? 1 : 0;
    return p;
}

// solve_rois (src/optflow.cpp:312-392)
void solve_rois(Driver& D, const FrameSlot& f0, const FrameSlot& f1_in, const Value& rois, Value& im, Value& args)
{
    // src/optflow.cpp:323-338: an explicit false at either level wins, then a true at either level
    bool features;
    if (im.isMember("features") && !im.at("features").asBool()) features = false;
    else if (args.isMember("features") && !args.at("features").asBool()) features = false;
    else features = im.get("features", Value(false)).asBool() || args.get("features", Value(false)).asBool();
    ck(tvl1_stream_wait(D.s_solve, D.s_copy), "stream wait");   // both frames have arrived and are prescaled
    FrameSlot f1 = f1_in;   // a view: replaced by the aligned frame below, the slot itself stays as decoded
    float affine[6] = {1.f, 0.f, 0.f, 0.f, 1.f, 0.f};
    int flip = 0;
    for (const auto& kv : *rois.o) {   // alphabetical, like Json::Value::getMemberNames()
        const std::string& key = kv.first;
        im["output_suffix"] = (key == "top" || key == "bottom") ? Value("_" + key) : Value("");
        if (key == "custom_diff") {
            if (features) std::cerr << "Features isn't compatible with different ROIs for each image.\n Ignoring features.\n";
            const Rect r0 = roi_from_array(kv.second.at("0")), r1 = roi_from_array(kv.second.at("1"));
            check_roi(r0, f0.w, f0.h, "custom 0");
            check_roi(r1, f1.w, f1.h, "custom 1");
            // the reference hands `features` through as is (:363): the map is still moved by whatever
            // `affine` holds (identity unless an earlier roi key of this pair aligned)
            solve_wrapper(D, f0, f1, r0, r1, im, args, affine, features);
        } else {
            const bool differ = f0.w != f1.w || f0.h != f1.h;
            if (features || differ || key == "default") {
                if (differ || (key == "default" && !features))
                    std::cerr << "Rows or columns differ between frames no ROI selected, reverting to features even though it wasn't selected.\n";
                // :373-376: frame1 is replaced by its aligned version for this and every later roi key of
                // the pair (a later key aligns the already aligned frame again, as the reference does)
                const tvl1_feature_params fp = feature_params(im, args);
                int nm = 0, ng = 0;
                ensure_solver(D, tv_params(im, args));
                ck(tvl1_find_alignment(D.solver, (const uint8_t*)f1.buf.ptr, (size_t)f1.w, f1.w, f1.h, (const uint8_t*)f0.buf.ptr, (size_t)f0.w,
                                       f0.w, f0.h, &fp, affine, &nm, &ng, D.s_solve), "tvl1_find_alignment");
                DeviceBuf& dst = D.aligned[flip];
                flip ^= 1;
                reserve(D, dst, (size_t)f0.w * f0.h);
                ck(tvl1_warp_affine_u8((const uint8_t*)f1.buf.ptr, (size_t)f1.w, f1.w, f1.h, affine, (uint8_t*)dst.ptr, (size_t)f0.w,
                                       f0.w, f0.h, D.s_solve), "tvl1_warp_affine_u8");
                f1.buf = dst; f1.w = f0.w; f1.h = f0.h;
                features = true;
            }
            const Rect r = roi_from_array(kv.second);
            check_roi(r, f0.w, f0.h, key.c_str());
            solve_wrapper(D, f0, f1, r, r, im, args, affine, features);
        }
    }
    if (pick(im, args, "output_type", Value("map")).asString() == "random_points") move_pm(im, args);
}

// from_file (src/optflow.cpp:75-178)
int from_file(Driver& D, Value& args, int shard, int nshards)
{
    const auto tsu0 = std::chrono::steady_clock::now();
    const Value images = args.at("images");
    if (!images.isArray()) die("\"images\" must be an array");
    // The reference keeps the previous pair's decoded frames so that a slice shared by adjacent pairs (q
    // of pair i-1 == p of pair i) is not read twice (:97-103).  Here the prescaled frames stay on the
    // DEVICE, in three slots: two for the pair being solved, one for the frame the next pair brings.
    bool any_upload_since = false;
    std::map<std::string, std::future<Decoded>> inflight;   // frames being decoded for the pairs ahead
    PinnedPool* pool = &D.pool;
    auto prefetch = [&](const std::string& name) {
        if (!inflight.count(name)) inflight.emplace(name, std::async(std::launch::async, decode_frame, name, pool));
    };
    const size_t n = images.size();
    const size_t base = n / nshards, rem = n % nshards;
    const size_t begin = shard * base + std::min<size_t>(shard, rem), end = begin + base + ((size_t)shard < rem ? 1 : 0);
    long long last_upload = (long long)begin;   // the batch counter starts where this shard starts
    D.shard = shard; D.nshards = nshards;
    D.pool.device = D.device;
    // the first pair's frames start decoding before this process has even touched CUDA: creating the context
    // takes as long as decoding a slice, and the two overlap
    if (D.prefetch > 0 && begin < end) {
        const Value& first = images[begin];
        if (first.isMember("p") && first.isMember("q") && first.at("p").type == Value::String && first.at("q").type == Value::String) {
            prefetch(first.at("p").asString());
            if (first.at("q").asString() != first.at("p").asString()) prefetch(first.at("q").asString());
        }
    }
    if (tvl1_dev_count() <= 0) die("no CUDA device: this driver has no CPU path");
    if (tvl1_stream_create(D.device, &D.s_solve) < 0 || tvl1_stream_create(D.device, &D.s_copy) < 0)
        die(std::string("stream creation: ") + tvl1_last_error());
    auto scale_of = [&](const Value& im) { return im.get("scale", args.get("scale", Value(0.5))).asFloat(); };
    auto find_slot = [&](const std::string& name, float scale) -> FrameSlot* {
        for (FrameSlot& sl : D.slot)
            if (!sl.name.empty() && sl.name == name && sl.scale == scale) return &sl;
        return nullptr;
    };
    // least recently used slot that neither `keep0` nor `keep1` occupies
    auto victim = [&](const FrameSlot* keep0, const FrameSlot* keep1) -> FrameSlot* {
        FrameSlot* v = nullptr;
        for (FrameSlot& sl : D.slot)
            if (&sl != keep0 && &sl != keep1 && (!v || sl.last_use < v->last_use)) v = &sl;
        return v;
    };
    D.t_setup = std::chrono::duration<double>(std::chrono::steady_clock::now() - tsu0).count();
    for (size_t i = begin; i < end; i++) {
        Value im = images[i];
        std::string n0, n1;
        try {
        n0 = im.at("p").asString(); n1 = im.at("q").asString();
        const float scale = scale_of(im);
        im["scale"] = Value((double)scale);
        std::cout << n0 << " " << n1 << "\n";
        // decode what the next pairs will need on host threads while this one is solved (decoding an
        // 8k x 8k PNG takes far longer than its solve, so the look-ahead -- not the GPU -- sets the pace
        // of a job); a frame that is on the device already, or that an earlier look-ahead covers, is not
        // decoded twice
        const auto tl0 = std::chrono::steady_clock::now();
        // this pair's own frames first, both at once, if nobody has them yet (the first pair of a job, or a pair
        // that shares no slice with its predecessor): otherwise they would be decoded one after the other below
        if (D.prefetch > 0) {
            if (!find_slot(n0, scale)) prefetch(n0);
            if (n1 != n0 && !find_slot(n1, scale)) prefetch(n1);
        }
        {
            std::string prev0 = n0, prev1 = n1;
            for (size_t j = i + 1; j < end && j <= i + (size_t)D.prefetch; j++) {
                const Value& nx = images[j];
                if (!nx.isMember("p") || !nx.isMember("q")) break;
                const std::string m0 = nx.at("p").asString(), m1 = nx.at("q").asString();
                const float sj = scale_of(nx);
                // the frame slots will still hold the previous pair's frames when pair j is reached
                if (m0 != prev0 && m0 != prev1 && !find_slot(m0, sj)) prefetch(m0);
                if (m1 != prev0 && m1 != prev1 && m1 != m0 && !find_slot(m1, sj)) prefetch(m1);
                prev0 = m0; prev1 = m1;
            }
        }
        recycle_uploads(D, false);
        D.t_lookahead += std::chrono::duration<double>(std::chrono::steady_clock::now() - tl0).count();
        // this pair's frames: on the device already, or decoded (by the look-ahead, else now) and staged
        auto fetch = [&](const std::string& name, const FrameSlot* keep) -> FrameSlot* {
            if (FrameSlot* sl = find_slot(name, scale)) { sl->last_use = (long long)i; return sl; }
            Decoded d;
            const auto tw0 = std::chrono::steady_clock::now();
            auto it = inflight.find(name);
            if (it != inflight.end()) { d = it->second.get(); inflight.erase(it); }
            else d = decode_frame(name, pool);
            const auto tw1 = std::chrono::steady_clock::now();
            D.t_decode_wait += std::chrono::duration<double>(tw1 - tw0).count();
            if (!d.ok) {
                std::cout << "Error: " << name << " (" << d.err << ")\n";   // :108-112, :120-124: log, next pair
                return nullptr;
            }
            FrameSlot* sl = victim(keep, nullptr);
            stage_frame(D, *sl, name, scale, d);
            D.t_stage += std::chrono::duration<double>(std::chrono::steady_clock::now() - tw1).count();
            sl->last_use = (long long)i;
            return sl;
        };
        FrameSlot* f0 = fetch(n0, find_slot(n1, scale));   // never evict the other frame of this pair
        FrameSlot* f1 = f0 ? (n1 == n0 ? f0 : fetch(n1, f0)) : nullptr;
        if (!f0 || !f1) continue;
        // the next pair's new frame goes up now, into the third slot, if its decode has finished: the copy
        // and the prescale then overlap this pair's solve
        if (i + 1 < end) {
            const Value& nx = images[i + 1];
            if (nx.isMember("p") && nx.isMember("q")) {
                const float sj = scale_of(nx);
                for (const char* key : {"p", "q"}) {
                    const std::string m = nx.at(key).asString();
                    auto it = inflight.find(m);
                    if (find_slot(m, sj) || it == inflight.end()) continue;
                    if (it->second.wait_for(std::chrono::seconds(0)) != std::future_status::ready) continue;
                    FrameSlot* sl = victim(f0, f1);
                    if (sl->last_use == (long long)i + 1) continue;   // the one free slot is taken already
                    Decoded d = it->second.get();
                    inflight.erase(it);
                    if (!d.ok) { std::cout << "Error: " << m << " (" << d.err << ")\n"; continue; }
                    stage_frame(D, *sl, m, sj, d);
                    sl->last_use = (long long)i + 1;
                }
            }
        }

        Value rois = Value::object();
        const int rows = std::min(f0->h, f1->h), cols = std::min(f0->w, f1->w);
        if (im.isMember("rois")) get_rois(rois, im.at("rois"), rows, cols);
        else if (args.isMember("rois")) get_rois(rois, args.at("rois"), rows, cols);
        if (rois.size() == 0) {
            Value r = Value::array();
            r.append(Value(0)); r.append(Value(0)); r.append(Value(cols)); r.append(Value(rows));
            rois["default"] = r;
        }
        char buffer[32];
        std::snprintf(buffer, sizeof(buffer), "%0.2f", scale);
        if (!im.isMember("output"))
            im["output"] = Value(args.at("output_dir").asString() + "/" + im.at("output_name").asString() + "_" + buffer);
        {
            const auto ts0 = std::chrono::steady_clock::now();
            solve_rois(D, *f0, *f1, rois, im, args);
            D.t_solve += std::chrono::duration<double>(std::chrono::steady_clock::now() - ts0).count();
        }
        } catch (const std::exception& e) {   // PairError, or a missing / mistyped key of this pair
            std::cout << "Error: pair " << n0 << " " << n1 << " skipped (" << e.what() << ")\n";
            std::cerr << "optflow_b200: pair " << i << " skipped: " << e.what() << "\n";
            D.skipped++;
            continue;
        }

        const auto tp0 = std::chrono::steady_clock::now();
        if (pick(im, args, "output_type", Value("map")).asString() == "random_points") {
            any_upload_since = true;
            if ((long long)i > last_upload + args.get("batch_size", Value(100)).asInt()) {
                upload_points(D, args);
                args["point_matches"] = Value::array();
                last_upload = (long long)i;
                any_upload_since = false;
            }
        }
        D.t_points += std::chrono::duration<double>(std::chrono::steady_clock::now() - tp0).count();
    }
    const auto tt0 = std::chrono::steady_clock::now();
    if (any_upload_since) upload_points(D, args);
    bool ok = true;
    for (auto& w : D.writers) ok = w.get() && ok;
    D.writers.clear();
    for (auto& f : inflight) {   // look-ahead decodes nobody asked for in the end
        Decoded d = f.second.get();
        if (d.px) D.pool.put(d.px, d.cap);
    }
    recycle_uploads(D, true);
    D.t_tail = std::chrono::duration<double>(std::chrono::steady_clock::now() - tt0).count();
    return ok ? 0 : 2;
}

}  // namespace

int main(int argc, const char* argv[])
{
    std::string filename;
    int device = 0, shard = 0, nshards = 1, prefetch = 8;
    bool timing = false;
    const auto t_start = std::chrono::steady_clock::now();
    for (int k = 1; k < argc; k++) {
        const std::string a = argv[k];
        if (a == "-h" || a == "--help") {
            std::cout << "usage: optflow_b200 [--device N] [--shard RANK/WORLD] [--prefetch N] [--timing] <job.json[.gz]>\n"
                         "  --shard: solve only this rank's contiguous block of \"images\" (one process per GPU)\n"
                         "  --prefetch: pairs whose frames are decoded ahead on host threads (default 8)\n";
            return 0;
        } else if (a == "--timing") {
            timing = true;
        } else if (a == "--device" && k + 1 < argc) {
            device = std::atoi(argv[++k]);
        } else if (a == "--prefetch" && k + 1 < argc) {
            prefetch = std::atoi(argv[++k]);
            if (prefetch < 0 || prefetch > 64) die("--prefetch wants 0..64");
        } else if (a == "--shard" && k + 1 < argc) {
            if (std::sscanf(argv[++k], "%d/%d", &shard, &nshards) != 2 || nshards < 1 || shard < 0 || shard >= nshards)
                die("--shard wants RANK/WORLD");
        } else {
            filename = a;
        }
    }
    if (filename.empty()) die("no job file given (see --help)");
    Value args;
    try {
        args = mj::parse(slurp(filename));
    } catch (const std::exception& e) {
        die(std::string(e.what()) + " in " + filename);   // the reference ignores parse errors (:51,56); we do not
    }
    const int style = (int)args.get("style", Value(1)).asInt();
    if (style != 1) die("only \"style\": 1 exists");
    Driver D;
    D.device = device;
    D.prefetch = prefetch;
    D.timing = timing;
    const auto t_parsed = std::chrono::steady_clock::now();
    const int rc = from_file(D, args, shard, nshards);
    if (timing) {
        const auto t_end = std::chrono::steady_clock::now();
        std::fprintf(stderr, "optflow_b200 timing: parse %.3f s, job %.3f s (waiting for decodes %.3f, staging %.3f, "
                     "solves + outputs %.3f, look-ahead %.3f, match batches %.3f, setup %.3f, tail %.3f)\n",
                     std::chrono::duration<double>(t_parsed - t_start).count(),
                     std::chrono::duration<double>(t_end - t_parsed).count(), D.t_decode_wait, D.t_stage, D.t_solve,
                     D.t_lookahead, D.t_points, D.t_setup, D.t_tail);
    }
    return rc;
}
