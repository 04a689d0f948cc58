"""Host-side mirror of the reference's flow-stage interface, on top of the C ABI.

Same names, argument meaning and defaults as the reference's C++ functions
(reference src/optflow.h:28-34, src/optflow.cpp), with dicts in place of Json::Value and
NumPy arrays in place of cv::Mat / GpuMat:

    generate_TV_args(im_args, args)            src/optflow.cpp:500-514
    TVL1_solve(frame0, frame1, TV_args)        src/optflow.cpp:516-520
    TVL1_solve_batch(frame0s, frame1s, TV_args, init_flows=None)
                                               many equal-size pairs in one call (no counterpart)
    find_alignment(frame0, frame1, ...)        src/features.cpp:46-167
    solve_rois(frame0, frame1, rois, ...)      src/optflow.cpp:312-392
    solve_wrapper(frame0, frame1, ...)         src/optflow.cpp:395-497
    random_points(...)                         src/optflow.cpp:522-572
    move_pm(im_args, args)                     src/optflow.cpp:574-593

The arithmetic runs in libtvl1_b200.so on the GPU; there is no CPU fallback and nothing in
this module imports oracle/.
"""
import numpy as np

from . import _native as N

TV_KEYS = ("tau", "lambda", "theta", "nscales", "warps", "epsilon", "iterations", "scaleStep",
           "gamma", "useInitialFlow")
# generate_TV_args defaults, src/optflow.cpp:503-512
TV_DEFAULTS = {"tau": 0.25, "lambda": 0.05, "theta": 0.3, "nscales": 10, "warps": 5,
               "epsilon": 0.01, "iterations": 300, "scaleStep": 0.8, "gamma": 0.0,
               "useInitialFlow": False}
# optional extra keys (SURVEY.md T3/T4): the CPU-class parameters the cv::cuda API lacks
EXTRA_KEYS = ("innerIterations", "outerIterations", "medianFiltering")
# "semantics": "cpu" (default) computes cv::DualTVL1OpticalFlow, "cuda" cv::cuda::OpticalFlowDual_TVL1's algorithm,
# which has none of EXTRA_KEYS
SEMANTICS = ("cpu", "cuda")


def _get(im_args, args, key, default):
    """im_args.get(key, args.get(key, default)): per-pair overrides global overrides default."""
    return im_args.get(key, args.get(key, default))


def generate_TV_args(im_args, args):
    tv = {}
    for k in TV_KEYS:
        v = _get(im_args, args, k, TV_DEFAULTS[k])
        if k in ("nscales", "warps", "iterations"):
            v = int(v)
        elif k == "useInitialFlow":
            v = bool(v)
        else:
            v = float(v)
        tv[k] = v
    for k in EXTRA_KEYS:
        v = _get(im_args, args, k, None)
        if v is not None:
            tv[k] = int(v)
    sem = _get(im_args, args, "semantics", None)
    if sem is None:   # the default, "cpu": the dict stays exactly generate_TV_args's
        return tv
    if sem not in SEMANTICS:
        raise ValueError("\"semantics\" must be \"cpu\" or \"cuda\", not %r" % (sem,))
    if sem == "cuda":
        bad = [k for k in EXTRA_KEYS if k in tv]
        if bad:
            raise ValueError("%s has no meaning with \"semantics\": \"cuda\"" % ", ".join('"%s"' % k for k in bad))
    tv["semantics"] = sem
    return tv


def params_from_TV_args(tv):
    """tvl1_params from the dict generate_TV_args returns.  useInitialFlow is read by the
    reference but never forwarded to the solver (src/optflow.cpp:512,518): ignored here too."""
    p = N.default_params()
    p.tau = tv["tau"]
    p.lambda_ = tv["lambda"]
    p.theta = tv["theta"]
    p.nscales = tv["nscales"]
    p.warps = tv["warps"]
    p.epsilon = tv["epsilon"]
    p.iterations = tv["iterations"]
    p.scale_step = tv["scaleStep"]
    p.gamma = tv["gamma"]
    p.use_initial_flow = 0
    p.inner_iterations = int(tv.get("innerIterations", 0))
    p.outer_iterations = int(tv.get("outerIterations", 0))
    p.median_filtering = int(tv.get("medianFiltering", 5))
    sem = tv.get("semantics", "cpu")
    p.semantics = N.semantics_code(sem)
    if sem == "cuda":
        bad = [k for k in EXTRA_KEYS if k in tv]
        if bad:
            raise ValueError("%s has no meaning with \"semantics\": \"cuda\"" % ", ".join('"%s"' % k for k in bad))
        p.median_filtering = 1
    return p


_solvers = {}


def _solver_for(tv, device):
    """The reference builds a new solver per call (src/optflow.cpp:518); a handle per
    (device, parameter set) is kept here so that its device arena is re-used across pairs."""
    key = (device,) + tuple(sorted(tv.items()))
    s = _solvers.get(key)
    if s is None:
        s = N.Solver(params_from_TV_args(tv), device)
        _solvers[key] = s
    return s


def release_solvers():
    for s in _solvers.values():
        s.close()
    _solvers.clear()


def TVL1_solve(frame0, frame1, TV_args, device=0, init_flow=None):
    """Flow from frame0 to frame1 (uint8, equal size) -> (flow_x, flow_y) float32 planes.  init_flow: (flow_x,
    flow_y) float32 planes the solve starts from (OpenCV's useInitialFlow + calc(I0, I1, flow)); with it, the frames
    may also both be float32 (scaled by 255, as the OpenCV classes' convertTo does)."""
    s = _solver_for(TV_args, device)
    if init_flow is None:
        return s.calc(frame0, frame1)
    return s.calc_ex(frame0, frame1, init=init_flow)


def TVL1_solve_batch(frame0s, frame1s, TV_args, device=0, init_flows=None):
    """TVL1_solve of many pairs of one size in one call: lists of frames (all uint8, or all float32 -- scaled by 255,
    as TVL1_solve does with an init_flow) in, a list of (flow_x, flow_y) float32 planes out, each exactly what
    TVL1_solve of that pair returns, in either "semantics" and with any gamma.  init_flows: None, or one (flow_x,
    flow_y) pair of float32 planes per pair, as TVL1_solve's init_flow.  Solving equal-size ROI strips a batch at a time keeps the GPU busy where one small pair leaves it
    mostly idle."""
    return _solver_for(TV_args, device).calc_batch_ex(frame0s, frame1s, init=init_flows)


# orb_defaults (src/features.cpp:19-32) and the matcher / RANSAC keys (:107, :133)
FEATURE_DEFAULTS = {"nfeatures": 5000, "scaleFactor": 1.2, "nlevels": 8, "edgeThreshold": 31, "firstLevel": 0,
                    "patchSize": 31, "fastThreshold": 20, "ratio": 0.8, "ransac": 5.0, "homo": 8}


def find_alignment(frame0, frame1, im_args, args, device=0):
    """find_alignment (src/features.cpp:46-167) with the reference's argument order: keypoints of `frame0`
    (the query set) are matched to `frame1` and the 2x3 float32 affine maps frame0 coordinates to frame1
    coordinates; identity when there are not enough good matches or the zoom check fails.  solve_rois
    calls it as find_alignment(frame1_of_the_pair, frame0_of_the_pair) (src/optflow.cpp:373)."""
    s = _solver_for(generate_TV_args(im_args, args), device)
    kw = {k: type(d)(_get(im_args, args, k, d)) for k, d in FEATURE_DEFAULTS.items()}
    kw["debug"] = int(bool(args.get("debug", False)))
    aff, _, _ = s.find_alignment(frame0, frame1, **kw)
    return aff


def _features_flag(im_args, args):
    # src/optflow.cpp:323-338: an explicit false at either level wins, then a true at either level
    if "features" in im_args and not im_args["features"]:
        return False
    if "features" in args and not args["features"]:
        return False
    return bool(im_args.get("features", False)) or bool(args.get("features", False))


def solve_rois(frame0, frame1, rois, im_args, args, device=0, seed=None):
    """solve_rois (src/optflow.cpp:312-392): walks the roi keys in alphabetical order (jsoncpp's member
    order); with `features`, frames of different size or the "default" roi, frame1 is first aligned to
    frame0 (find_alignment + warpAffine, :366-377) and stays aligned for the later keys.  Returns
    {roi_key: (flow_x, flow_y)}; "random_points" jobs get their record moved to args["point_matches"]."""
    frame0 = np.ascontiguousarray(frame0, np.uint8)
    frame1 = np.ascontiguousarray(frame1, np.uint8)
    features = _features_flag(im_args, args)
    affine = np.array([[1, 0, 0], [0, 1, 0]], np.float32)
    out = {}
    for key in sorted(rois):
        im_args["output_suffix"] = "_" + key if key in ("top", "bottom") else ""
        if key == "custom_diff":
            x0, y0, w0, h0 = (int(v) for v in rois[key]["0"])
            x1, y1, w1, h1 = (int(v) for v in rois[key]["1"])
            out[key] = solve_wrapper(frame0[y0:y0 + h0, x0:x0 + w0], frame1[y1:y1 + h1, x1:x1 + w1], im_args, args,
                                     roi_vec=((x0, y0), (x1, y1)), device=device, seed=seed, affine=affine, features=features)
            continue
        if features or frame0.shape != frame1.shape or key == "default":
            affine = find_alignment(frame1, frame0, im_args, args, device)
            frame1 = N.warp_affine(frame1, affine, (frame0.shape[1], frame0.shape[0]), device)
            features = True
        x, y, w, h = (int(v) for v in rois[key])
        out[key] = solve_wrapper(frame0[y:y + h, x:x + w], frame1[y:y + h, x:x + w], im_args, args,
                                 roi_vec=((x, y), (x, y)), device=device, seed=seed, affine=affine, features=features)
    if _get(im_args, args, "output_type", "map") == "random_points":
        move_pm(im_args, args)
    return out


def solve_wrapper(frame0, frame1, im_args, args, roi_vec=((0, 0), (0, 0)), device=0, seed=None, affine=None,
                  features=False):
    """solve_wrapper (src/optflow.cpp:395-497).  output_type "flow" | "map" | "random_points"
    (default "map", :407).  Returns (flow_x, flow_y) after the frame1 <= 1 mask (:471-473); for
    "random_points" appends im_args["point_matches"].  With `features` (frame1 was moved by `affine`
    before the call) the map is moved by the same affine (:411-444) and the match q's come from the map."""
    frame0 = np.ascontiguousarray(frame0, np.uint8)
    frame1 = np.ascontiguousarray(frame1, np.uint8)
    tv = generate_TV_args(im_args, args)
    s = _solver_for(tv, device)
    h, w = frame0.shape
    output_type = _get(im_args, args, "output_type", "map")
    b0 = N.DevBuf(frame0.nbytes, device).upload(frame0)
    b1 = N.DevBuf(frame1.nbytes, device).upload(frame1)
    bu = N.DevBuf(w * h * 4, device)
    bv = N.DevBuf(w * h * 4, device)
    bufs = [b0, b1, bu, bv]
    try:
        s.calc_device(b0.ptr, w, b1.ptr, w, w, h, bu.ptr, bv.ptr, w * 4)
        if features:
            aff = np.ascontiguousarray(affine, np.float32).reshape(6)
            mx = N.DevBuf(w * h * 4, device)
            my = N.DevBuf(w * h * 4, device)
            bufs += [mx, my]
            s.finish_flow_device(None, 0, w, h, bu.ptr, bv.ptr, w * 4, 1)          # map = flow + grid, no mask yet
            for src, dst in ((bu, mx), (bv, my)):
                N.check(N.lib().tvl1_warp_affine_f32(src.ptr, w * 4, w, h, aff.ctypes.data, dst.ptr, w * 4, w, h, None))
            s.finish_flow_device(b1.ptr, w, w, h, mx.ptr, my.ptr, w * 4, -1 if output_type == "flow" else 0)
            bu, bv = mx, my
        else:
            # coordinate grid ("map") added BEFORE the mask in the reference (:445-466 then :471-473), so
            # masked pixels are 0, not their coordinate; both on the device, in one pass
            s.finish_flow_device(b1.ptr, w, w, h, bu.ptr, bv.ptr, w * 4, output_type == "map")
        flow_x = bu.download((h, w), np.float32)
        flow_y = bv.download((h, w), np.float32)
        if output_type == "random_points":
            debug = bool(args.get("debug", False))
            if seed is None:
                import time
                seed = -1 if debug else int(time.time())   # srand(time(0)) unless debug (:532-535)
            scale = np.float32(_get(im_args, args, "scale", 0.5))
            npoints = int(_get(im_args, args, "npoints", 25))
            px, py, qx, qy, wg, _ = s.sample_matches_device(
                b0.ptr, w, b1.ptr, w, bu.ptr, bv.ptr, w * 4, w, h, roi0=roi_vec[0], roi1=roi_vec[1],
                scale=float(scale), npoints=npoints, seed=seed, q_is_map=features)
            pm = im_args.get("point_matches") or {"p": [[], []], "q": [[], []], "w": []}
            im_args["point_matches"] = pm
            pm["p"][0] += px.tolist(); pm["p"][1] += py.tolist()
            pm["q"][0] += qx.tolist(); pm["q"][1] += qy.tolist()
            pm["w"] += [int(x) for x in wg.tolist()]
        return flow_x, flow_y
    finally:
        for b in bufs:
            b.free()


def random_points(flow_x, flow_y, im_args, args, roi_vec, frame0, frame1, device=0, seed=None):
    """random_points (src/optflow.cpp:522-572) given host flow planes and the two frames the
    mask is built from (src/optflow.cpp:488-493).  Appends to im_args["point_matches"]."""
    tv = generate_TV_args(im_args, args)
    s = _solver_for(tv, device)
    if seed is None:
        import time
        seed = -1 if bool(args.get("debug", False)) else int(time.time())
    scale = float(np.float32(_get(im_args, args, "scale", 0.5)))
    npoints = int(_get(im_args, args, "npoints", 25))
    px, py, qx, qy, wg, pos = s.sample_matches(frame0, frame1, flow_x, flow_y, roi0=roi_vec[0],
                                               roi1=roi_vec[1], scale=scale, npoints=npoints,
                                               seed=seed)
    pm = im_args.get("point_matches") or {"p": [[], []], "q": [[], []], "w": []}
    im_args["point_matches"] = pm
    pm["p"][0] += px.tolist(); pm["p"][1] += py.tolist()
    pm["q"][0] += qx.tolist(); pm["q"][1] += qy.tolist()
    pm["w"] += [int(x) for x in wg.tolist()]
    return pos


def move_pm(im_args, args):
    """Moves a pair's point matches into the job-level list (src/optflow.cpp:574-593)."""
    single_pair = {
        "pGroupId": im_args.get("pGroupId"), "pId": im_args.get("pId"),
        "qGroupId": im_args.get("qGroupId"), "qId": im_args.get("qId"),
        "matches": im_args.get("point_matches"),
    }
    args.setdefault("point_matches", []).append(single_pair)
    im_args["point_matches"] = {}
    return single_pair


def shard_pairs(n_pairs, world_size, rank):
    """Contiguous block of pair indices for one rank (SURVEY.md 8(e)): blocks, not round-robin,
    so the slice shared by adjacent pairs is uploaded once per GPU.  No collective follows."""
    base, rem = divmod(n_pairs, world_size)
    start = rank * base + min(rank, rem)
    return range(start, start + base + (1 if rank < rem else 0))
