"""The reference's `tf_ops` operator surface on torch CUDA tensors.

Same function names, argument orders and error behaviour as
  /root/reference/lib/utils/tf_ops/sampling/tf_sampling.py      (:24 gather_point, :43 farthest_point_sample,
                                                                  :54 farthest_point_sample_with_distance)
  /root/reference/lib/utils/tf_ops/grouping/tf_grouping.py      (:53 query_ball_point, :68 query_ball_point_dilated,
                                                                  :114 group_point)
  /root/reference/lib/utils/tf_ops/interpolation/tf_interpolate.py (:8 three_nn, :21 three_interpolate)
with the TF custom-op layer replaced by ctypes calls into libssd3d.so (include/ssd3d.h).  Shape / attribute
checks mirror the reference's OP_REQUIRES (InvalidArgument -> ValueError); outputs are allocated here, like
TF's allocate_output, and the kernels run on torch's current stream (CUDA-graph capturable).
"""
import ctypes

import torch

from ._lib import check, lib


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _p(t):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else ctypes.c_void_p(0)


def _req(t, name, dtype, rank, last=None, contiguous=True):
    if not isinstance(t, torch.Tensor):
        raise ValueError("%s must be a torch.Tensor" % name)
    if not t.is_cuda:
        raise ValueError("%s must be a CUDA tensor (there is no CPU path)" % name)
    if t.dtype != dtype:
        raise ValueError("%s must be %s, got %s" % (name, dtype, t.dtype))
    if t.dim() != rank:
        raise ValueError("%s must have rank %d, got shape %s" % (name, rank, tuple(t.shape)))
    if last is not None and t.shape[-1] != last:
        raise ValueError("%s must have last dimension %d, got shape %s" % (name, last, tuple(t.shape)))
    return t if (t.is_contiguous() or not contiguous) else t.contiguous()


def _scene_strided(t, name, rank=3, last=None):
    """A float32 CUDA tensor (b, n, c) whose rows are dense but whose scenes may be strided (a [:, a:b] slice of a
    dense tensor): returns (tensor, scene stride in floats) without copying; anything else is made contiguous."""
    t = _req(t, name, torch.float32, rank, last, contiguous=False)
    b, n, c = t.shape
    if c > 0 and n > 0 and t.stride(2) == 1 and t.stride(1) == c and (b <= 1 or t.stride(0) >= n * c):
        return t, (t.stride(0) if b > 1 else n * c)
    t = t.contiguous()
    return t, n * c


def _idx_out(out, b, npoint, device):
    """Resolve the optional (buffer, column) output placement of the sampling ops -> (tensor to return, ptr, ldo)."""
    if out is None:
        o = torch.empty((b, npoint), dtype=torch.int32, device=device)
        return o, o.data_ptr(), npoint
    buf, col = out
    if buf.dtype != torch.int32 or buf.dim() != 2 or not buf.is_contiguous() or buf.shape[0] != b or col < 0 or col + npoint > buf.shape[1]:
        raise ValueError("out must be (int32 contiguous (b, >= col + npoint) buffer, col)")
    return buf[:, col:col + npoint], buf.data_ptr() + 4 * col, buf.shape[1]


def _fps_flags(packet_kernel, bucket_kernel):
    return (1 if packet_kernel else 0) | (0 if bucket_kernel is None else (4 if bucket_kernel else 2))


def fps_temp_elems(n, c=3, npoint=0, packet_kernel=False, bucket_kernel=None):
    """float32 elements per scene of the `temp` buffer farthest_point_sample(..., rounds=...) carries its state in."""
    return int(lib().ssd3d_fps_temp_elems(int(n), int(c), int(npoint), _fps_flags(packet_kernel, bucket_kernel)))


def farthest_point_sample(npoint, inp, *, out=None, idx_offset=0, rounds=None, temp=None, cluster=0, packet_kernel=False,
                          bucket_kernel=None):
    """inp: (batch, ndataset, c) float32 -> (batch, npoint) int32.  tf_sampling.py:43-51; shape check
    tf_sampling.cpp:142 (rank 3).

    Keyword extensions (include/ssd3d.h, ssd3d_farthest_point_sample_ex; none changes the sampled indices):
      out=(buffer, col)   write into columns [col, col+npoint) of an int32 (batch, L) buffer and return that view;
      idx_offset          added to every index (segment offset of a fusion-sampling layer, layers_util.py:109);
      rounds=(j0, j1), temp   run only rounds [j0, j1); `temp` (batch, fps_temp_elems(n, c, npoint)) float32 carries the
                          running state between the calls (j0 == 0 starts fresh); the output must be the same buffer in
                          every call;
      cluster             CTAs per scene: 0 heuristic, >0 exact, <0 heuristic capped at -cluster;
      packet_kernel       use the general cluster kernel even where the resident-scene one applies (tests);
      bucket_kernel       None: automatic (xyz scenes of 8192 < n <= 16384 points take the single-CTA kernel with spatial
                          pruning, csrc/fps_bucket.cu), True / False: force (64 <= n <= 16384) / forbid it."""
    inp, stride = _scene_strided(inp, "inp")
    npoint = int(npoint)
    if npoint < 0:
        raise ValueError("npoint must be non-negative")
    b, n, c = inp.shape
    o, optr, ldo = _idx_out(out, b, npoint, inp.device)
    j0, j1 = (0, npoint) if rounds is None else (int(rounds[0]), int(rounds[1]))
    flags = _fps_flags(packet_kernel, bucket_kernel)
    elems = int(lib().ssd3d_fps_temp_elems(n, c, npoint, flags))
    if temp is None and (lib().ssd3d_fps_needs_temp(n, c) or (j0, j1) != (0, npoint)):
        if (j0, j1) != (0, npoint):
            raise ValueError("a partial range of rounds needs the caller's temp (batch, fps_temp_elems(...)) float32 buffer")
        temp = torch.empty((b, elems), dtype=torch.float32, device=inp.device)
    if temp is not None and (temp.dtype != torch.float32 or not temp.is_contiguous() or temp.numel() < b * elems):
        raise ValueError("temp must be a contiguous float32 buffer of at least batch * fps_temp_elems(n, c, npoint) elements")
    check(lib().ssd3d_farthest_point_sample_ex(b, n, c, npoint, _p(inp), stride, _p(temp), ctypes.c_void_p(optr), ldo,
                                               int(idx_offset), j0, j1, int(cluster), flags, _stream()),
          "farthest_point_sample")
    return o


furthest_point_sample = farthest_point_sample  # spelling used by BASELINE.json's north star


def fps_supports_rounds(n, c=3):
    """True when farthest_point_sample(..., rounds=...) is available for n points of c channels."""
    return bool(lib().ssd3d_fps_supports_rounds(int(n), int(c)))


def farthest_point_sample_with_distance(npoint, dist, *, out=None, idx_offset=0, cluster=0):
    """dist: (batch, n, n) float32 distance matrix -> (batch, npoint) int32.  tf_sampling.py:54-62; the
    square-matrix check is tf_sampling.cpp:175.  Keyword extensions as farthest_point_sample."""
    dist = _req(dist, "dist", torch.float32, 3)
    b, n, n2 = dist.shape
    if n != n2:
        raise ValueError("FarthestPointSampleWithDistance expects (batch_size,num_points,num_points) inp shape")
    npoint = int(npoint)
    o, optr, ldo = _idx_out(out, b, npoint, dist.device)
    temp = torch.empty((b, n), dtype=torch.float32, device=dist.device) if n > 65536 else None
    check(lib().ssd3d_farthest_point_sample_with_distance_ex(b, n, npoint, _p(dist), _p(temp), ctypes.c_void_p(optr), ldo,
                                                             int(idx_offset), int(cluster), _stream()),
          "farthest_point_sample_with_distance")
    return o


def ffps_supported(n, c):
    """True when the matrix-free F-FPS kernel covers n points with c concatenated channels."""
    return bool(lib().ssd3d_ffps_supported(int(n), int(c)))


def farthest_point_sample_features(npoint, xyz, points=None, *, out=None, idx_offset=0, rounds=None, temp=None):
    """F-FPS on concat[xyz, points] without the distance matrix: the same indices as
    farthest_point_sample_with_distance(npoint, calc_square_dist(concat[xyz, points])) (layers_util.py:94-96).
    Keyword extensions as farthest_point_sample (out, idx_offset, rounds + temp)."""
    xyz, sa = _scene_strided(xyz, "xyz")
    b, n, ca = xyz.shape
    cb, sb = 0, 0
    if points is not None and points.shape[-1] > 0:
        points, sb = _scene_strided(points, "points")
        if points.shape[:2] != (b, n):
            raise ValueError("points must be (batch, n, c) like xyz")
        cb = points.shape[2]
    else:
        points = None
    npoint = int(npoint)
    o, optr, ldo = _idx_out(out, b, npoint, xyz.device)
    j0, j1 = (0, npoint) if rounds is None else (int(rounds[0]), int(rounds[1]))
    if (j0, j1) != (0, npoint) and (temp is None or temp.dtype != torch.float32 or not temp.is_contiguous() or temp.numel() < b * n):
        raise ValueError("a partial range of rounds needs a contiguous float32 temp buffer of batch * n elements")
    check(lib().ssd3d_farthest_point_sample_features_ex(b, n, ca, cb, npoint, _p(xyz), sa, _p(points), sb, _p(temp),
                                                        ctypes.c_void_p(optr), ldo, int(idx_offset), j0, j1, _stream()),
          "farthest_point_sample_features")
    return o


def _gather_point_fwd(inp, idx):
    b, n, c = inp.shape
    m = idx.shape[1]
    out = torch.empty((b, m, c), dtype=torch.float32, device=inp.device)
    # idx may be a column block of a wider contiguous (b, L) tensor: read in place
    check(lib().ssd3d_gather_point_ex(b, n, m, c, _p(inp), _p(idx), idx.stride(0) if b > 1 else m, _p(out), _stream()),
          "gather_point")
    return out


def gather_point_grad(inp, idx, out_g):
    """Gradient of gather_point w.r.t. inp (tf_sampling.py:38-42 _gather_point_grad): scatter-add of out_g."""
    idx = _req(idx, "idx", torch.int32, 2)
    out_g = _req(out_g, "out_g", torch.float32, 3)
    b, n, c = inp.shape
    inp_g = torch.empty((b, n, c), dtype=torch.float32, device=out_g.device)
    check(lib().ssd3d_gather_point_grad(b, n, idx.shape[1], c, _p(out_g), _p(idx), _p(inp_g), _stream()), "gather_point_grad")
    return inp_g


class _GatherPoint(torch.autograd.Function):
    @staticmethod
    def forward(ctx, inp, idx):
        ctx.save_for_backward(idx)
        ctx.shape = inp.shape
        return _gather_point_fwd(inp, idx)

    @staticmethod
    def backward(ctx, out_g):
        (idx,) = ctx.saved_tensors
        return gather_point_grad(torch.empty(ctx.shape, device="meta"), idx, out_g.contiguous()), None


def gather_point(inp, idx):
    """inp (batch, ndataset, c) float32, idx (batch, npoints) int32 -> (batch, npoints, c).  tf_sampling.py:24-32.
    Differentiable w.r.t. inp (the reference registers GatherPoint's gradient, tf_sampling.py:37-42)."""
    inp = _req(inp, "inp", torch.float32, 3)
    if not (isinstance(idx, torch.Tensor) and idx.is_cuda and idx.dtype == torch.int32 and idx.dim() == 2
            and idx.stride(1) == 1 and idx.stride(0) >= idx.shape[1]):
        idx = _req(idx, "idx", torch.int32, 2)
    if idx.shape[0] != inp.shape[0]:
        raise ValueError("GatherPoint expects (batch_size,num_result) idx shape")
    if inp.requires_grad and torch.is_grad_enabled():
        return _GatherPoint.apply(inp, idx)
    return _gather_point_fwd(inp, idx)


def _bq_shapes(xyz1, xyz2):
    xyz1 = _req(xyz1, "xyz1", torch.float32, 3, 3)   # tf_grouping.cpp:283
    xyz2 = _req(xyz2, "xyz2", torch.float32, 3, 3)   # tf_grouping.cpp:288
    if xyz1.shape[0] != xyz2.shape[0]:
        raise ValueError("xyz1 and xyz2 must share the batch dimension")
    return xyz1, xyz2


def _query_ball(min_radius, max_radius, nsample, xyz1, xyz2, dilated):
    xyz1, xyz2 = _bq_shapes(xyz1, xyz2)
    op = "QueryBallPointDilated" if dilated else "QueryBallPoint"
    if not max_radius > 0:
        raise ValueError("%s expects positive radius" % op)              # tf_grouping.cpp:275
    if not int(nsample) > 0:
        raise ValueError("%s expects positive nsample" % op)             # tf_grouping.cpp:278
    b, n, _ = xyz1.shape
    m = xyz2.shape[1]
    if n >= BQ_GRID_MIN_N and lib().ssd3d_query_ball_point_workspace(b, n):
        i, c = query_ball_point_multi([min_radius], [max_radius], [nsample], xyz1, xyz2, dilated)
        return i[0], c[0]
    idx = torch.empty((b, m, int(nsample)), dtype=torch.int32, device=xyz1.device)
    cnt = torch.empty((b, m), dtype=torch.int32, device=xyz1.device)
    io = (_p(xyz1), _p(xyz2), _p(idx), _p(cnt), _stream())
    if dilated:
        check(lib().ssd3d_query_ball_point_dilated(b, n, m, float(min_radius), float(max_radius), int(nsample), *io),
              "query_ball_point_dilated")
    else:
        check(lib().ssd3d_query_ball_point(b, n, m, float(max_radius), int(nsample), *io), "query_ball_point")
    return idx, cnt


def query_ball_point(radius, nsample, xyz1, xyz2):
    """xyz1 (batch, ndataset, 3), xyz2 (batch, npoint, 3) -> idx (batch, npoint, nsample) int32,
    pts_cnt (batch, npoint) int32.  tf_grouping.py:53-65."""
    return _query_ball(0.0, radius, nsample, xyz1, xyz2, False)


def query_ball_point_dilated(min_radius, max_radius, nsample, xyz1, xyz2):
    """Shell query  d == 0 or min_radius <= d < max_radius.  tf_grouping.py:68-81."""
    return _query_ball(min_radius, max_radius, nsample, xyz1, xyz2, True)


BQ_GRID_MIN_N = 2048     # candidate sets at least this large take the spatially culled kernel (csrc/ball_query_grid.cu)


def query_ball_point_multi(min_radius_list, max_radius_list, nsample_list, xyz1, xyz2, dilated, grid=None, return_units=False):
    """All radius shells of one SA layer in a single pass over the candidates (B200 fast path; same results
    as calling query_ball_point[_dilated] once per shell).  Returns lists (idx_list, pts_cnt_list).
    grid: None = automatic (the culled kernel for ndataset >= BQ_GRID_MIN_N), True / False = force / forbid it;
    the outputs are identical either way.
    return_units: also return, per shell, the UNIT LIST of the grouped MLP (int32 tensor, include/ssd3d.h
    ssd3d_query_ball_point_multi_ws), or None for nsample > 128: (idx_list, pts_cnt_list, units_list)."""
    xyz1, xyz2 = _bq_shapes(xyz1, xyz2)
    nq = len(max_radius_list)
    if not (len(nsample_list) == nq and len(min_radius_list) == nq and 1 <= nq <= 4):
        raise ValueError("query_ball_point_multi takes 1..4 shells with matching list lengths")
    for r, k in zip(max_radius_list, nsample_list):
        if not r > 0:
            raise ValueError("QueryBallPoint expects positive radius")
        if not int(k) > 0:
            raise ValueError("QueryBallPoint expects positive nsample")
    b, n, _ = xyz1.shape
    m = xyz2.shape[1]
    idx = [torch.empty((b, m, int(k)), dtype=torch.int32, device=xyz1.device) for k in nsample_list]
    cnt = [torch.empty((b, m), dtype=torch.int32, device=xyz1.device) for _ in nsample_list]
    lo = (ctypes.c_float * nq)(*[float(v) for v in min_radius_list])
    hi = (ctypes.c_float * nq)(*[float(v) for v in max_radius_list])
    ks = (ctypes.c_int * nq)(*[int(v) for v in nsample_list])
    pi = (ctypes.c_void_p * nq)(*[t.data_ptr() for t in idx])
    pc = (ctypes.c_void_p * nq)(*[t.data_ptr() for t in cnt])
    ws_bytes = int(lib().ssd3d_query_ball_point_workspace(b, n)) if (b and m) else 0
    use_grid = ws_bytes > 0 and (n >= BQ_GRID_MIN_N if grid is None else bool(grid))
    if grid and not use_grid and b and m:
        raise ValueError("the culled ball query covers ndataset <= 16384, got %d" % n)
    ws = torch.empty((ws_bytes,), dtype=torch.uint8, device=xyz1.device) if use_grid else None
    units = [None] * nq
    pu = ctypes.c_void_p(0)
    if return_units and all(int(k) <= 128 for k in nsample_list):
        units = [torch.empty((1 + b * m * ((int(k) + 7) // 8),), dtype=torch.int32, device=xyz1.device) for k in nsample_list]
        parr = (ctypes.c_void_p * nq)(*[t.data_ptr() for t in units])
        pu = ctypes.cast(parr, ctypes.c_void_p)
    check(lib().ssd3d_query_ball_point_multi_ws(b, n, m, nq, 1 if dilated else 0, ctypes.cast(lo, ctypes.c_void_p),
                                                ctypes.cast(hi, ctypes.c_void_p), ctypes.cast(ks, ctypes.c_void_p),
                                                _p(xyz1), _p(xyz2), ctypes.cast(pi, ctypes.c_void_p),
                                                ctypes.cast(pc, ctypes.c_void_p), pu, _p(ws), ws_bytes if use_grid else 0,
                                                _stream()), "query_ball_point_multi")
    if return_units:
        return idx, cnt, units
    return idx, cnt


def _group_point_fwd(points, idx):
    b, n, c = points.shape
    _, m, ns = idx.shape
    out = torch.empty((b, m, ns, c), dtype=torch.float32, device=points.device)
    check(lib().ssd3d_group_point(b, n, c, m, ns, _p(points), _p(idx), _p(out), _stream()), "group_point")
    return out


def group_point_grad(points, idx, grad_out):
    """Gradient of group_point w.r.t. points (tf_grouping.py:123-128 _group_point_grad)."""
    idx = _req(idx, "idx", torch.int32, 3)
    grad_out = _req(grad_out, "grad_out", torch.float32, 4)
    b, n, c = points.shape
    _, m, ns = idx.shape
    g = torch.empty((b, n, c), dtype=torch.float32, device=grad_out.device)
    check(lib().ssd3d_group_point_grad(b, n, c, m, ns, _p(grad_out), _p(idx), _p(g), _stream()), "group_point_grad")
    return g


class _GroupPoint(torch.autograd.Function):
    @staticmethod
    def forward(ctx, points, idx):
        ctx.save_for_backward(idx)
        ctx.shape = points.shape
        return _group_point_fwd(points, idx)

    @staticmethod
    def backward(ctx, grad_out):
        (idx,) = ctx.saved_tensors
        return group_point_grad(torch.empty(ctx.shape, device="meta"), idx, grad_out.contiguous()), None


def group_point(points, idx):
    """points (batch, ndataset, channel) float32, idx (batch, npoint, nsample) int32 ->
    (batch, npoint, nsample, channel); idx == -1 gives zeros.  tf_grouping.py:114-122; differentiable w.r.t. points."""
    points = _req(points, "points", torch.float32, 3)
    idx = _req(idx, "idx", torch.int32, 3)
    if idx.shape[0] != points.shape[0]:
        raise ValueError("GroupPoint expects (batch_size, npoints, nsample) idx shape")
    if points.requires_grad and torch.is_grad_enabled():
        return _GroupPoint.apply(points, idx)
    return _group_point_fwd(points, idx)


def three_nn(xyz1, xyz2):
    """xyz1 (b,n,3) unknown, xyz2 (b,m,3) known -> dist (b,n,3) float32 (squared), idx (b,n,3) int32.
    tf_interpolate.py:8-19."""
    xyz1 = _req(xyz1, "xyz1", torch.float32, 3, 3)   # tf_interpolate.cpp:222
    xyz2 = _req(xyz2, "xyz2", torch.float32, 3, 3)   # tf_interpolate.cpp:227
    if xyz1.shape[0] != xyz2.shape[0]:
        raise ValueError("xyz1 and xyz2 must share the batch dimension")
    b, n, _ = xyz1.shape
    m = xyz2.shape[1]
    dist = torch.empty((b, n, 3), dtype=torch.float32, device=xyz1.device)
    idx = torch.empty((b, n, 3), dtype=torch.int32, device=xyz1.device)
    check(lib().ssd3d_three_nn(b, n, m, _p(xyz1), _p(xyz2), _p(dist), _p(idx), _stream()), "three_nn")
    return dist, idx


def three_interpolate(points, idx, weight):
    """points (b,m,c), idx (b,n,3) int32, weight (b,n,3) -> (b,n,c).  tf_interpolate.py:21-31."""
    points = _req(points, "points", torch.float32, 3)
    idx = _req(idx, "idx", torch.int32, 3, 3)
    weight = _req(weight, "weight", torch.float32, 3, 3)
    b, m, c = points.shape
    n = idx.shape[1]
    if idx.shape[0] != b or weight.shape != idx.shape:
        raise ValueError("ThreeInterpolate expects (b,n,3) idx and weight shapes")
    if points.requires_grad and torch.is_grad_enabled():
        return _ThreeInterpolate.apply(points, idx, weight)
    return _three_interpolate_fwd(points, idx, weight)


def _three_interpolate_fwd(points, idx, weight):
    b, m, c = points.shape
    n = idx.shape[1]
    out = torch.empty((b, n, c), dtype=torch.float32, device=points.device)
    check(lib().ssd3d_three_interpolate(b, m, c, n, _p(points), _p(idx), _p(weight), _p(out), _stream()),
          "three_interpolate")
    return out


def three_interpolate_grad(points, idx, weight, grad_out):
    """Gradient of three_interpolate w.r.t. points (tf_interpolate.py:32-37 _three_interpolate_grad)."""
    grad_out = _req(grad_out, "grad_out", torch.float32, 3)
    b, m, c = points.shape
    n = idx.shape[1]
    g = torch.empty((b, m, c), dtype=torch.float32, device=grad_out.device)
    check(lib().ssd3d_three_interpolate_grad(b, n, c, m, _p(grad_out), _p(idx), _p(weight), _p(g), _stream()),
          "three_interpolate_grad")
    return g


class _ThreeInterpolate(torch.autograd.Function):
    @staticmethod
    def forward(ctx, points, idx, weight):
        ctx.save_for_backward(idx, weight)
        ctx.shape = points.shape
        return _three_interpolate_fwd(points, idx, weight)

    @staticmethod
    def backward(ctx, grad_out):
        idx, weight = ctx.saved_tensors
        return three_interpolate_grad(torch.empty(ctx.shape, device="meta"), idx, weight, grad_out.contiguous()), None, None


# ---- dense pieces that are stock TF ops in the reference -------------------------------------------------

def calc_square_dist(a):
    """model_util.calc_square_dist(a, a, norm=False) (/root/reference/lib/utils/model_util.py:144-160)."""
    a = _req(a, "a", torch.float32, 3)
    b, n, c = a.shape
    out = torch.empty((b, n, n), dtype=torch.float32, device=a.device)
    check(lib().ssd3d_calc_square_dist(b, n, c, _p(a), _p(out), _stream()), "calc_square_dist")
    return out


def _grouping(xyz, points, new_xyz, idx):
    """Checks of the grouping inputs xyz (b, n, 3), points (b, n, c) or None, new_xyz (b, m, 3), idx (b, m, nsample)
    -> (xyz, points, new_xyz, idx, c)."""
    xyz = _req(xyz, "xyz", torch.float32, 3, 3)
    new_xyz = _req(new_xyz, "new_xyz", torch.float32, 3, 3)
    idx = _req(idx, "idx", torch.int32, 3)
    c = 0
    if points is not None:
        points = _req(points, "points", torch.float32, 3)
        c = points.shape[2]
    return xyz, points, new_xyz, idx, c


def group_concat(xyz, points, new_xyz, idx, ldx=None):
    """concat[group_point(points, idx), group_point(xyz, idx) - new_xyz] (layers_util.py:160-165) in one kernel.
    Returns x (b, m, nsample, ldx) with zero padding beyond c+3."""
    xyz, points, new_xyz, idx, c = _grouping(xyz, points, new_xyz, idx)
    b, n, _ = xyz.shape
    _, m, ns = idx.shape
    ldx = c + 3 if ldx is None else int(ldx)
    x = torch.empty((b, m, ns, ldx), dtype=torch.float32, device=xyz.device)
    check(lib().ssd3d_group_concat(b, n, c, m, ns, _p(xyz), _p(points), _p(new_xyz), _p(idx), _p(x), ldx, _stream()),
          "group_concat")
    return x


def linear_bn_relu(x, w, scale, shift, relu=True, pool=1, rowmask=None, cin=None):
    """act((x[..., :cin] @ w) * scale + shift) over the last axis; pool > 1 max-pools runs of `pool` rows and
    multiplies by rowmask != 0 (layers_util.py:178-180).  x (..., ldx), w (cin, cout)."""
    if x.dtype != torch.float32 or not x.is_cuda:
        raise ValueError("x must be a float32 CUDA tensor")
    x = x if x.is_contiguous() else x.contiguous()
    w = _req(w, "w", torch.float32, 2)
    wcin, cout = w.shape
    cin = wcin if cin is None else cin
    ldx = x.shape[-1]
    if cin != wcin or ldx < cin:
        raise ValueError("linear_bn_relu: x last dim %d / cin %d do not match w %s" % (ldx, cin, tuple(w.shape)))
    rows = x.numel() // ldx
    pool = int(pool)
    lead = tuple(x.shape[:-1])
    if pool > 1:
        if lead[-1] != pool:
            raise ValueError("pool must equal the second-to-last dimension of x")
        if 128 % pool != 0:
            y = linear_bn_relu(x, w, scale, shift, relu, 1, None, cin)
            out = torch.empty(lead[:-1] + (cout,), dtype=torch.float32, device=x.device)
            check(lib().ssd3d_rowgroup_max(rows // pool, pool, cout, _p(y), cout, _p(rowmask), _p(out), _stream()),
                  "rowgroup_max")
            return out
        y = torch.empty(lead[:-1] + (cout,), dtype=torch.float32, device=x.device)
    else:
        y = torch.empty(lead + (cout,), dtype=torch.float32, device=x.device)
    check(lib().ssd3d_linear_bn_relu(rows, cin, cout, _p(x), ldx, _p(w), _p(scale), _p(shift), 1 if relu else 0, pool,
                                     _p(rowmask), _p(y), cout, _stream()), "linear_bn_relu")
    return y


# ---- tensor-core (tcgen05) path of the MLP: operands split in two bf16 terms ---------------------------------

def round16(x):
    return (int(x) + 15) // 16 * 16


def split_rows(x, kp=None):
    """fp32 (..., c) -> (hi, lo) bf16 (..., kp) with hi + lo ~= x (16 mantissa bits), zero padded to kp."""
    if x.dtype != torch.float32 or not x.is_cuda:
        raise ValueError("x must be a float32 CUDA tensor")
    x = x if x.is_contiguous() else x.contiguous()
    c = x.shape[-1]
    kp = round16(c) if kp is None else int(kp)
    rows = x.numel() // c
    hi = torch.empty(tuple(x.shape[:-1]) + (kp,), dtype=torch.bfloat16, device=x.device)
    lo = torch.empty_like(hi)
    check(lib().ssd3d_split_rows(rows, c, _p(x), c, _p(hi), _p(lo), kp, _stream()), "split_rows")
    return hi, lo


def group_concat_split(xyz, points, new_xyz, idx, kp=None):
    """group_concat + split in one kernel: (hi, lo) bf16 (b, m, nsample, kp)."""
    xyz, points, new_xyz, idx, c = _grouping(xyz, points, new_xyz, idx)
    b, n, _ = xyz.shape
    _, m, ns = idx.shape
    kp = round16(c + 3) if kp is None else int(kp)
    hi = torch.empty((b, m, ns, kp), dtype=torch.bfloat16, device=xyz.device)
    lo = torch.empty_like(hi)
    check(lib().ssd3d_group_concat_split(b, n, c, m, ns, _p(xyz), _p(points), _p(new_xyz), _p(idx), _p(hi), _p(lo), kp,
                                         _stream()), "group_concat_split")
    return hi, lo


def _hoisted(z, zoff, wx, b, n, aligned=False):
    """Checks of the hoisted inputs: z (b, n, ldz) fp32 holding this scale's n1 columns from zoff, wx (3, n1); aligned:
    ldz and zoff multiples of 4.  Returns (z, (pointer to column zoff, ldz), wx, n1)."""
    z = _req(z, "z", torch.float32, 3)
    wx = _req(wx, "wx", torch.float32, 2)
    n1 = wx.shape[1]
    if (z.shape[:2] != (b, n) or wx.shape[0] != 3 or zoff < 0 or zoff + n1 > z.shape[2]
            or (aligned and (zoff % 4 or z.shape[2] % 4))):
        raise ValueError("z must be (b, n, ldz) with zoff + n1 <= ldz%s, and wx (3, n1)" % (", ldz and zoff multiples of 4" * aligned))
    return z, (ctypes.c_void_p(z.data_ptr() + 4 * zoff), z.shape[2]), wx, n1


def _pooled(pool, lead):
    """A pool width over rows of leading shape (..., nsample) -> (pool, leading shape of the outputs)."""
    pool = int(pool)
    if pool > 1 and (lead[-1] != pool or pool not in (8, 16, 32, 64, 128)):
        raise ValueError("pool must equal nsample (the second-to-last dimension) and be one of 8, 16, 32, 64, 128")
    return pool, (lead[:-1] if pool > 1 else lead)


def _units_check(units, unit_pool=False, pool=1, rowmask=None, relu=True, out_f32=None, out_split=None, want_split=False):
    """units: None, or the int32 CUDA unit list of query_ball_point_multi(return_units=True), which replaces pool / rowmask.
    unit_pool: every listed 8-row unit is max-pooled into its group's row of out_f32 by atomicMax (a zero-filled buffer)."""
    if units is None:
        if unit_pool:
            raise ValueError("unit_pool needs a unit list")
        return
    if units.dtype != torch.int32 or not units.is_cuda or not units.is_contiguous():
        raise ValueError("units must be the int32 CUDA unit list returned by query_ball_point_multi(return_units=True)")
    if int(pool) != 1 or rowmask is not None:
        raise ValueError("a unit list replaces pool / rowmask (unit_pool=True pools the listed 8-row units)")
    if unit_pool and (not relu or out_f32 is None or out_split is not None or want_split):
        raise ValueError("pooling 8-row units needs relu, out_f32=(zero-filled buffer, col_offset) and no split output")


def _tc_outputs(lead, n, pool, dev, want_f32, want_split, out_f32, out_split):
    """Output placement of the tensor-core kernels -> (y, (hi, lo), C arguments (f32 ptr, ldf, hi ptr, lo ptr, lds)).
    out_f32=(buffer, col) / out_split=(hi, lo, col) write into column slices of the caller's buffers, otherwise want_f32 /
    want_split allocate lead + (n,) results (split ones padded to 16 columns, zero-filled when pooled)."""
    y, pf, ldf = None, 0, 0
    if out_f32 is not None:
        y, off = out_f32
        pf, ldf = y.data_ptr() + 4 * off, y.shape[-1]
    elif want_f32:
        y = torch.empty(lead + (n,), dtype=torch.float32, device=dev)
        pf, ldf = y.data_ptr(), n
    sp, ph, pl, lds = None, 0, 0, 0
    if out_split is not None:
        hb, lb, off = out_split
        sp, ph, pl, lds = (hb, lb), hb.data_ptr() + 2 * off, lb.data_ptr() + 2 * off, hb.shape[-1]
    elif want_split:
        lds = round16(n)
        alloc = torch.zeros if (pool > 1 and lds != n) else torch.empty
        sp = tuple(alloc(lead + (lds,), dtype=torch.bfloat16, device=dev) for _ in range(2))
        ph, pl = sp[0].data_ptr(), sp[1].data_ptr()
    vp = ctypes.c_void_p
    return y, sp, (vp(pf), ldf, vp(ph), vp(pl), lds)


def _layer(f, relu):
    return _p(f.b_hi), _p(f.b_lo), _p(f.scale), _p(f.shift), 1 if relu else 0


def linear_tc(a_hi, a_lo, f, relu=True, pool=1, rowmask=None, want_f32=True, want_split=False, out_f32=None,
              out_split=None, units=None, unit_pool=False):
    """One folded conv layer on the tensor cores.  a_hi/a_lo (..., kp) bf16; f: params.FoldedConv.
    Returns (y_f32 or None, (hi, lo) or None).  out_f32=(buffer, col_offset) / out_split=(hi_buf, lo_buf, col_offset)
    write into slices of preallocated (..., ld) buffers (the concat of the SA scales) instead of allocating.
    units: the operand holds COMPACT rows (8 per listed unit, include/ssd3d.h ssd3d_linear_tc_units) in its first
    units[0] * 8 rows; outputs are compact likewise, or -- unit_pool=True, the last conv of a scale -- every unit is
    max-pooled and combined into out_f32[group] by atomicMax (buffer zero-filled by the caller)."""
    _units_check(units, unit_pool, pool, rowmask, relu, out_f32, out_split, want_split)
    if a_hi.dtype != torch.bfloat16 or a_lo.dtype != torch.bfloat16 or a_hi.shape != a_lo.shape:
        raise ValueError("a_hi / a_lo must be bfloat16 tensors of the same shape")
    kp = a_hi.shape[-1]
    if kp != f.kp:
        raise ValueError("operand K (%d) does not match the layer's padded K (%d)" % (kp, f.kp))
    rows = a_hi.numel() // kp
    pool, lead = _pooled(pool, tuple(a_hi.shape[:-1]))
    y, sp, io = _tc_outputs(lead, f.cout, pool, a_hi.device, want_f32, want_split, out_f32, out_split)
    a = (rows, kp, f.cout, _p(a_hi), _p(a_lo)) + _layer(f, relu)
    if units is not None:
        check(lib().ssd3d_linear_tc_units(*a, _p(units), 1 if unit_pool else 0, *io, _stream()), "linear_tc_units")
    else:
        check(lib().ssd3d_linear_tc(*a, pool, _p(rowmask), *io, _stream()), "linear_tc")
    return y, sp


def linear_tc_gather(xyz, points, new_xyz, idx, f, relu=True, pool=1, rowmask=None, want_f32=False, want_split=True,
                     out_f32=None, out_split=None):
    """First conv layer of an SA scale with the gather / centre-subtract / concat of layers_util.py:160-165 fused
    into the tensor-core kernel's operand load (no [B,M,K,C] tensor in HBM).  Outputs as linear_tc, leading shape
    (b, m, nsample) or (b, m) when pooled."""
    xyz, points, new_xyz, idx, c = _grouping(xyz, points, new_xyz, idx)
    if round16(c + 3) != f.kp or c + 3 != f.cin:
        raise ValueError("layer input width %d does not match c+3 = %d" % (f.cin, c + 3))
    b, n, _ = xyz.shape
    _, m, ns = idx.shape
    pool, lead = _pooled(pool, (b, m, ns))
    y, sp, io = _tc_outputs(lead, f.cout, pool, xyz.device, want_f32, want_split, out_f32, out_split)
    check(lib().ssd3d_linear_tc_gather(b, n, c, m, ns, _p(xyz), _p(points), _p(new_xyz), _p(idx), f.cout, *_layer(f, relu),
                                       pool, _p(rowmask), *io, _stream()), "linear_tc_gather")
    return y, sp


def linear_tc_hoisted(xyz, z, zoff, wx, new_xyz, idx, f, relu=True, pool=1, rowmask=None, want_f32=False, want_split=True,
                      out_f32=None, out_split=None, units=None, unit_pool=False):
    """Second conv of an SA scale fed by the hoisted first conv (include/ssd3d.h, ssd3d_linear_tc_hoisted).
    z: (b, n, ldz) fp32 per-point table = (features . Wf) * s1 + t1 for all scales of the layer, this scale's
    columns start at zoff; wx: (3, n1) fp32 = Wx * s1; f: params.FoldedConv of the second conv (cin == n1).
    units / unit_pool: as linear_tc (the source rows are looked up through the list, outputs are compact)."""
    _units_check(units, unit_pool, pool, rowmask, relu, out_f32, out_split, want_split)
    xyz, _, new_xyz, idx, _ = _grouping(xyz, None, new_xyz, idx)
    b, n, _ = xyz.shape
    z, zcols, wx, n1 = _hoisted(z, zoff, wx, b, n)
    if f.cin != n1:
        raise ValueError("second conv expects %d inputs, the hoisted first conv has %d outputs" % (f.cin, n1))
    _, m, ns = idx.shape
    pool, lead = _pooled(pool, (b, m, ns))
    y, sp, io = _tc_outputs(lead, f.cout, pool, xyz.device, want_f32, want_split, out_f32, out_split)
    a = (b, n, n1, m, ns, _p(xyz), *zcols, _p(wx), _p(new_xyz), _p(idx))
    if units is not None:
        check(lib().ssd3d_linear_tc_hoisted_units(*a, _p(units), f.cout, *_layer(f, relu), 1 if unit_pool else 0, *io,
                                                  _stream()), "linear_tc_hoisted_units")
    else:
        check(lib().ssd3d_linear_tc_hoisted(*a, f.cout, *_layer(f, relu), pool, _p(rowmask), *io, _stream()),
              "linear_tc_hoisted")
    return y, sp


def hoist_expand_split(xyz, z, zoff, wx, new_xyz, idx, units=None):
    """The operand linear_tc_hoisted would build in its producer warps, materialised: (hi, lo) bf16 (b, m, nsample, kp) =
    split(relu(z[idx] + (xyz[idx] - new_xyz) . wx)).  Followed by the plain linear_tc this is the faster route for wide
    layers (K >= 256), where the resident operand of the in-kernel route leaves the weight ring two narrow stages.
    units: only the listed 8-row units are built, as compact rows at the start of the buffers."""
    _units_check(units)
    xyz, _, new_xyz, idx, _ = _grouping(xyz, None, new_xyz, idx)
    b, n, _ = xyz.shape
    z, zcols, wx, n1 = _hoisted(z, zoff, wx, b, n, aligned=True)
    _, m, ns = idx.shape
    kp = round16(n1)
    hi = torch.empty((b, m, ns, kp), dtype=torch.bfloat16, device=xyz.device)
    lo = torch.empty_like(hi)
    a = (b, n, n1, m, ns, _p(xyz), *zcols, _p(wx), _p(new_xyz), _p(idx))
    if units is not None:
        check(lib().ssd3d_hoist_expand_split_units(*a, _p(units), _p(hi), _p(lo), kp, _stream()), "hoist_expand_split_units")
    else:
        check(lib().ssd3d_hoist_expand_split(*a, _p(hi), _p(lo), kp, _stream()), "hoist_expand_split")
    return hi, lo


def _stack(stack):
    nout = (ctypes.c_int * len(stack.nout))(*stack.nout)        # the cast keeps the array alive
    return (len(stack.nout), ctypes.cast(nout, ctypes.c_void_p), _p(stack.w_blob), _p(stack.ss_blob),
            1 if stack.last_scale_nonneg else 0)


def sa_mlp_fused(xyz, points, new_xyz, idx, cnt, stack, out_f32=None, out_split=None, units=None):
    """One SA scale in one kernel: gather + concat + conv stack + max-pool + mask (layers_util.py:157-180).
    stack: params.FusedStack.  out_f32=(buffer, col_offset) / out_split=(hi, lo, col_offset) as linear_tc;
    without them a fresh (b, m, C3) fp32 tensor is returned.
    units: the scale's unit list (query_ball_point_multi(return_units=True)): only the listed 8-row units are convolved
    -- the skipped rows repeat a group's first neighbour and cannot change the max-pool -- and results are combined with
    atomicMax into out_f32, which must be zero-filled (fill_zero)."""
    _units_check(units, units is not None, out_f32=out_f32, out_split=out_split)
    xyz, points, new_xyz, idx, c = _grouping(xyz, points, new_xyz, idx)
    if c + 3 != stack.cin:
        raise ValueError("feature channels (%d) do not match the stack's input width (%d)" % (c, stack.cin - 3))
    b, n, _ = xyz.shape
    _, m, ns = idx.shape
    y, _, io = _tc_outputs((b, m), stack.nout[-1], 1, xyz.device, out_split is None, False, out_f32, out_split)
    check(lib().ssd3d_sa_mlp_fused(b, n, c, m, ns, _p(xyz), _p(points), _p(new_xyz), _p(idx), _p(cnt), _p(units),
                                   *_stack(stack), *io, _stream()), "sa_mlp_fused")
    return y


def sa_mlp_fused_hoisted(xyz, z, zoff, wx, new_xyz, idx, cnt, stack, out_f32=None, out_split=None, units=None):
    """sa_mlp_fused with the scale's first conv hoisted into the per-point table z (see linear_tc_hoisted): `stack` is the
    params.FusedStack of the REMAINING convs (its input width == wx.shape[1]).  units: as sa_mlp_fused."""
    _units_check(units, units is not None, out_f32=out_f32, out_split=out_split)
    xyz, _, new_xyz, idx, _ = _grouping(xyz, None, new_xyz, idx)
    b, n, _ = xyz.shape
    z, zcols, wx, n1 = _hoisted(z, zoff, wx, b, n)
    if n1 != stack.cin:
        raise ValueError("hoisted width (%d) does not match the stack's input width (%d)" % (n1, stack.cin))
    _, m, ns = idx.shape
    y, _, io = _tc_outputs((b, m), stack.nout[-1], 1, xyz.device, out_split is None, False, out_f32, out_split)
    check(lib().ssd3d_sa_mlp_fused_hoisted(b, n, n1, m, ns, _p(xyz), *zcols, _p(wx), _p(new_xyz), _p(idx), _p(cnt), _p(units),
                                           *_stack(stack), *io, _stream()), "sa_mlp_fused_hoisted")
    return y


def bev_nms(boxes, scores, iou_threshold, max_output, cls_id=0, out=None):
    """Greedy BEV NMS per scene (postprocessor.py:76-88): boxes (b,n,7) = (x,y,z,l,h,w,ry), scores (b,n) ->
    block (b,max_output,9) = (box7, score, class) zero padded, count (b,) int32.  out=(block, count) writes into
    preallocated contiguous tensors (the send buffer of the multi-GPU gather)."""
    boxes = _req(boxes, "boxes", torch.float32, 3, 7)
    scores = _req(scores, "scores", torch.float32, 2)
    b, n, _ = boxes.shape
    if scores.shape != (b, n):
        raise ValueError("scores must be (b, n)")
    if out is None:
        block = torch.empty((b, int(max_output), 9), dtype=torch.float32, device=boxes.device)
        cnt = torch.empty((b,), dtype=torch.int32, device=boxes.device)
    else:
        block, cnt = out
        if (block.dtype != torch.float32 or tuple(block.shape) != (b, int(max_output), 9) or not block.is_contiguous()
                or cnt.dtype != torch.int32 or tuple(cnt.shape) != (b,) or not cnt.is_contiguous()):
            raise ValueError("out must be (float32 (b, max_output, 9), int32 (b,)) contiguous tensors")
    check(lib().ssd3d_bev_nms(b, n, _p(boxes), _p(scores), float(iou_threshold), int(max_output), int(cls_id),
                              _p(block), _p(cnt), _stream()), "bev_nms")
    return block, cnt


# ---- the small elementwise stages (csrc/misc.cu): one kernel each, so a captured step holds no framework kernels ----

def fill_zero(t):
    """t[...] = 0 for a contiguous float32 CUDA tensor, as a kernel of this library."""
    if t.dtype != torch.float32 or not t.is_cuda or not t.is_contiguous():
        raise ValueError("fill_zero takes a contiguous float32 CUDA tensor")
    check(lib().ssd3d_fill_zero(_p(t), t.numel(), _stream()), "fill_zero")
    return t


def peer_allgather(send, peers, world, rank, slice_bytes, recv_off, flag_off, state, out):
    """All-gather of one slice per rank over NVLink peer memory (include/ssd3d.h, ssd3d_peer_allgather).
    send: uint8 [slice_bytes]; peers: int64 CUDA tensor [world] of the ranks' symmetric-buffer bases as mapped in THIS
    process; state: int32 [>= 3] zero-initialised, owned by this exchange (state[2] counts waits that timed out); out: uint8
    [world * slice_bytes]."""
    for name, t, dt in (("send", send, torch.uint8), ("peers", peers, torch.int64), ("state", state, torch.int32), ("out", out, torch.uint8)):
        if t.dtype != dt or not t.is_cuda or not t.is_contiguous():
            raise ValueError("%s must be a contiguous CUDA tensor of %s" % (name, dt))
    if send.numel() < slice_bytes or out.numel() < world * slice_bytes or peers.numel() < world or state.numel() < 3:
        raise ValueError("peer_allgather: buffers smaller than world=%d slices of %d bytes" % (world, slice_bytes))
    check(lib().ssd3d_peer_allgather(_p(send), int(slice_bytes), _p(peers), int(world), int(rank), int(recv_off[0]), int(recv_off[1]),
                                     int(flag_off[0]), int(flag_off[1]), _p(state), _p(out), _stream()), "peer_allgather")
    return out


def split_points(points):
    """(b, n, 3 + c) -> xyz (b, n, 3), features (b, n, c): single_stage_detector.py:116-117."""
    points = _req(points, "points", torch.float32, 3)
    b, n, c = points.shape
    if c < 3:
        raise ValueError("points must have at least 3 channels")
    xyz = torch.empty((b, n, 3), dtype=torch.float32, device=points.device)
    feat = torch.empty((b, n, c - 3), dtype=torch.float32, device=points.device)
    check(lib().ssd3d_split_points(b * n, c, _p(points), _p(xyz), _p(feat) if c > 3 else ctypes.c_void_p(0), _stream()),
          "split_points")
    return xyz, feat


def iota_idx(b, npoint, device, *, out=None, start=0):
    """tf.tile(tf.range(npoint)) + start: the identity sampling of layers_util.py:91-92, :100-101."""
    o, optr, ldo = _idx_out(out, b, int(npoint), device)
    check(lib().ssd3d_iota_idx(b, int(npoint), int(start), ctypes.c_void_p(optr), ldo, _stream()), "iota_idx")
    return o


def concat_cols(a, bsrc):
    """tf.concat([a, bsrc], -1) for (b, n, ca) / (b, n, cb) float32 tensors whose scenes may be strided."""
    a, sa = _scene_strided(a, "a")
    bsrc, sb = _scene_strided(bsrc, "bsrc")
    b, n, ca = a.shape
    if bsrc.shape[:2] != (b, n):
        raise ValueError("concat_cols: leading shapes differ")
    cb = bsrc.shape[2]
    out = torch.empty((b, n, ca + cb), dtype=torch.float32, device=a.device)
    check(lib().ssd3d_concat_cols(b, n, ca, cb, _p(a), sa, _p(bsrc), sb, _p(out), _stream()), "concat_cols")
    return out


def vote_translate(xyz, offsets, min_range):
    """xyz + min(max(offsets, min_range), -min_range) (layers_util.py:20-23); offsets (b, n, >= 3)."""
    xyz = _req(xyz, "xyz", torch.float32, 3, 3)
    offsets = _req(offsets, "offsets", torch.float32, 3)
    if offsets.shape[:2] != xyz.shape[:2] or offsets.shape[2] < 3:
        raise ValueError("offsets must be (b, n, >= 3) like xyz")
    out = torch.empty_like(xyz)
    check(lib().ssd3d_vote_translate(xyz.shape[0] * xyz.shape[1], _p(xyz), _p(offsets), offsets.shape[2], float(min_range[0]),
                                     float(min_range[1]), float(min_range[2]), _p(out), _stream()), "vote_translate")
    return out


def decode_dist_anchor_free(center_xyz, pred_reg, pred_cls, angle_bins=12):
    """anchor_decoder.decode_dist_anchor_free + decode_class2angle + sigmoid in one kernel: center_xyz (b, n, 3),
    pred_reg (b, n, 6 + 2*angle_bins), pred_cls (b, n, >= 1) -> boxes (b, n, 7), scores (b, n)."""
    center_xyz = _req(center_xyz, "center_xyz", torch.float32, 3, 3)
    pred_reg = _req(pred_reg, "pred_reg", torch.float32, 3)
    pred_cls = _req(pred_cls, "pred_cls", torch.float32, 3)
    b, n, _ = center_xyz.shape
    if pred_reg.shape[:2] != (b, n) or pred_cls.shape[:2] != (b, n) or pred_reg.shape[2] < 6 + 2 * angle_bins:
        raise ValueError("pred_reg must be (b, n, >= 6 + 2*angle_bins) and pred_cls (b, n, >= 1)")
    boxes = torch.empty((b, n, 7), dtype=torch.float32, device=center_xyz.device)
    scores = torch.empty((b, n), dtype=torch.float32, device=center_xyz.device)
    check(lib().ssd3d_decode_dist_anchor_free(b * n, int(angle_bins), _p(center_xyz), _p(pred_reg), pred_reg.shape[2],
                                              _p(pred_cls), pred_cls.shape[2], _p(boxes), _p(scores), _stream()),
          "decode_dist_anchor_free")
    return boxes, scores


def concat_rows(parts):
    """tf.concat(parts, axis=1) for contiguous float32 (b, m_i, c) tensors (at most 8) in one kernel."""
    parts = [_req(t, "part", torch.float32, 3) for t in parts]
    if len(parts) == 1:
        return parts[0]
    if len(parts) > 8:
        raise ValueError("concat_rows joins at most 8 parts")
    b, _, c = parts[0].shape
    if any(t.shape[0] != b or t.shape[2] != c for t in parts):
        raise ValueError("concat_rows: parts must agree in batch and channel size")
    ms = [t.shape[1] for t in parts]
    out = torch.empty((b, sum(ms), c), dtype=torch.float32, device=parts[0].device)
    src = (ctypes.c_void_p * len(parts))(*[t.data_ptr() for t in parts])
    marr = (ctypes.c_int * len(parts))(*ms)
    check(lib().ssd3d_concat_rows(b, len(parts), ctypes.cast(src, ctypes.c_void_p), ctypes.cast(marr, ctypes.c_void_p), c,
                                  _p(out), _stream()), "concat_rows")
    return out


# ---- training-mode BatchNorm (SURVEY.md 8f row f3) -----------------------------------------------------------------

BN_EPS = 1e-3   # tf.contrib.layers.batch_norm default epsilon


def bn_train(x, gamma, beta, moving_mean=None, moving_var=None, decay=0.9, relu=True, eps=BN_EPS):
    """Batch-statistics BatchNorm + activation over the last axis of x (tf_util.py:424-444, is_training=True);
    moving_mean / moving_var (float32 CUDA tensors [c]) are updated IN PLACE like updates_collections=None does.
    Returns (y, scale, shift, batch_mean, batch_var); (scale, shift) is the folded per-channel form."""
    if x.dtype != torch.float32 or not x.is_cuda:
        raise ValueError("x must be a float32 CUDA tensor")
    x = x if x.is_contiguous() else x.contiguous()
    c = x.shape[-1]
    rows = x.numel() // c
    for t, name in ((gamma, "gamma"), (beta, "beta"), (moving_mean, "moving_mean"), (moving_var, "moving_var")):
        if t is not None and (t.dtype != torch.float32 or not t.is_cuda or tuple(t.shape) != (c,) or not t.is_contiguous()):
            raise ValueError("%s must be a contiguous float32 CUDA tensor of shape (%d,)" % (name, c))
    if (moving_mean is None) != (moving_var is None):
        raise ValueError("moving_mean and moving_var go together")
    dev = x.device
    y = torch.empty_like(x)
    scale, shift, bmean, bvar = (torch.empty((c,), dtype=torch.float32, device=dev) for _ in range(4))
    ws = torch.empty((int(lib().ssd3d_bn_train_workspace(c)),), dtype=torch.uint8, device=dev)
    check(lib().ssd3d_bn_train(rows, c, _p(x), c, _p(gamma), _p(beta), _p(moving_mean), _p(moving_var), float(decay), float(eps),
                               _p(ws), _p(scale), _p(shift), _p(bmean), _p(bvar), 1 if relu else 0, _p(y), c, _stream()),
          "bn_train")
    return y, scale, shift, bmean, bvar


def rowgroup_max(y, pool, rowmask=None):
    """tf.reduce_max over runs of `pool` rows times (rowmask != 0) (layers_util.py:178-180): y (..., pool, c) -> (..., c)."""
    if y.dtype != torch.float32 or not y.is_cuda:
        raise ValueError("y must be a float32 CUDA tensor")
    y = y if y.is_contiguous() else y.contiguous()
    c, pool = y.shape[-1], int(pool)
    if y.shape[-2] != pool:
        raise ValueError("pool must equal the second-to-last dimension")
    out = torch.empty(tuple(y.shape[:-2]) + (c,), dtype=torch.float32, device=y.device)
    check(lib().ssd3d_rowgroup_max(y.numel() // (c * pool), pool, c, _p(y), c, _p(rowmask), _p(out), _stream()), "rowgroup_max")
    return out
