"""SA / FP / vote layers with the reference's signatures, on the B200 operators.

Mirrors /root/reference/lib/utils/layers_util.py: vote_layer :12-24, pointnet_sa_module :27-55,
pointnet_sa_module_msg :59-189, pointnet_fp_module :192-225 -- same positional arguments and return values,
torch CUDA tensors instead of TF tensors.  What TF resolved through variable scopes is passed explicitly as
`params` (a dict keyed by the reference's variable names, or a params.PreparedParams).  is_training=True runs the
convs with batch-statistics BatchNorm and updates the moving statistics in place (tf_util.py:424-444); the fused
inference kernels fold BN and therefore serve is_training=False only.
"""
from typing import NamedTuple

import torch

from . import config as _cfg
from . import tf_ops
from .params import prepare


def _conv(f, x, relu=True, pool=1, rowmask=None):
    return tf_ops.linear_bn_relu(x, f.w, f.scale, f.shift, relu=relu, pool=pool, rowmask=rowmask, cin=f.cin)


def _conv_train(pp, scope, x, bn, bn_decay, relu=True):
    """conv (+bias) -> training-mode BatchNorm -> ReLU, tf_util.conv2d / conv1d with is_training=True
    (/root/reference/lib/utils/tf_util.py:51-124, :127-201, :424-444).  The contraction runs on the tensor-core path with
    the BN-less fold (scale = 1, shift = bias); the batch statistics, the normalisation and the in-place update of the
    moving statistics are one ssd3d_bn_train call."""
    hi, lo = tf_ops.split_rows(x)
    y, _ = tf_ops.linear_tc(hi, lo, pp.conv(scope, False), relu=bool(relu and not bn), want_f32=True, want_split=False)
    if not bn:
        return y
    st = pp.bn_state(scope)
    return tf_ops.bn_train(y, st["gamma"], st["beta"], st["moving_mean"], st["moving_variance"],
                           decay=0.9 if bn_decay is None else float(bn_decay), relu=relu)[0]


def _ball_query(xyz, new_xyz, radius_list, nsample_list, dilated_group, want_units=False):
    """The neighbour lists of every shell (:137-145) -> (idx_list, cnt_list, units_list); units_list holds the unit lists
    of the grouped MLPs when want_units (None where query_ball_point_multi has none), else Nones."""
    nscale = len(radius_list)
    min_r = [0.0 if (i == 0 or not dilated_group) else radius_list[i - 1] for i in range(nscale)]   # :137-141
    if nscale <= 4:                                                       # one pass over the candidates for all shells
        res = tf_ops.query_ball_point_multi(min_r, radius_list, nsample_list, xyz, new_xyz, dilated_group,
                                            return_units=want_units)
        return res[0], res[1], res[2] if want_units else [None] * nscale
    res = [tf_ops.query_ball_point_dilated(min_r[i], radius_list[i], nsample_list[i], xyz, new_xyz) if dilated_group
           else tf_ops.query_ball_point(radius_list[i], nsample_list[i], xyz, new_xyz) for i in range(nscale)]
    return [r[0] for r in res], [r[1] for r in res], [None] * nscale


def _group_and_mlp_train(pp, scope, xyz, points, new_xyz, radius_list, nsample_list, mlp_list, bn, bn_decay, dilated_group,
                         use_agg):
    """Training-mode twin of _group_and_mlp: the literal op sequence of layers_util.py:137-185 (grouped tensor
    materialised once, conv -> batch-norm -> relu per layer, reduce_max, mask, concat, aggregation)."""
    idx_list, cnt_list, _ = _ball_query(xyz, new_xyz, radius_list, nsample_list, dilated_group)
    outs = []
    for i in range(len(radius_list)):
        g = tf_ops.group_concat(xyz, points, new_xyz, idx_list[i])                                  # :160-165
        for j in range(len(mlp_list[i])):
            g = _conv_train(pp, "%s/conv%d_%d" % (scope, i, j), g, bn, bn_decay)                    # :167-176
        outs.append(tf_ops.rowgroup_max(g, nsample_list[i], cnt_list[i]))                           # :178-180
    new_points = outs[0] if len(outs) == 1 else torch.cat(outs, dim=-1)
    if use_agg:
        new_points = _conv_train(pp, scope + "/ensemble", new_points, bn, bn_decay)                 # :183-185
    return new_points, idx_list, cnt_list


_CONSTS = {}


def _const(values, device):
    """Small device constants, created once (so that layer calls stay CUDA-graph capturable)."""
    key = (values, str(device))
    if key not in _CONSTS:
        _CONSTS[key] = torch.tensor(values, dtype=torch.float32, device=device)
    return _CONSTS[key]


_SIDE_STREAMS = {}


def _side_stream(device, i=0):
    key = (str(device), i)
    if key not in _SIDE_STREAMS:
        _SIDE_STREAMS[key] = torch.cuda.Stream(device=device)
    return _SIDE_STREAMS[key]


def ffps_indices(npoint, xyz, points, mode, out=None, idx_offset=0):
    """F-FPS on concat[xyz, points] (layers_util.py:94-96, :102-104).
    mode 'direct': one kernel, no [B,N,N] tensor, the SAME indices as 'matrix' (each round evaluates the picked point's
                   matrix row on chip with calc_square_dist's arithmetic); falls back to 'matrix' for uncovered shapes;
    mode 'matrix': calc_square_dist + farthest_point_sample_with_distance, the reference's route;
    mode 'fused' : matrix-free -- the generic-c FPS kernel evaluates the feature distance on the fly (no
                   [B,N,N] tensor); identical to the reference's own farthest_point_sample on the features.
    xyz / points may be [:, a:b] slices of dense tensors (read in place); out=(buffer, col) / idx_offset as in
    tf_ops.farthest_point_sample."""
    if mode == "direct":
        c = xyz.shape[2] + points.shape[2]
        # the 132-channel variant walks a 131-long dependent fma chain per round: at layer-3 sizes (512 points) the
        # small matrix is faster, so 'direct' is used where the matrix is the expensive part (c <= 68, layer 2)
        if c <= 68 and tf_ops.ffps_supported(xyz.shape[1], c):
            return tf_ops.farthest_point_sample_features(npoint, xyz, points, out=out, idx_offset=idx_offset)
        mode = "matrix"
    feats = tf_ops.concat_cols(xyz, points) if points.shape[2] else xyz
    if mode == "matrix":
        return tf_ops.farthest_point_sample_with_distance(npoint, tf_ops.calc_square_dist(feats), out=out,
                                                          idx_offset=idx_offset)
    if mode == "fused":
        return tf_ops.farthest_point_sample(npoint, feats, out=out, idx_offset=idx_offset)
    raise ValueError("ffps_mode must be 'direct', 'matrix' or 'fused'")


def _part_bounds(npoint, fps_parts):
    """Round ranges of a D-FPS consumed in parts: fps_parts = number of equal parts or a list of fractions."""
    if isinstance(fps_parts, int):
        fr = [1.0 / fps_parts] * fps_parts
    else:
        fr = [float(f) for f in fps_parts]
    cuts, acc = [0], 0.0
    for f in fr[:-1]:
        acc += f
        c = int(round(acc / sum(fr) * npoint / 128.0)) * 128          # parts are whole 128-row tiles of every scale
        cuts.append(min(max(c, cuts[-1]), npoint))
    cuts.append(npoint)
    return [(cuts[i], cuts[i + 1]) for i in range(len(cuts) - 1) if cuts[i + 1] > cuts[i]]


COMPACT_GROUPS = True      # fused SA scales convolve only the 8-row units that hold distinct neighbours (tf_ops.sa_mlp_fused `units`)
HOIST_EXPAND_MIN_K = 256   # hoisted second convs at least this wide materialise their operand (tf_ops.hoist_expand_split)


class _Scale(NamedTuple):
    """Route of one scale's grouped MLP."""
    stack: object     # FusedStack: the whole scale in one kernel (of the convs after the hoisted one); None: conv by conv
    hoisted: bool     # the first conv comes from the layer's per-point table z
    first: str        # tensor cores, conv by conv: how the first conv not in z gets its operand -- "gather" (in the kernel's
                      # operand load, linear_tc_gather), "split" (group_concat_split), "hoisted" (in the kernel, from z:
                      # linear_tc_hoisted), "expand" (from z, materialised: hoist_expand_split); otherwise None
    units: bool       # convolve only the 8-row units that hold distinct neighbours, pool them into the concat buffer
    convs: tuple      # FoldedConvs of the convs not in z


class _Plan(NamedTuple):
    """Route of the grouped MLPs of one pointnet_sa_module_msg call (see _plan)."""
    tc: bool          # tensor-core route (else fp32)
    scales: list      # a _Scale per scale
    zconv: object     # FoldedConv of the per-point table z = the feature part of every hoisted first conv (None: none)
    hoist: dict       # hoisted scale -> (its first column in z, wx = its Wx * s1 (3, n1))
    agg: object       # FoldedConv of the aggregation conv, or None
    split: bool       # the scales also write the aggregation conv's split bf16 operand (else split_rows of the concat)

    def __str__(self):
        return repr(self._replace(hoist={i: (zoff, "wx%s" % list(wx.shape)) for i, (zoff, wx) in self.hoist.items()}))


def _plan(pp, scope, mlp_list, nsample_list, bn, c_feat, use_agg, mlp_mode, fuse_scale, gather_in_kernel, hoist_first):
    scopes = [["%s/conv%d_%d" % (scope, i, j) for j in range(len(m))] for i, m in enumerate(mlp_list)]
    agg = pp.conv(scope + "/ensemble", bn) if use_agg else None
    # tensor cores: pooling widths the epilogue covers and 16-byte aligned column slices of the concat buffers
    if not (mlp_mode == "tc" and all(k in (8, 16, 32, 64, 128) for k in nsample_list) and all(m[-1] % 8 == 0 for m in mlp_list)):
        return _Plan(False, [_Scale(None, False, None, False, tuple(pp.conv(s, bn) for s in sc)) for sc in scopes],
                     None, {}, agg, False)
    stacks = [pp.fused_stack(sc, bn, c_feat + 3) if fuse_scale else None for sc in scopes]
    # hoisted first convs: the feature part of conv0 of a scale, once per POINT (independent of the sampling).
    # hoist_first: 0 off, 1 conv-by-conv scales only, 2 all.  An xyz-only cloud (c_feat == 0) has no feature part to
    # hoist: the first conv then runs in the grouped domain (linear_tc_gather / sa_mlp_fused accept c = 0).
    hoisted = [i for i, sc in enumerate(scopes) if len(sc) >= 2 and (int(hoist_first) >= 2 or stacks[i] is None)] \
        if (gather_in_kernel and hoist_first and c_feat > 0) else []
    zconv, hoist = None, {}
    if hoisted:
        zconv, wxs, n1s = pp.hoisted([scopes[i][0] for i in hoisted], bn, c_feat)
        hoist = {i: (sum(n1s[:t]), wxs[t]) for t, i in enumerate(hoisted)}
    scales = []
    for i, sc in enumerate(scopes):
        # unit lists come from the one-pass ball query; the fused kernels and the hoisted convs have *_units forms
        units = COMPACT_GROUPS and len(scopes) <= 4 and (stacks[i] is not None or i in hoist)
        convs = tuple(pp.conv(s, bn) for s in (sc[1:] if i in hoist else sc))
        if stacks[i] is not None:
            hstack = pp.fused_stack(sc[1:], bn, hoist[i][1].shape[1]) if i in hoist else None
            scales.append(_Scale(stacks[i] if hstack is None else hstack, hstack is not None, None, units, convs))
        elif i in hoist:
            # wide layer: materialise the operand once (elementwise, memory speed), then the plain TMA-fed GEMM
            expand = convs[0].kp >= HOIST_EXPAND_MIN_K and hoist[i][0] % 4 == 0 and zconv.cout % 4 == 0
            scales.append(_Scale(None, True, "expand" if expand else "hoisted", units, convs))
        else:
            scales.append(_Scale(None, False, "gather" if gather_in_kernel else "split", units, convs))
    return _Plan(True, scales, zconv, hoist, agg, agg is not None and not any(s.units for s in scales))


def _hoist_table(plan, points):
    """The per-point table z of the hoisted first convs (b, n, sum n1)."""
    p_hi, p_lo = tf_ops.split_rows(points)
    return tf_ops.linear_tc(p_hi, p_lo, plan.zconv, relu=False, want_f32=True, want_split=False)[0]


def _fused_scale(s, xyz, points, z, zx, new_xyz, idx, cnt, out_f32, out_split, units):
    """A whole scale in one kernel: gather (or the hoisted operand) + conv stack + max-pool + mask."""
    if s.hoisted:
        tf_ops.sa_mlp_fused_hoisted(xyz, z, *zx, new_xyz, idx, cnt, s.stack, out_f32=out_f32, out_split=out_split, units=units)
    else:
        tf_ops.sa_mlp_fused(xyz, points, new_xyz, idx, cnt, s.stack, out_f32=out_f32, out_split=out_split, units=units)


def _layered_scale(s, xyz, points, z, zx, new_xyz, idx, last_kw, ukw):
    """A scale conv by conv on the tensor cores: activations stay split bf16 between the convs, the last one pools into
    the concat buffers (last_kw); ukw carries the unit list of the compact rows."""
    convs = list(s.convs)
    if s.first in ("gather", "hoisted"):          # the first conv builds its operand inside the kernel (no [B,M,K,C] tensor)
        run, args = ((tf_ops.linear_tc_hoisted, (xyz, z, *zx, new_xyz, idx)) if s.first == "hoisted"
                     else (tf_ops.linear_tc_gather, (xyz, points, new_xyz, idx)))        # :160-165 in the operand load
        if len(convs) == 1:
            run(*args, convs[0], want_split=False, **last_kw)
            return
        _, (hi, lo) = run(*args, convs.pop(0), **ukw)
    elif s.first == "expand":
        hi, lo = tf_ops.hoist_expand_split(xyz, z, *zx, new_xyz, idx, **ukw)
    else:                                         # :160-165 fused with the split, materialised once in bf16 hi/lo
        hi, lo = tf_ops.group_concat_split(xyz, points, new_xyz, idx)
    for f in convs[:-1]:
        _, (hi, lo) = tf_ops.linear_tc(hi, lo, f, want_f32=False, want_split=True, **ukw)
    tf_ops.linear_tc(hi, lo, convs[-1], **last_kw)                         # :167-180 conv+BN+ReLU+max+mask


def _group_and_mlp(plan, xyz, points, z, new_xyz, radius_list, nsample_list, dilated_group):
    """Everything of pointnet_sa_module_msg after the sampling, for one block of query points new_xyz (b, m_q, 3):
    ball queries (:137-145), grouping + MLP + max-pool + mask per scale (:157-180), concat + aggregation (:182-185).
    Returns (new_points, idx_list, cnt_list)."""
    idx_list, cnt_list, units_list = _ball_query(xyz, new_xyz, radius_list, nsample_list, dilated_group,
                                                 any(s.units for s in plan.scales))
    if any(s.units and u is None for s, u in zip(plan.scales, units_list)):      # no unit list: those scales run dense
        scales = [s._replace(units=s.units and u is not None) for s, u in zip(plan.scales, units_list)]
        plan = plan._replace(scales=scales, split=plan.agg is not None and not any(s.units for s in scales))
    if not plan.tc:
        outs = []
        for s, idx, cnt in zip(plan.scales, idx_list, cnt_list):
            # rows with cnt == 0 come back zero-filled, which is what idx * (cnt > 0) produces (:157-159)
            g = tf_ops.group_concat(xyz, points, new_xyz, idx)                 # :160-165 fused
            for f in s.convs[:-1]:
                g = _conv(f, g)                                                # :167-176
            outs.append(_conv(s.convs[-1], g, pool=idx.shape[-1], rowmask=cnt))   # :167-180
        new_points = outs[0] if len(outs) == 1 else torch.cat(outs, dim=-1)
        return (new_points if plan.agg is None else _conv(plan.agg, new_points)), idx_list, cnt_list   # :183-185
    # tensor cores: every scale pools straight into its slice of the concat buffer (fp32 for the caller, split bf16 for
    # the aggregation conv).  Unit lists combine their 8-row units with atomicMax on the ZERO-FILLED fp32 buffer; the
    # split copy the aggregation conv reads is then made once, from the finished buffer.
    bs, m_q, _ = new_xyz.shape
    ctot = sum(s.convs[-1].cout for s in plan.scales)
    concat = torch.empty((bs, m_q, ctot), dtype=torch.float32, device=xyz.device)
    if any(s.units for s in plan.scales):
        tf_ops.fill_zero(concat)
    cat_hi = cat_lo = None
    if plan.split:
        ldc = tf_ops.round16(ctot)
        mk = torch.zeros if ldc != ctot else torch.empty
        cat_hi, cat_lo = (mk((bs, m_q, ldc), dtype=torch.bfloat16, device=xyz.device) for _ in range(2))
    off = 0
    for i, s in enumerate(plan.scales):
        idx, cnt, zx = idx_list[i], cnt_list[i], plan.hoist.get(i)
        units = units_list[i] if s.units else None
        out_split = (cat_hi, cat_lo, off) if plan.split else None
        if s.stack is not None:
            _fused_scale(s, xyz, points, z, zx, new_xyz, idx, cnt, (concat, off), out_split, units)
        elif units is not None:                   # compact rows; the last conv pools 8-row units into the zero-filled concat
            _layered_scale(s, xyz, points, z, zx, new_xyz, idx, dict(out_f32=(concat, off), units=units, unit_pool=True),
                           dict(units=units))
        else:
            _layered_scale(s, xyz, points, z, zx, new_xyz, idx,
                           dict(pool=idx.shape[-1], rowmask=cnt, out_f32=(concat, off), out_split=out_split), {})
        off += s.convs[-1].cout
    if plan.agg is None:
        return concat, idx_list, cnt_list
    if not plan.split:
        cat_hi, cat_lo = tf_ops.split_rows(concat)
    return tf_ops.linear_tc(cat_hi, cat_lo, plan.agg)[0], idx_list, cnt_list                    # :183-185


def _sample(xyz, points, vote_ctr, fps_sample_range_list, fps_method_list, npoint_list, in_parts, fps_parts, ffps_mode,
            fps_cluster, fps_packet, fps_bucket):
    """The sampling of pointnet_sa_module_msg (:84-111): every segment writes its indices, segment offset included,
    straight into fps_idx.  Returns (fps_idx, parts, nside, keep): fps_idx[:, col0:col1] is complete at `event` for each
    (col0, col1, event) of parts (None: on the current stream), side streams 0..nside-1 ran segments, and keep holds the
    temporaries those streams share."""
    bs, n, _ = xyz.shape
    dev = xyz.device
    main = torch.cuda.current_stream()
    segs, last = [], 0
    for rng, method, npoint in zip(fps_sample_range_list, fps_method_list, npoint_list):
        end = n if rng == -1 else last + rng                      # tf.slice size -1 (:86-87)
        if npoint == 0:                                           # :88-90
            last += rng
            continue
        if vote_ctr is not None:                                  # :91-93
            kind, width = "iota", vote_ctr.shape[1]
        elif method == "FS":                                      # :94-99 fusion sampling
            kind, width = "FS", 2 * npoint
        elif npoint == end - last:                                # :100-101
            kind, width = "iota", npoint
        elif method == "F-FPS":                                   # :102-105
            kind, width = "F", npoint
        else:                                                     # D-FPS :106-107
            kind, width = "D", npoint
        segs.append((kind, last, end, npoint, width))
        last += rng
    mtot = sum(sg[4] for sg in segs)
    fps_idx = torch.empty((bs, mtot), dtype=torch.int32, device=dev)
    parts = []                                 # (col0, col1, event): fps_idx[:, col0:col1] is complete at `event`
    keep = []                                  # temporaries shared between streams stay alive until the final join
    col, nside = 0, 0

    def on_side(fn):
        nonlocal nside
        side = _side_stream(dev, nside)
        nside += 1
        side.wait_stream(main)
        with torch.cuda.stream(side):
            fn()
            ev = torch.cuda.Event()
            ev.record(side)
        return ev

    def ev_main():
        ev = torch.cuda.Event()
        ev.record(main)
        return ev

    def ffps_segment(npoint, tmp_xyz, tmp_points, lo, col):
        """F-FPS of one segment; in latency mode the matrix-free kernel runs as two resumable launches, so the first
        half of its samples is handed to the consumers while the second half is still being picked."""
        c = tmp_xyz.shape[2] + tmp_points.shape[2]
        if in_parts and ffps_mode == "direct" and c <= 68 and npoint >= 256 and tf_ops.ffps_supported(tmp_xyz.shape[1], c):
            temp = torch.empty((bs, tmp_xyz.shape[1]), dtype=torch.float32, device=dev)
            keep.append(temp)
            for j0, j1 in _part_bounds(npoint, 2):
                tf_ops.farthest_point_sample_features(npoint, tmp_xyz, tmp_points, out=(fps_idx, col), idx_offset=lo,
                                                      rounds=(j0, j1), temp=temp)
                parts.append((col + j0, col + j1, ev_main()))
            return
        ffps_indices(npoint, tmp_xyz, tmp_points, ffps_mode, out=(fps_idx, col), idx_offset=lo)
        parts.append((col, col + npoint, ev_main() if in_parts else None))

    lone = len(segs) == 1
    for kind, lo, hi, npoint, width in segs:
        tmp_xyz, tmp_points = xyz[:, lo:hi], points[:, lo:hi]     # read in place (scene-strided)
        if kind == "iota":
            tf_ops.iota_idx(bs, width, dev, out=(fps_idx, col), start=lo)
            parts.append((col, col + width, ev_main() if in_parts else None))
        elif kind == "FS":
            # F-FPS and D-FPS are independent latency-bound chains on a handful of SMs each: run them concurrently
            c0 = col
            ev_d = on_side(lambda: tf_ops.farthest_point_sample(npoint, tmp_xyz, out=(fps_idx, c0 + npoint), idx_offset=lo,
                                                                cluster=fps_cluster))
            ffps_segment(npoint, tmp_xyz, tmp_points, lo, col)
            parts.append((col + npoint, col + 2 * npoint, ev_d))
        elif kind == "F":
            ffps_segment(npoint, tmp_xyz, tmp_points, lo, col)
        elif not lone:                                            # D-FPS segment next to other segments: side stream
            c0 = col
            ev_d = on_side(lambda: tf_ops.farthest_point_sample(npoint, tmp_xyz, out=(fps_idx, c0), idx_offset=lo,
                                                                cluster=fps_cluster))
            parts.append((col, col + npoint, ev_d))
        elif in_parts and not isinstance(fps_parts, bool) and tf_ops.fps_supports_rounds(hi - lo, 3):
            temp = torch.empty((bs, tf_ops.fps_temp_elems(hi - lo, 3, npoint, bucket_kernel=fps_bucket)), dtype=torch.float32, device=dev)
            keep.append(temp)
            for j0, j1 in _part_bounds(npoint, fps_parts):
                tf_ops.farthest_point_sample(npoint, tmp_xyz, out=(fps_idx, col), idx_offset=lo, rounds=(j0, j1), temp=temp,
                                             cluster=fps_cluster, bucket_kernel=fps_bucket)
                parts.append((col + j0, col + j1, ev_main()))
        else:
            tf_ops.farthest_point_sample(npoint, tmp_xyz, out=(fps_idx, col), idx_offset=lo, cluster=fps_cluster,
                                         packet_kernel=fps_packet, bucket_kernel=fps_bucket)
            parts.append((col, col + npoint, ev_main() if in_parts else None))
        col += width
    return fps_idx, parts, nside, keep


def pointnet_sa_module_msg(xyz, points, radius_list, nsample_list, mlp_list, is_training, bn_decay, bn,
                           fps_sample_range_list, fps_method_list, npoint_list, former_fps_idx, use_attention, scope,
                           dilated_group, vote_ctr=None, aggregation_channel=None, debugging=False, epsilon=1e-5, *,
                           params, ffps_mode="direct", aggregation=None, return_debug=False, mlp_mode="tc",
                           fuse_scale=True, gather_in_kernel=True, hoist_first=2, fps_cluster=0, fps_parts=None,
                           fps_packet=False, fps_bucket=None):
    """PointNet++ SA module with multi-scale grouping; returns (new_xyz, new_points, fps_idx).

    Keyword extensions (none changes a result):
      fps_cluster  CTAs per scene of the D-FPS kernels (tf_ops.farthest_point_sample `cluster`);
      fps_bucket   lone D-FPS kernel choice (tf_ops.farthest_point_sample `bucket_kernel`: None automatic, False = cluster kernel);
      fps_packet   D-FPS with the coordinates-in-packet kernel (64 KiB of shared memory per CTA instead of the whole
                   scene: other kernels can share its SMs);
      fps_parts    latency mode.  FPS emits its samples in order, and a sample is final once its round is done, so the
                   layer consumes the sampling IN PARTS: a lone D-FPS runs as resumable launches of rounds (an int =
                   that many equal parts, or a list of fractions), a fusion-sampling layer hands over its F-FPS and
                   D-FPS halves separately; ball query + grouped MLP + aggregation of a part run on a side stream
                   while the sampling of the next part continues, and the per-part results are joined at the end.
                   Captured in a CUDA graph this is a plain dependency graph -- nothing polls."""
    if use_attention:
        raise NotImplementedError("query_ball_point_withidx (use_attention) is unused by the shipped 3DSSD configs")
    if is_training:
        fps_parts = None                      # training takes the literal layer-by-layer schedule
    if mlp_mode not in ("tc", "fp32"):
        raise ValueError("mlp_mode must be 'tc' or 'fp32'")
    pp = prepare(params, xyz.device)
    aggregation = _cfg.AGGREGATION_SA_FEATURE if aggregation is None else aggregation
    use_agg = bool(aggregation and aggregation_channel is not None and aggregation_channel != -1)
    dev = xyz.device
    nscale = len(radius_list)
    main = torch.cuda.current_stream()
    in_parts = bool(fps_parts) and nscale > 0 and former_fps_idx is None
    plan = _plan(pp, scope, mlp_list, nsample_list, bn, points.shape[-1], use_agg, mlp_mode, fuse_scale, gather_in_kernel,
                 hoist_first) if (nscale and not is_training) else None
    z = None
    if in_parts and plan.hoist:                # the hoisted first convs overlap the first rounds of the sampling
        zs = _side_stream(dev, 7)
        zs.wait_stream(main)
        with torch.cuda.stream(zs):
            z = _hoist_table(plan, points)
        z_ready = torch.cuda.Event()
        z_ready.record(zs)
    fps_idx, parts, nside, keep = _sample(xyz, points, vote_ctr, fps_sample_range_list, fps_method_list, npoint_list, in_parts,
                                          fps_parts, ffps_mode, fps_cluster, fps_packet, fps_bucket)
    src_xyz = vote_ctr if vote_ctr is not None else xyz

    if not in_parts:
        for _, _, ev in parts:
            if ev is not None:
                main.wait_event(ev)
        if former_fps_idx is not None:
            fps_idx = torch.cat([fps_idx, former_fps_idx], dim=-1).contiguous()    # :113-114
        new_xyz = tf_ops.gather_point(src_xyz, fps_idx)                            # :116-119
        debug = {"idx": [], "cnt": []}
        if nscale and is_training:
            new_points, debug["idx"], debug["cnt"] = _group_and_mlp_train(
                pp, scope, xyz, points, new_xyz, radius_list, nsample_list, mlp_list, bn, bn_decay, dilated_group, use_agg)
        elif nscale:
            z = _hoist_table(plan, points) if plan.hoist else None
            new_points, debug["idx"], debug["cnt"] = _group_and_mlp(plan, xyz, points, z, new_xyz, radius_list, nsample_list,
                                                                    dilated_group)
        else:
            new_points = tf_ops.gather_point(points.contiguous(), fps_idx)         # :186-187
    else:
        # ---- one consumer chain per part, each on its own stream, joined at the end
        xyz_parts, pts_parts, nbrs, done = [], [], [], []
        for pi, (c0, c1, ev) in enumerate(parts):
            st = _side_stream(dev, 8 + pi)
            st.wait_event(ev)
            if z is not None:
                st.wait_event(z_ready)
            with torch.cuda.stream(st):
                nx = tf_ops.gather_point(src_xyz, fps_idx[:, c0:c1])
                npnts, idx_list, cnt_list = _group_and_mlp(plan, xyz, points, z, nx, radius_list, nsample_list, dilated_group)
                e2 = torch.cuda.Event()
                e2.record(st)
            xyz_parts.append(nx); pts_parts.append(npnts); nbrs.append((idx_list, cnt_list)); done.append(e2)
        for e2 in done:
            main.wait_event(e2)
        for i in range(nside):
            main.wait_stream(_side_stream(dev, i))
        new_xyz = tf_ops.concat_rows(xyz_parts)
        new_points = tf_ops.concat_rows(pts_parts)
        keep.extend(xyz_parts + pts_parts)
        debug = None
        if return_debug:
            debug = {"idx": [torch.cat([p[0][i] for p in nbrs], dim=1) for i in range(nscale)],
                     "cnt": [torch.cat([p[1][i] for p in nbrs], dim=1) for i in range(nscale)]}
        _KEEPALIVE.append((keep, None if return_debug else nbrs, z))
        del _KEEPALIVE[:-8]
    if return_debug:
        return new_xyz, new_points, fps_idx, debug
    return new_xyz, new_points, fps_idx


_KEEPALIVE = []   # latency mode: the last layers' cross-stream temporaries (freed a few calls later, long after their use)


def pointnet_sa_module(xyz, points, mlp, is_training, bn_decay, bn, scope, *, params):
    """Global SA layer (layer type SA_Layer_SSG_Last): concat[xyz, points] -> MLP -> max over all points."""
    pp = prepare(params, xyz.device)
    g = torch.cat([xyz, points], dim=-1).contiguous()              # xyz FIRST here (:42)
    n = g.shape[1]
    for j in range(len(mlp)):
        g = _conv_train(pp, "%s/conv%d" % (scope, j), g, bn, bn_decay) if is_training else _conv(pp.conv("%s/conv%d" % (scope, j), bn), g)
    return g.max(dim=1).values if n else g


def pointnet_fp_module(xyz1, xyz2, points1, points2, mlp, is_training, bn_decay, scope, bn=True, *, params):
    """Feature propagation: inverse-distance interpolation from (xyz2, points2) onto xyz1, then an MLP."""
    pp = prepare(params, xyz1.device)
    dist, idx = tf_ops.three_nn(xyz1, xyz2)
    dist = torch.clamp_min(dist, 1e-10)                            # :207
    inv = 1.0 / dist
    weight = inv / inv.sum(dim=2, keepdim=True)                    # :208-210
    x = tf_ops.three_interpolate(points2, idx, weight.contiguous())
    if points1 is not None:
        x = torch.cat([x, points1], dim=2).contiguous()            # :213-214
    for i in range(len(mlp)):
        x = _conv_train(pp, "%s/conv_%d" % (scope, i), x, bn, bn_decay) if is_training else _conv(pp.conv("%s/conv_%d" % (scope, i), bn), x)
    return x


def vote_layer(xyz, points, mlp_list, is_training, bn_decay, bn, scope, *, params,
               max_translate_range=_cfg.MAX_TRANSLATE_RANGE, mlp_mode="tc"):
    """Vote layer: per-point MLP -> 3 offsets, clamped to +-max_translate_range (layers_util.py:12-24)."""
    pp = prepare(params, xyz.device)
    if is_training:
        for i in range(len(mlp_list)):
            points = _conv_train(pp, "%s/vote_layer_%d" % (scope, i), points, bn, bn_decay)
        off = _conv_train(pp, scope + "/vote_offsets", points, False, bn_decay, relu=False)
    elif mlp_mode == "tc":
        hi, lo = tf_ops.split_rows(points)
        for i in range(len(mlp_list)):
            points, (hi, lo) = tf_ops.linear_tc(hi, lo, pp.conv("%s/vote_layer_%d" % (scope, i), bn), want_split=True)
        off, _ = tf_ops.linear_tc(hi, lo, pp.conv(scope + "/vote_offsets", False), relu=False)
    else:
        for i in range(len(mlp_list)):
            points = _conv(pp.conv("%s/vote_layer_%d" % (scope, i), bn), points)
        off = _conv(pp.conv(scope + "/vote_offsets", False), points, relu=False)
    return tf_ops.vote_translate(xyz, off, max_translate_range), points, off                       # :20-23
