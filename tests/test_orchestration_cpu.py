"""CPU dry run of the layer orchestration (3dssd_b200/layers_util.py, backbone.py): every tf_ops entry point the fp32
route touches is replaced by a few lines on top of the CPU oracle, and torch.cuda's streams / events by inert stand-ins,
so that the PYTHON around the kernels -- segment placement into the shared fps_idx buffer, offsets, scene-strided slices,
resumable rounds, the latency-mode part schedule and its joins -- runs here without a GPU and must reproduce the
oracle's own layer code.  (The kernels themselves are covered by the -m gpu tests.)"""
import copy
import importlib
import inspect
import json
import os

import numpy as np
import pytest
import torch


class _Inert:
    def __init__(self, *a, **k):
        pass

    def wait_stream(self, *a):
        pass

    def wait_event(self, *a):
        pass

    def record(self, *a):
        pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        return False


@pytest.fixture()
def dry(monkeypatch, oracle_ops):
    pkg = importlib.import_module("3dssd_b200")
    T, L = pkg.tf_ops, pkg.layers_util
    o = oracle_ops
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a))
    n = lambda x: x.detach().cpu().numpy()

    def place(res, out, idx_offset, b, npoint, rounds=None):
        res = res.astype(np.int32) + int(idx_offset)
        if out is None:
            return t(res)
        buf, col = out
        j0, j1 = (0, npoint) if rounds is None else rounds
        buf[:, col + j0: col + j1] = t(res[:, j0:j1])
        return buf[:, col: col + npoint]

    def fps(npoint, inp, *, out=None, idx_offset=0, rounds=None, temp=None, cluster=0, packet_kernel=False, bucket_kernel=None):
        if rounds is not None and tuple(rounds) != (0, npoint):
            assert temp is not None and temp.shape == (inp.shape[0], 2 * inp.shape[1])      # fps_temp_elems of the fake
        return place(o.farthest_point_sample(npoint, n(inp)), out, idx_offset, inp.shape[0], npoint, rounds)

    def ffps(npoint, xyz, points=None, *, out=None, idx_offset=0, rounds=None, temp=None):
        f = n(xyz) if points is None else np.concatenate([n(xyz), n(points)], -1)
        return place(o.farthest_point_sample_with_distance(npoint, o.calc_square_dist(f)), out, idx_offset, xyz.shape[0], npoint, rounds)

    def fpsd(npoint, dist, *, out=None, idx_offset=0, cluster=0):
        return place(o.farthest_point_sample_with_distance(npoint, n(dist)), out, idx_offset, dist.shape[0], npoint)

    def iota(b, npoint, device, *, out=None, start=0):
        return place(np.tile(np.arange(npoint, dtype=np.int32)[None], (b, 1)), out, start, b, npoint)

    def bq_multi(lows, highs, ks, xyz1, xyz2, dilated, grid=None, return_units=False):
        res = [(o.query_ball_point_dilated(lo, hi, k, n(xyz1), n(xyz2)) if dilated else o.query_ball_point(hi, k, n(xyz1), n(xyz2)))
               for lo, hi, k in zip(lows, highs, ks)]
        out = [t(r[0]) for r in res], [t(r[1]) for r in res]
        if not return_units:
            return out
        units = []                                                   # the unit lists of include/ssd3d.h, in REVERSED group order
        for r, k in zip(res, ks):                                    # (the order is unspecified: consumers may not rely on it)
            cnt = r[1].reshape(-1)
            lst = [(g << 4) | j for g in range(cnt.size - 1, -1, -1) for j in range((min(int(cnt[g]), k) + 7) // 8)]
            u = np.full(1 + cnt.size * ((k + 7) // 8), -1, np.int32)
            u[0] = len(lst); u[1:1 + len(lst)] = lst
            units.append(t(u))
        return out + (units,)

    def group_concat(xyz, points, new_xyz, idx, ldx=None):
        g = np.concatenate([o.group_point(n(points), n(idx)), o.group_point(n(xyz), n(idx)) - n(new_xyz)[:, :, None]], -1)
        return t(g.astype(np.float32))

    def linear_bn_relu(x, w, scale, shift, relu=True, pool=1, rowmask=None, cin=None):
        y = (n(x).astype(np.float64)[..., : w.shape[0]] @ n(w).astype(np.float64)) * n(scale) + n(shift)
        if relu:
            y = np.maximum(y, 0)
        if pool > 1:
            y = y.max(axis=-2) * (n(rowmask) > 0)[..., None]
        return t(y.astype(np.float32))

    # ---- tensor-core route: split bf16 operands are real (hi + lo), the contraction is float64 on the folded layers
    def split_rows(x, kp=None):
        c = x.shape[-1]
        kp = T.round16(c) if kp is None else int(kp)
        hi = torch.zeros(tuple(x.shape[:-1]) + (kp,), dtype=torch.bfloat16)
        lo = torch.zeros_like(hi)
        hi[..., :c] = x.to(torch.bfloat16)
        lo[..., :c] = (x - hi[..., :c].float()).to(torch.bfloat16)
        return hi, lo

    unsplit = lambda hi, lo: hi.float() + lo.float()

    def emit(y, pool, rowmask, want_f32, want_split, out_f32, out_split):
        if pool > 1:
            y = y.max(dim=-2).values * (rowmask > 0).unsqueeze(-1).to(y.dtype) if rowmask is not None else y.max(dim=-2).values
        nn = y.shape[-1]
        ret = None
        if out_f32 is not None:
            buf, off = out_f32
            buf[..., off: off + nn] = y
            ret = buf
        elif want_f32:
            ret = y
        sp = None
        if out_split is not None:
            hb, lb, off = out_split
            h, l = split_rows(y, nn)
            hb[..., off: off + nn] = h; lb[..., off: off + nn] = l
            sp = (hb, lb)
        elif want_split:
            sp = split_rows(y)
        return ret, sp

    def compact(x, units):
        """Dense grouped rows (b, m, ns, C) -> the compact layout of the *_units kernels: 8 rows per listed unit at the start
        of the buffer, NaN beyond (so that anything consuming rows it should not shows up)."""
        b, m, ns, c = x.shape
        u = n(units); nu = int(u[0])
        flat = x.reshape(b * m, ns, c)
        out = torch.full((b * m * ns, c), float("nan"), dtype=x.dtype)
        for i in range(nu):
            g, j = int(u[1 + i]) >> 4, int(u[1 + i]) & 15
            out[8 * i: 8 * i + 8] = flat[g, 8 * j: 8 * j + 8]
        return out.reshape(b, m, ns, c)

    def unit_pool_into(y, units, out_f32):
        """atomicMax of every unit's column maxima into its group's row of the caller's buffer (no fill of other groups)."""
        buf, off = out_f32
        u = n(units); nu = int(u[0])
        rows = y.reshape(-1, y.shape[-1])
        flat = buf.view(-1, buf.shape[-1])
        assert not torch.isnan(flat[:, off: off + rows.shape[1]]).any()
        for i in range(nu):
            g = int(u[1 + i]) >> 4
            mx = rows[8 * i: 8 * i + 8].max(dim=0).values
            assert not torch.isnan(mx).any() and (mx >= 0).all()
            flat[g, off: off + rows.shape[1]] = torch.maximum(flat[g, off: off + rows.shape[1]], mx)
        return buf, None

    def conv(x, f, relu=True):
        y = (x[..., : f.cin].double() @ f.w.double()) * f.scale.double() + f.shift.double()
        return (torch.relu(y) if relu else y).float()

    def linear_tc(a_hi, a_lo, f, relu=True, pool=1, rowmask=None, want_f32=True, want_split=False, out_f32=None, out_split=None,
                  units=None, unit_pool=False):
        assert a_hi.shape[-1] == f.kp and a_hi.dtype == torch.bfloat16
        y = conv(unsplit(a_hi, a_lo), f, relu)
        if unit_pool:
            assert units is not None and relu and pool == 1 and rowmask is None and out_split is None and not want_split
            return unit_pool_into(y, units, out_f32)
        return emit(y, pool, rowmask, want_f32, want_split, out_f32, out_split)

    def grouped(xyz, points, new_xyz, idx):
        return group_concat(xyz, points, new_xyz, idx)

    def hoisted_operand(xyz, z, zoff, wx, new_xyz, idx):
        n1 = wx.shape[1]
        d = t(o.group_point(n(xyz), n(idx)) - n(new_xyz)[:, :, None])
        zg = t(o.group_point(n(z[..., zoff: zoff + n1].contiguous()), n(idx)))
        return torch.relu(zg + d @ wx)

    def linear_tc_gather(xyz, points, new_xyz, idx, f, relu=True, pool=1, rowmask=None, want_f32=False, want_split=True, out_f32=None, out_split=None):
        return emit(conv(grouped(xyz, points, new_xyz, idx), f, relu), pool, rowmask, want_f32, want_split, out_f32, out_split)

    def linear_tc_hoisted(xyz, z, zoff, wx, new_xyz, idx, f, relu=True, pool=1, rowmask=None, want_f32=False, want_split=True, out_f32=None, out_split=None,
                          units=None, unit_pool=False):
        assert f.cin == wx.shape[1]
        x = hoisted_operand(xyz, z, zoff, wx, new_xyz, idx)
        if units is not None:
            y = conv(compact(x, units), f, relu)
            if unit_pool:
                return unit_pool_into(y, units, out_f32)
            return emit(y, 1, None, want_f32, want_split, out_f32, out_split)
        return emit(conv(x, f, relu), pool, rowmask, want_f32, want_split, out_f32, out_split)

    def fused(x, cnt, stack, out_f32, out_split, ns, units=None):
        if units is not None:
            assert out_split is None
            x = compact(x, units)
        for f in stack.convs:
            x = conv(x, f)
        if units is not None:
            return unit_pool_into(x, units, out_f32)[0]
        y, _ = emit(x, ns, cnt if cnt is not None else None, out_f32 is None and out_split is None, False, out_f32, out_split)
        return y

    def sa_mlp_fused(xyz, points, new_xyz, idx, cnt, stack, out_f32=None, out_split=None, units=None):
        assert points.shape[-1] + 3 == stack.cin
        return fused(grouped(xyz, points, new_xyz, idx), cnt, stack, out_f32, out_split, idx.shape[-1], units)

    def sa_mlp_fused_hoisted(xyz, z, zoff, wx, new_xyz, idx, cnt, stack, out_f32=None, out_split=None, units=None):
        assert wx.shape[1] == stack.cin
        return fused(hoisted_operand(xyz, z, zoff, wx, new_xyz, idx), cnt, stack, out_f32, out_split, idx.shape[-1], units)

    fakes = dict(
        fill_zero=lambda x: x.zero_(),
        split_rows=split_rows, linear_tc=linear_tc, linear_tc_gather=linear_tc_gather, linear_tc_hoisted=linear_tc_hoisted,
        sa_mlp_fused=sa_mlp_fused, sa_mlp_fused_hoisted=sa_mlp_fused_hoisted,
        hoist_expand_split=lambda xyz, z, zoff, wx, new_xyz, idx, units=None: split_rows(
            hoisted_operand(xyz, z, zoff, wx, new_xyz, idx) if units is None else compact(hoisted_operand(xyz, z, zoff, wx, new_xyz, idx), units)),
        group_concat_split=lambda xyz, points, new_xyz, idx, kp=None: split_rows(grouped(xyz, points, new_xyz, idx), kp),
        split_points=lambda p: (p[..., :3].contiguous(), p[..., 3:].contiguous()),
        farthest_point_sample=fps, farthest_point_sample_features=ffps, farthest_point_sample_with_distance=fpsd,
        calc_square_dist=lambda a: t(o.calc_square_dist(n(a))), concat_cols=lambda a, b: torch.cat([a, b], -1).contiguous(),
        iota_idx=iota, gather_point=lambda inp, idx: t(o.gather_point(n(inp), n(idx))),
        query_ball_point_multi=bq_multi, group_concat=group_concat, linear_bn_relu=linear_bn_relu,
        concat_rows=lambda parts: torch.cat(list(parts), dim=1).contiguous(),
        fps_supports_rounds=lambda nn, c=3: True, ffps_supported=lambda nn, c: c <= 68,
        fps_temp_elems=lambda nn, c=3, npoint=0, **kw: 2 * nn,
        vote_translate=lambda xyz, off, rng: xyz + torch.minimum(torch.maximum(off[..., :3], torch.tensor(rng)), -torch.tensor(rng)),
    )
    for k, v in fakes.items():
        monkeypatch.setattr(T, k, v)
    monkeypatch.setattr(torch.cuda, "current_stream", lambda *a, **k: _Inert())
    monkeypatch.setattr(torch.cuda, "Stream", _Inert)
    monkeypatch.setattr(torch.cuda, "Event", _Inert)
    monkeypatch.setattr(torch.cuda, "stream", lambda s: _Inert())
    monkeypatch.setattr(L, "_SIDE_STREAMS", {})
    return pkg


def _scaled(pkg, div):
    arch = copy.deepcopy(pkg.config.ARCH_3DSSD)
    for spec in arch:
        spec[6] = [r if r == -1 else max(1, r // div) for r in spec[6]]
        spec[8] = [p if p in (-1, 0) else max(1, p // div) for p in spec[8]]
    return arch


ROUTE_TRACE = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "sa_route_trace.json")


def _record_calls(monkeypatch, pkg):
    """Wrap every tf_ops entry point: each call the layers make is appended to the returned list as [name, positional
    args, keyword args], tensors reduced to dtype and shape, folded convs to (cin, cout), fused stacks to their widths.
    The sequence is the host-side launch schedule of the forward: same calls, same order, same operand shapes."""
    T, P = pkg.tf_ops, pkg.params
    calls = []

    def enc(v):
        if isinstance(v, torch.Tensor):
            return "%s%s" % (str(v.dtype).replace("torch.", ""), list(v.shape))
        if isinstance(v, P.FoldedConv):
            return ["FoldedConv", v.cin, v.cout]
        if isinstance(v, P.FusedStack):
            return ["FusedStack", list(v.nout)]
        if isinstance(v, (list, tuple)):
            return [enc(x) for x in v]
        if isinstance(v, torch.device):
            return str(v.type)
        if v is None or isinstance(v, (bool, int, float, str)):
            return v
        raise TypeError("no trace encoding for %r" % (v,))

    for name, fn in list(vars(T).items()):
        if name.startswith("_") or name in ("check", "lib", "round16") or not inspect.isfunction(fn):
            continue

        def rec(*a, _fn=fn, _name=name, **kw):
            calls.append([_name, enc(a), {k: enc(kw[k]) for k in sorted(kw)}])
            return _fn(*a, **kw)
        monkeypatch.setattr(T, name, rec)
    return calls


def _check_route_trace(key, calls):
    """Compare with the stored trace; SSD3D_WRITE_ROUTE_TRACE=1 stores this run's trace instead (a deliberate change of
    the launch schedule)."""
    store = {}
    if os.path.exists(ROUTE_TRACE):
        with open(ROUTE_TRACE) as fh:
            store = json.load(fh)
    got = json.loads(json.dumps(calls))
    if os.environ.get("SSD3D_WRITE_ROUTE_TRACE"):
        store[key] = got
        with open(ROUTE_TRACE, "w") as fh:
            fh.write("{\n" + ",\n".join("%s: [\n%s\n]" % (json.dumps(k), ",\n".join(json.dumps(c) for c in store[k]))
                                        for k in sorted(store)) + "\n}\n")
        return
    assert key in store, "no stored route trace for %s (SSD3D_WRITE_ROUTE_TRACE=1 records it)" % key
    exp = store[key]
    for i, (g, e) in enumerate(zip(got, exp)):
        assert g == e, "call %d of the route differs:\n  got      %s\n  expected %s" % (i, g, e)
    assert len(got) == len(exp), "the route makes %d tf_ops calls, expected %d" % (len(got), len(exp))


@pytest.mark.parametrize("mlp_mode,gather,hoist,fuse", [("fp32", True, 2, True), ("tc", True, 2, True), ("tc", True, 1, True),
                                                        ("tc", True, 0, True), ("tc", False, 0, False), ("tc", True, 2, False)])
@pytest.mark.parametrize("latency,parts", [(False, None), (True, 2), (True, [0.5, 0.25, 0.25])])
def test_backbone_orchestration_dry_run_matches_oracle_layers(dry, oracle_ops, monkeypatch, request, latency, parts, mlp_mode,
                                                              gather, hoist, fuse):
    """The layer outputs equal the oracle's, and the sequence of tf_ops calls equals tests/golden/sa_route_trace.json
    (the tc / fused / default-latency case also with layers_util.COMPACT_GROUPS off)."""
    pkg = dry
    from oracle import layers as olayers
    synth = importlib.import_module("3dssd_b200.synth")
    arch = _scaled(pkg, 16)                                       # 1024 -> 256 -> 64+.. centres
    params = pkg.params.init_params(arch, 1, seed=4, random_bias=True)
    pts = synth.kitti_like(2, 1024, seed=40)
    pts[..., 0] *= 0.2; pts[..., 2] *= 0.2
    kw = dict(fps_parts=parts) if parts is not None else {}
    net = pkg.SABackbone(arch, params, in_channels=1, device="cpu", mlp_mode=mlp_mode, latency_mode=latency,
                         gather_in_kernel=gather, hoist_first=hoist, fuse_scale=fuse, **kw)
    exp = olayers.backbone_forward(arch, pts, params, ffps_mode="matrix", return_debug=True)
    calls = _record_calls(monkeypatch, pkg)
    runs = [request.node.callspec.id]
    if (mlp_mode, gather, hoist, fuse, latency) == ("tc", True, 2, True, False):
        runs.append(runs[0] + "-nocompact")
    for key in runs:
        monkeypatch.setattr(pkg.layers_util, "COMPACT_GROUPS", not key.endswith("-nocompact"))
        del calls[:]
        got = net.forward(torch.from_numpy(pts), return_debug=True)
        for li in range(1, len(arch) + 1):
            if exp[2][li] is not None:
                np.testing.assert_array_equal(got[2][li].numpy(), exp[2][li], err_msg="fps_idx of layer %d" % li)
            for a, b in zip(got[3][li - 1].get("idx", []), exp[3][li - 1].get("idx", [])):
                np.testing.assert_array_equal(a.numpy(), b)
            if exp[0][li] is not None:
                assert np.abs(got[0][li].numpy() - exp[0][li]).max() < 1e-5
            assert np.abs(got[1][li].numpy() - exp[1][li]).max() <= 1e-4 * max(1.0, np.abs(exp[1][li]).max()), "features of layer %d" % li
        _check_route_trace(key, calls)


def test_head_orchestration_dry_run_writes_into_gather_buffers(dry, oracle_ops, monkeypatch):
    """DetectionHead + DetectionGather plumbing on the CPU: conv chain -> one-kernel decode -> NMS writing straight into
    the send buffer of the (single-rank) gather, against the oracle's head."""
    pkg = dry
    from oracle import head as ohead
    T = pkg.tf_ops

    def decode(center_xyz, pred_reg, pred_cls, angle_bins=12):
        reg, cls = pred_reg.numpy(), pred_cls.numpy()
        off, acls, ares = reg[..., :6], reg[..., 6:6 + angle_bins], reg[..., 6 + angle_bins:]
        bins = np.argmax(acls, -1)
        res = np.take_along_axis(ares, bins[..., None], -1)[..., 0]
        ang = ((bins.astype(np.float32) + res) * np.float32(2 * np.pi / angle_bins)).astype(np.float32)
        ctr = center_xyz.numpy() + off[..., :3]
        ctr[..., 1] += off[..., 4]
        boxes = np.concatenate([ctr, np.maximum(off[..., 3:6] * np.float32(2), np.float32(0.1)), ang[..., None]], -1).astype(np.float32)
        return torch.from_numpy(boxes), torch.from_numpy((1 / (1 + np.exp(-cls[..., 0].astype(np.float64)))).astype(np.float32))

    def nms(boxes, scores, thr, max_output, cls_id=0, out=None):
        blk, cnt = oracle_ops.bev_nms(boxes.numpy(), scores.numpy(), thr, max_output, cls_id)
        if out is None:
            return torch.from_numpy(blk), torch.from_numpy(cnt)
        out[0].copy_(torch.from_numpy(blk)); out[1].copy_(torch.from_numpy(cnt))
        return out

    monkeypatch.setattr(T, "decode_dist_anchor_free", decode)
    monkeypatch.setattr(T, "bev_nms", nms)
    rng = np.random.default_rng(3)
    xyz = rng.uniform(-10, 10, (3, 64, 3)).astype(np.float32)
    feat = np.maximum(rng.standard_normal((3, 64, 512)), 0).astype(np.float32)
    prm = pkg.params.init_head_params(512, seed=5)
    head = pkg.DetectionHead(params=prm, device="cpu")
    g = pkg.dist.DetectionGather(3, "cpu")
    blk, cnt = head.forward([None] * 6 + [torch.from_numpy(xyz)], [None] * 6 + [torch.from_numpy(feat)], out=g.out())
    g.gather()
    rb, rc = g.result()
    eboxes, escore, _ = ohead.head_forward(xyz, feat, prm)
    eb, ec = ohead.bev_nms(eboxes, escore, 0.1, 100)
    assert rb.data_ptr() == blk.data_ptr() and torch.equal(rc, cnt)
    np.testing.assert_array_equal(rc.numpy(), ec)
    assert np.abs(rb.numpy() - eb).max() < 2e-3


@pytest.mark.parametrize("decay", [None, 0.5])
def test_training_mode_orchestration_dry_run_matches_oracle(dry, oracle_ops, monkeypatch, decay):
    """is_training=True through pointnet_sa_module_msg on the CPU (SURVEY 8f row f3): the literal conv -> batch-norm -> relu
    schedule with ssd3d_bn_train / ssd3d_rowgroup_max replaced by a few float64 lines, against the oracle's restatement of
    tf_util.py:424-444; the moving statistics are updated in place, commit_bn() writes them back and inference then folds
    the NEW statistics."""
    pkg = dry
    from oracle import layers as olayers
    T = pkg.tf_ops

    def bn_train(x, gamma, beta, moving_mean=None, moving_var=None, decay=0.9, relu=True, eps=1e-3):
        flat = x.reshape(-1, x.shape[-1]).double()
        mean = flat.mean(0)
        var = ((flat - mean) ** 2).mean(0)
        inv = gamma.double() / torch.sqrt(var + eps)
        y = x.double() * inv + (beta.double() - mean * inv)
        if moving_mean is not None:                                  # in place, like updates_collections=None
            moving_mean.sub_(((moving_mean.double() - mean) * (1.0 - decay)).float())
            moving_var.sub_(((moving_var.double() - var) * (1.0 - decay)).float())
        return (torch.relu(y) if relu else y).float(), inv.float(), (beta.double() - mean * inv).float(), mean.float(), var.float()

    def rowgroup_max(y, pool, rowmask=None):
        out = y.max(dim=-2).values
        return out * (rowmask > 0).unsqueeze(-1).to(out.dtype) if rowmask is not None else out

    monkeypatch.setattr(T, "bn_train", bn_train)
    monkeypatch.setattr(T, "rowgroup_max", rowgroup_max)
    rng = np.random.default_rng(11)
    synth = importlib.import_module("3dssd_b200.synth")
    pts = synth.kitti_like(2, 512, seed=61)
    pts[..., 0] *= 0.1; pts[..., 2] *= 0.1
    xyz, feats = pts[..., :3].copy(), rng.standard_normal((2, 512, 16)).astype(np.float32)
    arch = [[[0], [0], [0.4, 0.8], [16, 32], [[16, 16, 32], [16, 32, 48]], True, [-1], ['D-FPS'], [64],
             -1, False, 'SA_Layer', 'trn', True, -1, 64]]
    params = dict(pkg.params.init_params(arch, 16, seed=8, random_bias=True))
    args = (arch[0][2], arch[0][3], arch[0][4], True, decay, True, [-1], ['D-FPS'], [64], None, False, 'trn', True)
    params_ref = {k: np.array(v, copy=True) for k, v in params.items()}            # on the CPU torch.from_numpy ALIASES the dict's
    pp = pkg.params.prepare(params, "cpu")                                        # arrays: the oracle gets its own copy
    got = pkg.pointnet_sa_module_msg(torch.from_numpy(xyz), torch.from_numpy(feats), *args, aggregation_channel=64, params=pp,
                                     return_debug=True, fps_parts=2)              # fps_parts is ignored when training
    upd = {}
    exp = olayers.pointnet_sa_module_msg(xyz, feats, *args, aggregation_channel=64, params=params_ref, return_debug=True, bn_updates=upd)
    np.testing.assert_array_equal(got[2].numpy(), exp[2])
    for a, b in zip(got[3]["idx"], exp[3]["idx"]):
        np.testing.assert_array_equal(a.numpy(), b)
    assert np.abs(got[1].numpy() - exp[1]).max() <= 1e-4 * np.abs(exp[1]).max()
    assert set(upd) == {"trn/conv%d_%d" % (i, j) for i in range(2) for j in range(3)} | {"trn/ensemble"}
    for scope, u in upd.items():
        st = pp.bn_state(scope)
        for k in ("moving_mean", "moving_variance"):
            assert np.abs(st[k].numpy() - u[k]).max() <= 1e-4 * max(1e-3, np.abs(u[k]).max()), (scope, k)
    pp.commit_bn()
    assert not np.array_equal(params["trn/conv0_0/bn/moving_mean"], params_ref["trn/conv0_0/bn/moving_mean"])
    for scope, u in upd.items():                                                  # the oracle's view of "after one training step"
        for k in ("moving_mean", "moving_variance"):
            params_ref[scope + "/bn/" + k] = u[k]
    args_inf = args[:3] + (False,) + args[4:]
    got_i = pkg.pointnet_sa_module_msg(torch.from_numpy(xyz), torch.from_numpy(feats), *args_inf, aggregation_channel=64, params=pp)
    exp_i = olayers.pointnet_sa_module_msg(xyz, feats, *args_inf, aggregation_channel=64, params=params_ref)
    assert np.abs(got_i[1].numpy() - exp_i[1]).max() <= 1e-4 * np.abs(exp_i[1]).max()
