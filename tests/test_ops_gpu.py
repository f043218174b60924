"""GPU parity tests (-m gpu): every operator of libssd3d.so, called through the tf_ops surface (ctypes ->
C ABI), against (a) the CPU oracle and (b) the outputs of the reference's own kernels on the same inputs (ref_ops:
stored under tests/golden/ref_kernels/, see oracle/ref_golden.py).
Integer outputs must be bit-exact; fp32 copies / interpolation bit-exact; the MLP within 1e-3 relative."""
import importlib

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

synth = importlib.import_module("3dssd_b200.synth")


def T(a, dev):
    return torch.from_numpy(np.ascontiguousarray(a)).to(dev)


def N(t):
    return t.detach().cpu().numpy()


# ---------------------------------------------------------------------------------------------------------
# farthest point sampling
# ---------------------------------------------------------------------------------------------------------
FPS_CASES = [
    ("rand300", lambda: np.random.default_rng(0).uniform(-1, 1, (3, 300, 3)).astype(np.float32), 64),
    ("rand1000", lambda: np.random.default_rng(1).uniform(-1, 1, (2, 1000, 3)).astype(np.float32), 100),
    ("rand1500", lambda: np.random.default_rng(2).uniform(-1, 1, (2, 1500, 3)).astype(np.float32), 200),
    ("rand5000", lambda: np.random.default_rng(3).uniform(-1, 1, (2, 5000, 3)).astype(np.float32), 300),
    ("kitti4096", lambda: synth.kitti_like(2, 4096, seed=7)[..., :3].copy(), 512),
    ("lattice3000", lambda: synth.lattice(2, 3000, seed=3), 256),
    ("dups", lambda: np.repeat(np.random.default_rng(4).uniform(-1, 1, (1, 500, 3)).astype(np.float32), 3, axis=1), 600),
    ("allsame", lambda: np.ones((2, 700, 3), np.float32), 50),
    ("single", lambda: np.random.default_rng(5).uniform(-1, 1, (1, 1, 3)).astype(np.float32), 4),
]


@pytest.mark.parametrize("name,gen,m", FPS_CASES, ids=[c[0] for c in FPS_CASES])
def test_fps_xyz_bit_exact_vs_oracle(pkg, oracle_ops, cuda, name, gen, m):
    pts = gen()
    exp = oracle_ops.farthest_point_sample(m, pts)
    got = N(pkg.farthest_point_sample(m, T(pts, cuda)))
    np.testing.assert_array_equal(got, exp)


@pytest.mark.parametrize("variant", [0, 1])
@pytest.mark.parametrize("cl", [1, 2, 4, 8, 16])
def test_fps_every_cluster_size(pkg, oracle_ops, cuda, cl, variant):
    """The result must not depend on how a scene is split over the cluster, nor on the kernel variant
    (0 = automatic: scene-resident 'direct' kernel when it fits; 1 = coordinates-in-packet kernel)."""
    pts = synth.kitti_like(3, 4096, seed=21)[..., :3].copy()
    pts[:, 2000:2100] = pts[:, 100:200]                              # extra duplicates
    exp = oracle_ops.farthest_point_sample(300, pts)
    got = N(pkg.farthest_point_sample(300, T(pts, cuda), cluster=cl, packet_kernel=bool(variant)))   # per-call, no library state
    np.testing.assert_array_equal(got, exp)


@pytest.mark.parametrize("cluster", [0, -4, 8])
@pytest.mark.parametrize("cuts", [(0, 700, 1024), (0, 1, 2, 513, 1024), (0, 1024)])
def test_fps_resumable_rounds(pkg, oracle_ops, cuda, cuts, cluster):
    """Rounds [j0, j1) in separate launches (running distances through `temp`) give the indices of one launch."""
    pts = synth.kitti_like(3, 4096, seed=33)[..., :3].copy()
    pts[:, 3000:3050] = pts[:, 10:60]
    exp = oracle_ops.farthest_point_sample(1024, pts)
    d = T(pts, cuda)
    assert pkg.tf_ops.fps_supports_rounds(4096)
    buf = torch.full((3, 1024), -7, dtype=torch.int32, device=cuda)
    temp = torch.empty((3, 4096), dtype=torch.float32, device=cuda)
    for j0, j1 in zip(cuts[:-1], cuts[1:]):
        pkg.farthest_point_sample(1024, d, out=(buf, 0), rounds=(j0, j1), temp=temp, cluster=cluster)
        assert (N(buf)[:, j1:] == -7).all()                       # later rounds untouched
        np.testing.assert_array_equal(N(buf)[:, :j1], exp[:, :j1])   # a sample is final once its round is done


def _bucket_scenes(kind, b, n, seed):
    rng = np.random.default_rng(seed)
    if kind == "kitti":
        pts = synth.kitti_like(b, n, seed=seed)[..., :3].copy()
        pts[:, n // 2: n // 2 + 40] = pts[:, 3:43]                       # exact duplicates (the loader pads with them)
    elif kind == "uniform":
        pts = rng.uniform(-40, 40, (b, n, 3)).astype(np.float32)
    elif kind == "lattice":                                              # many exactly equal distances: the tie-break decides
        pts = rng.integers(0, 12, (b, n, 3)).astype(np.float32) * 0.5
    elif kind == "line":                                                 # zero extent on two axes
        pts = np.zeros((b, n, 3), np.float32); pts[..., 1] = rng.uniform(0, 100, (b, n))
    else:                                                                # one location only
        pts = np.full((b, n, 3), 2.5, np.float32)
    return pts


@pytest.mark.parametrize("kind,n,m", [("kitti", 16384, 4096), ("kitti", 12001, 3000), ("uniform", 9000, 700), ("lattice", 16384, 2500),
                                      ("line", 8200, 300), ("point", 10000, 260), ("kitti", 4096, 1024), ("uniform", 777, 200),
                                      ("lattice", 64, 64)])
def test_fps_bucket_kernel_bit_exact(pkg, oracle_ops, cuda, kind, n, m):
    """The single-CTA D-FPS with spatial pruning (csrc/fps_bucket.cu) returns the indices of the exhaustive kernels and of
    the CPU oracle, on every kind of scene: skipping a bucket is only ever done when no distance in it can change."""
    pts = _bucket_scenes(kind, 2, n, seed=n + m)
    d = T(pts, cuda)
    got = N(pkg.farthest_point_sample(m, d, bucket_kernel=True))
    exhaustive = N(pkg.farthest_point_sample(m, d, bucket_kernel=False))
    np.testing.assert_array_equal(got, exhaustive)
    np.testing.assert_array_equal(got, oracle_ops.farthest_point_sample(m, pts))
    if n > 8192 and m >= 256:                                            # the default route for these sizes
        np.testing.assert_array_equal(N(pkg.farthest_point_sample(m, d)), got)


@pytest.mark.parametrize("cuts", [(0, 1400, 2500, 3300, 4096), (0, 1, 2, 4096)])
def test_fps_bucket_kernel_resumable_rounds(pkg, cuda, cuts):
    """Rounds in separate launches (distances + bucket permutation through `temp`), strided input, offset output."""
    full = synth.kitti_like(2, 16384 + 512, seed=77)[..., :3].copy()
    d = T(full, cuda)[:, 256:256 + 16384]                                # a slice read in place
    one = pkg.farthest_point_sample(4096, d, bucket_kernel=False)
    elems = pkg.tf_ops.fps_temp_elems(16384, 3, 4096)
    assert elems == 2 * 16384
    buf = torch.full((2, 5000), -7, dtype=torch.int32, device=cuda)
    temp = torch.empty((2, elems), dtype=torch.float32, device=cuda)
    for j0, j1 in zip(cuts[:-1], cuts[1:]):
        pkg.farthest_point_sample(4096, d, out=(buf, 300), idx_offset=1000, rounds=(j0, j1), temp=temp)
        assert bool((buf[:, 300 + j1:] == -7).all()) and bool((buf[:, :300] == -7).all())
        assert torch.equal(buf[:, 300:300 + j1], one[:, :j1] + 1000)


def test_ffps_resumable_rounds(pkg, cuda):
    """The matrix-free F-FPS in separate launches of rounds equals one launch (and therefore the matrix route)."""
    rng = np.random.default_rng(21)
    xyz = T(synth.kitti_like(2, 4096, seed=12)[..., :3].copy(), cuda)
    feat = T(np.maximum(rng.standard_normal((2, 4096, 64)), 0).astype(np.float32), cuda)
    feat[:, 2000:2040] = feat[:, :40]; xyz[:, 2000:2040] = xyz[:, :40]        # duplicates
    one = pkg.tf_ops.farthest_point_sample_features(512, xyz, feat)
    buf = torch.full((2, 512), -3, dtype=torch.int32, device=cuda)
    temp = torch.empty((2, 4096), dtype=torch.float32, device=cuda)
    for j0, j1 in ((0, 256), (256, 300), (300, 512)):
        pkg.tf_ops.farthest_point_sample_features(512, xyz, feat, out=(buf, 0), rounds=(j0, j1), temp=temp)
        assert torch.equal(buf[:, :j1], one[:, :j1]) and bool((buf[:, j1:] == -3).all())


def test_fps_strided_input_offset_output(pkg, oracle_ops, cuda):
    """A [:, a:b] slice read in place; indices written, segment offset added, into a column block of a wider
    buffer (what a fusion-sampling SA layer does, layers_util.py:84-111)."""
    full = synth.kitti_like(3, 2048, seed=8)
    xyz = T(full[..., :3].copy(), cuda)
    feat = T(np.random.default_rng(1).standard_normal((3, 2048, 64)).astype(np.float32), cuda)
    buf = torch.full((3, 600), -1, dtype=torch.int32, device=cuda)
    seg = xyz[:, 1024:2048]
    pkg.farthest_point_sample(200, seg, out=(buf, 100), idx_offset=1024)
    exp = oracle_ops.farthest_point_sample(200, N(seg.contiguous())) + 1024
    np.testing.assert_array_equal(N(buf)[:, 100:300], exp)
    assert (N(buf)[:, :100] == -1).all() and (N(buf)[:, 300:] == -1).all()
    # F-FPS (matrix-free and matrix route) on slices of xyz and features
    segf = feat[:, 1024:2048]
    ref = N(pkg.farthest_point_sample_with_distance(150, pkg.calc_square_dist(torch.cat([seg, segf], -1).contiguous()))) + 1024
    pkg.tf_ops.farthest_point_sample_features(150, seg, segf, out=(buf, 300), idx_offset=1024)
    np.testing.assert_array_equal(N(buf)[:, 300:450], ref)
    pkg.farthest_point_sample_with_distance(150, pkg.calc_square_dist(pkg.tf_ops.concat_cols(seg, segf)), out=(buf, 450), idx_offset=1024)
    np.testing.assert_array_equal(N(buf)[:, 450:600], ref)


def test_fps_65536_vs_reference_kernel(pkg, ref_ops, cuda):
    """BASELINE configs[2] top size: 65536 -> 1024 of 16384 rounds checked against the reference kernel (the 16-CTA
    cluster path, P = 16), D-FPS on xyz and the generic-c kernel on xyz + 5 features."""
    rng = np.random.default_rng(65536)
    pts = np.concatenate([synth.kitti_like(2, 16384, seed=70 + i)[..., :3] for i in range(4)], axis=1).copy()
    pts[:, 60000:60100] = pts[:, 5:105]                              # duplicates far apart in index
    d = T(pts, cuda)
    got = pkg.farthest_point_sample(1024, d)
    assert torch.equal(got, ref_ops.farthest_point_sample(1024, d))
    assert (got[:, 0] == 0).all() and int(got.max()) < 65536
    f = T(np.concatenate([pts, rng.standard_normal((2, 65536, 5)).astype(np.float32)], -1), cuda)
    assert torch.equal(pkg.farthest_point_sample(256, f), ref_ops.farthest_point_sample(256, f))
    # F-FPS 'fused' route where no on-chip kernel holds the features (67 channels x 65536 points): the temp-based kernel
    f67 = T(np.concatenate([pts[:1], rng.standard_normal((1, 65536, 64)).astype(np.float32)], -1), cuda)
    assert pkg.lib().ssd3d_fps_needs_temp(65536, 67) == 1
    assert torch.equal(pkg.farthest_point_sample(48, f67), ref_ops.farthest_point_sample(48, f67))


def test_fps_full_size_vs_reference_kernel(pkg, ref_ops, cuda):
    """BASELINE config-2 layer-1 shape: 16384 -> 4096 on KITTI-like clouds (with duplicate padding)."""
    pts = T(synth.kitti_like(2, 16384, seed=1000)[..., :3].copy(), cuda)
    exp = ref_ops.farthest_point_sample(4096, pts)
    got = pkg.farthest_point_sample(4096, pts)
    assert torch.equal(got, exp)
    # size-independent properties: first index 0, every index in range
    assert (got[:, 0] == 0).all() and int(got.min()) >= 0 and int(got.max()) < 16384


@pytest.mark.parametrize("n,c,m", [(512, 67, 128), (512, 131, 256), (4096, 67, 512), (300, 5, 40), (1000, 19, 77)])
def test_fps_generic_c_bit_exact(pkg, oracle_ops, cuda, n, c, m):
    rng = np.random.default_rng(n + c)
    f = rng.standard_normal((2, n, c)).astype(np.float32)
    f[:, n // 2: n // 2 + 10] = f[:, :10]                            # duplicates
    exp = oracle_ops.farthest_point_sample(m, f)
    got = N(pkg.farthest_point_sample(m, T(f, cuda)))
    np.testing.assert_array_equal(got, exp)


def test_fps_generic_c_vs_reference_kernel(pkg, ref_ops, cuda):
    f = T(np.random.default_rng(9).standard_normal((2, 2048, 67)).astype(np.float32), cuda)
    assert torch.equal(pkg.farthest_point_sample(256, f), ref_ops.farthest_point_sample(256, f))


@pytest.mark.parametrize("n,m,quant", [(384, 96, False), (384, 96, True), (1500, 128, False), (4096, 200, True)])
def test_fps_with_distance_bit_exact(pkg, oracle_ops, ref_ops, cuda, n, m, quant):
    rng = np.random.default_rng(n)
    f = rng.standard_normal((2, n, 6)).astype(np.float32)
    d = T(f, cuda)
    dist = pkg.calc_square_dist(d)
    if quant:
        dist = torch.round(dist * 2) / 2                             # many exact ties
    got = pkg.farthest_point_sample_with_distance(m, dist)
    assert torch.equal(got, ref_ops.farthest_point_sample_with_distance(m, dist))
    if n <= 1500:
        np.testing.assert_array_equal(N(got), oracle_ops.farthest_point_sample_with_distance(m, N(dist)))


def test_calc_square_dist_bit_exact_vs_oracle(pkg, oracle_ops, cuda):
    rng = np.random.default_rng(12)
    for n, c in ((200, 67), (333, 131), (64, 4)):
        f = rng.standard_normal((2, n, c)).astype(np.float32)
        np.testing.assert_array_equal(N(pkg.calc_square_dist(T(f, cuda))), oracle_ops.calc_square_dist(f))


# ---------------------------------------------------------------------------------------------------------
# ball query
# ---------------------------------------------------------------------------------------------------------
def _masked(idx, cnt):
    return idx * (cnt > 0)[..., None].astype(idx.dtype)


BQ_INPUTS = [
    ("kitti4096", lambda: synth.kitti_like(2, 4096, seed=11)[..., :3].copy(), 384),
    ("odd1001", lambda: np.random.default_rng(1).uniform(0, 1, (2, 1001, 3)).astype(np.float32), 77),   # n % 4 != 0: non-TMA path
    ("lattice1500", lambda: synth.lattice(1, 1500, seed=5), 200),
    ("tiny", lambda: np.random.default_rng(2).uniform(0, 1, (3, 5, 3)).astype(np.float32), 5),
]


@pytest.mark.parametrize("name,gen,m", BQ_INPUTS, ids=[c[0] for c in BQ_INPUTS])
@pytest.mark.parametrize("radius,k", [(0.25, 16), (0.5, 32), (2.0, 64), (0.5, 5)])
def test_query_ball_point_bit_exact(pkg, oracle_ops, ref_ops, cuda, name, gen, m, radius, k):
    xyz1 = gen()
    xyz2 = np.array(xyz1[:, :m], copy=True)
    xyz2[:, -1] += 1000.0                                            # one query with an empty ball
    eidx, ecnt = oracle_ops.query_ball_point(radius, k, xyz1, xyz2)
    idx, cnt = pkg.query_ball_point(radius, k, T(xyz1, cuda), T(xyz2, cuda))
    np.testing.assert_array_equal(N(cnt), ecnt)
    np.testing.assert_array_equal(N(idx), eidx)
    ridx, rcnt = ref_ops.query_ball_point(radius, k, T(xyz1, cuda), T(xyz2, cuda))
    assert torch.equal(cnt, rcnt)
    np.testing.assert_array_equal(N(idx), _masked(N(ridx), N(rcnt)))


@pytest.mark.parametrize("name,gen,m", BQ_INPUTS, ids=[c[0] for c in BQ_INPUTS])
@pytest.mark.parametrize("lo,hi,k", [(0.0, 0.25, 16), (0.25, 0.5, 32), (0.5, 2.0, 64)])
def test_query_ball_point_dilated_bit_exact(pkg, oracle_ops, ref_ops, cuda, name, gen, m, lo, hi, k):
    xyz1 = gen()
    xyz2 = np.array(xyz1[:, :m], copy=True)
    xyz2[:, -1] += 1000.0
    eidx, ecnt = oracle_ops.query_ball_point_dilated(lo, hi, k, xyz1, xyz2)
    idx, cnt = pkg.query_ball_point_dilated(lo, hi, k, T(xyz1, cuda), T(xyz2, cuda))
    np.testing.assert_array_equal(N(cnt), ecnt)
    np.testing.assert_array_equal(N(idx), eidx)
    ridx, rcnt = ref_ops.query_ball_point_dilated(lo, hi, k, T(xyz1, cuda), T(xyz2, cuda))
    assert torch.equal(cnt, rcnt)
    np.testing.assert_array_equal(N(idx), _masked(N(ridx), N(rcnt)))


@pytest.mark.parametrize("dilated", [True, False])
def test_query_ball_point_multi_equals_single_calls(pkg, cuda, dilated):
    xyz1 = T(synth.kitti_like(2, 4096, seed=31)[..., :3].copy(), cuda)
    xyz2 = xyz1[:, :500].contiguous()
    radii, ks = [0.4, 0.8, 1.6], [32, 32, 64]
    lows = [0.0, 0.4, 0.8]
    idxs, cnts = pkg.query_ball_point_multi(lows, radii, ks, xyz1, xyz2, dilated)
    for i in range(3):
        if dilated:
            a, c = pkg.query_ball_point_dilated(lows[i], radii[i], ks[i], xyz1, xyz2)
        else:
            a, c = pkg.query_ball_point(radii[i], ks[i], xyz1, xyz2)
        assert torch.equal(idxs[i], a) and torch.equal(cnts[i], c)


@pytest.mark.parametrize("dilated", [False, True])
def test_ball_query_nan_inf_coordinates_vs_reference_kernel(pkg, ref_ops, oracle_ops, cuda, dilated):
    """Non-finite coordinates follow the reference's arithmetic, not an input contract: in the plain query
    max(sqrt(NaN), 1e-20) = 1e-20 < r, so a NaN distance HITS (tf_grouping_g.cu:237-241); in the dilated query every
    comparison with NaN is false, so it never hits (:337-343).  +-Inf distances miss in both."""
    rng = np.random.default_rng(77)
    xyz1 = rng.uniform(0, 1, (2, 700, 3)).astype(np.float32)
    xyz2 = np.array(xyz1[:, :96], copy=True)
    xyz1[0, 5, 0] = np.nan; xyz1[0, 300, 2] = np.nan; xyz1[1, 17, 1] = np.inf; xyz1[1, 400] = -np.inf
    xyz2[0, 3, 1] = np.nan; xyz2[1, 9, 0] = np.inf; xyz2[1, 10, 2] = -np.inf      # NaN / Inf queries too (inf - inf = NaN)
    a, q = T(xyz1, cuda), T(xyz2, cuda)
    for lo, hi, k in ((0.0, 0.3, 16), (0.3, 0.6, 32)):
        if dilated:
            idx, cnt = pkg.query_ball_point_dilated(lo, hi, k, a, q)
            ridx, rcnt = ref_ops.query_ball_point_dilated(lo, hi, k, a, q)
            eidx, ecnt = oracle_ops.query_ball_point_dilated(lo, hi, k, xyz1, xyz2)
        else:
            idx, cnt = pkg.query_ball_point(hi, k, a, q)
            ridx, rcnt = ref_ops.query_ball_point(hi, k, a, q)
            eidx, ecnt = oracle_ops.query_ball_point(hi, k, xyz1, xyz2)
        assert torch.equal(cnt, rcnt)
        np.testing.assert_array_equal(N(idx), _masked(N(ridx), N(rcnt)))
        np.testing.assert_array_equal(N(cnt), ecnt)
        np.testing.assert_array_equal(N(idx), eidx)
    if not dilated:   # the NaN query hits everything in index order: its list is 0..k-1
        idx, cnt = pkg.query_ball_point(0.3, 16, a, q)
        assert N(cnt)[0, 3] == 16 and N(idx)[0, 3].tolist() == list(range(16))
    # the one-pass multi-shell kernel agrees with the single calls on the same inputs
    idxs, cnts = pkg.query_ball_point_multi([0.0, 0.3], [0.3, 0.6], [16, 32], a, q, dilated)
    for i, (lo, hi, k) in enumerate(((0.0, 0.3, 16), (0.3, 0.6, 32))):
        r = pkg.query_ball_point_dilated(lo, hi, k, a, q) if dilated else pkg.query_ball_point(hi, k, a, q)
        assert torch.equal(idxs[i], r[0]) and torch.equal(cnts[i], r[1])


BQG_INPUTS = [
    ("kitti8192", lambda: synth.kitti_like(2, 8192, seed=51)[..., :3].copy()),
    ("cube3000", lambda: synth.uniform_cube(2, 3000, seed=4)),                       # n % 32 != 0
    ("line2048", lambda: np.stack([np.linspace(0, 500, 2048, dtype=np.float32)] + [np.zeros(2048, np.float32)] * 2, -1)[None].repeat(2, 0)),
    ("allsame2048", lambda: np.ones((1, 2048, 3), np.float32)),
    ("nonfinite4096", None),
]


@pytest.mark.parametrize("name,gen", BQG_INPUTS, ids=[c[0] for c in BQG_INPUTS])
@pytest.mark.parametrize("dilated", [False, True])
def test_ball_query_culled_kernel_equals_exhaustive_and_oracle(pkg, oracle_ops, cuda, name, gen, dilated):
    """The spatially culled kernel (uniform grid + index bitmap, csrc/ball_query_grid.cu) returns the bits of the
    exhaustive kernel and of the oracle: clustered, uniform, collinear, coincident and non-finite inputs."""
    if gen is None:
        xyz1 = synth.kitti_like(2, 4096, seed=52)[..., :3].copy()
        xyz1[0, 7, 1] = np.nan; xyz1[0, 3000] = np.inf          # scene 0: non-finite candidates -> one cell; scene 1 finite
    else:
        xyz1 = gen()
    rng = np.random.default_rng(5)
    m = 300
    pick = rng.choice(xyz1.shape[1], m, replace=False)
    xyz2 = np.ascontiguousarray(xyz1[:, pick] + rng.normal(0, 0.05, (xyz1.shape[0], m, 3)).astype(np.float32))
    xyz2[:, 0] = xyz1[:, pick[0]]                                 # an exact self-hit (d == 0)
    xyz2[:, 1] += 1.0e4                                           # far outside the bounding box: empty ball
    if gen is None:
        xyz2[1, 2, 0] = np.nan                                    # non-finite QUERY in a finite scene: scans every cell
    a, q = T(xyz1, cuda), T(xyz2, cuda)
    lows, highs, ks = [0.0, 0.3, 0.6], [0.3, 0.6, 1.7], [16, 32, 64]
    gi, gc = pkg.query_ball_point_multi(lows, highs, ks, a, q, dilated, grid=True)
    ei, ec = pkg.query_ball_point_multi(lows, highs, ks, a, q, dilated, grid=False)
    for s in range(3):
        assert torch.equal(gc[s], ec[s]), "cnt of shell %d" % s
        assert torch.equal(gi[s], ei[s]), "idx of shell %d" % s
        if dilated:
            oi, oc = oracle_ops.query_ball_point_dilated(lows[s], highs[s], ks[s], xyz1, xyz2)
        else:
            oi, oc = oracle_ops.query_ball_point(highs[s], ks[s], xyz1, xyz2)
        np.testing.assert_array_equal(N(gc[s]), oc)
        np.testing.assert_array_equal(N(gi[s]), oi)
    assert int(gc[2][:, 1].max()) == 0 or gen is None             # the far query found nothing


def test_ball_query_full_size_vs_reference_kernel(pkg, ref_ops, cuda):
    """Layer-1 shape of BASELINE config 2: 4096 D-FPS queries over 16384 points, the three dilated shells."""
    pts = T(synth.kitti_like(1, 16384, seed=1003)[..., :3].copy(), cuda)
    fidx = pkg.farthest_point_sample(4096, pts)
    q = pkg.gather_point(pts, fidx)
    idxs, cnts = pkg.query_ball_point_multi([0.0, 0.2, 0.4], [0.2, 0.4, 0.8], [32, 32, 64], pts, q, True)
    for i, (lo, hi, k) in enumerate(((0.0, 0.2, 32), (0.2, 0.4, 32), (0.4, 0.8, 64))):
        ridx, rcnt = ref_ops.query_ball_point_dilated(lo, hi, k, pts, q)
        assert torch.equal(cnts[i], rcnt)
        assert torch.equal(idxs[i], ridx * (rcnt > 0).unsqueeze(-1).to(ridx.dtype))
        assert int(cnts[i].min()) >= 1                               # queries are input points: d == 0 self hit
        valid = torch.arange(1, k, device=cuda)[None, None, :] < cnts[i][..., None]   # slots 1..cnt-1
        ascending = idxs[i][..., 1:] > idxs[i][..., :-1]             # neighbour lists are strictly ascending up to cnt
        assert bool((ascending | ~valid).all())
        backfill = idxs[i] == idxs[i][..., :1]                       # slots >= cnt repeat the first hit
        assert bool((backfill[..., 1:] | valid).all())


# ---------------------------------------------------------------------------------------------------------
# gather / group / interpolation
# ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("c", [3, 13, 64])
def test_gather_and_group_point(pkg, oracle_ops, cuda, c):
    rng = np.random.default_rng(c)
    feats = rng.standard_normal((2, 700, c)).astype(np.float32)
    gi = rng.integers(0, 700, (2, 90)).astype(np.int32)
    np.testing.assert_array_equal(N(pkg.gather_point(T(feats, cuda), T(gi, cuda))), oracle_ops.gather_point(feats, gi))
    gidx = rng.integers(-1, 700, (2, 40, 6)).astype(np.int32)
    np.testing.assert_array_equal(N(pkg.group_point(T(feats, cuda), T(gidx, cuda))), oracle_ops.group_point(feats, gidx))


def test_group_concat_equals_reference_op_sequence(pkg, oracle_ops, cuda):
    rng = np.random.default_rng(3)
    xyz = rng.uniform(0, 1, (2, 300, 3)).astype(np.float32)
    feats = rng.standard_normal((2, 300, 7)).astype(np.float32)
    new_xyz = np.ascontiguousarray(xyz[:, :20])
    idx = rng.integers(0, 300, (2, 20, 8)).astype(np.int32)
    exp = np.concatenate([oracle_ops.group_point(feats, idx), oracle_ops.group_point(xyz, idx) - new_xyz[:, :, None]], -1)
    got = N(pkg.group_concat(T(xyz, cuda), T(feats, cuda), T(new_xyz, cuda), T(idx, cuda), ldx=12))
    np.testing.assert_array_equal(got[..., :10], exp)
    assert (got[..., 10:] == 0).all()


@pytest.mark.parametrize("n,m", [(600, 150), (1030, 2100), (17, 2), (5, 1)])
def test_three_nn_bit_exact(pkg, oracle_ops, ref_ops, cuda, n, m):
    rng = np.random.default_rng(n + m)
    u = rng.uniform(0, 1, (2, n, 3)).astype(np.float32)
    kn = rng.uniform(0, 1, (2, m, 3)).astype(np.float32)
    ed, ei = oracle_ops.three_nn(u, kn)
    d, i = pkg.three_nn(T(u, cuda), T(kn, cuda))
    np.testing.assert_array_equal(N(i), ei)
    np.testing.assert_array_equal(N(d), ed)
    rd, ri = ref_ops.three_nn(T(u, cuda), T(kn, cuda))
    assert torch.equal(i, ri) and torch.equal(d, rd)


def test_three_nn_ties_lattice(pkg, oracle_ops, cuda):
    u, kn = synth.lattice(1, 400, seed=8), synth.lattice(1, 120, seed=9)
    ed, ei = oracle_ops.three_nn(u, kn)
    d, i = pkg.three_nn(T(u, cuda), T(kn, cuda))
    np.testing.assert_array_equal(N(i), ei)
    np.testing.assert_array_equal(N(d), ed)


def test_three_interpolate_bit_exact(pkg, oracle_ops, ref_ops, cuda):
    rng = np.random.default_rng(6)
    pf = rng.standard_normal((2, 150, 20)).astype(np.float32)
    idx = rng.integers(0, 150, (2, 600, 3)).astype(np.int32)
    w = rng.uniform(0, 1, (2, 600, 3)).astype(np.float32)
    got = pkg.three_interpolate(T(pf, cuda), T(idx, cuda), T(w, cuda))
    np.testing.assert_array_equal(N(got), oracle_ops.three_interpolate(pf, idx, w))
    assert torch.equal(got, ref_ops.three_interpolate(T(pf, cuda), T(idx, cuda), T(w, cuda)))


# ---------------------------------------------------------------------------------------------------------
# conv + BN + ReLU (+ max-pool): 1e-3 relative fp32 (BASELINE.json north star)
# ---------------------------------------------------------------------------------------------------------
def rel_err(got, exp, rtol=1e-3, atol_frac=2e-5):
    """max|got-exp| / max|exp| (the global norm the tolerances are quoted in), after ALSO asserting the elementwise
    bound |got - exp| <= rtol*|exp| + atol_frac*max|exp|: a small-magnitude feature may not hide behind a large one."""
    g, e = got.astype(np.float64), exp.astype(np.float64)
    scale = max(1e-12, np.abs(e).max())
    excess = np.abs(g - e) - (rtol * np.abs(e) + atol_frac * scale)
    if excess.size and excess.max() > 0:
        k = np.unravel_index(np.argmax(excess), excess.shape)
        raise AssertionError("elementwise bound exceeded at %s: got %r expected %r (max|exp| %g, %d of %d elements over)"
                             % (k, g[k], e[k], scale, int((excess > 0).sum()), excess.size))
    return float(np.abs(g - e).max() / scale)


@pytest.mark.parametrize("rows,c", [(1000, 1), (333, 3), (4096, 64), (257, 67), (129, 130), (50, 512)])
def test_split_rows_exact(pkg, cuda, rows, c):
    """x = hi + lo with hi = bf16(x), lo = bf16(x - hi), zero padding up to the multiple of 16 (both kernels: 16-byte path
    for c % 4 == 0, scalar otherwise)."""
    x = torch.from_numpy(np.random.default_rng(rows + c).standard_normal((rows, c)).astype(np.float32) * 37.0).to(cuda)
    hi, lo = pkg.split_rows(x)
    kp = (c + 15) // 16 * 16
    assert hi.shape == (rows, kp) and lo.shape == (rows, kp)
    eh = x.to(torch.bfloat16)
    el = (x - eh.float()).to(torch.bfloat16)
    assert torch.equal(hi[:, :c], eh) and torch.equal(lo[:, :c], el)
    assert bool((hi[:, c:] == 0).all()) and bool((lo[:, c:] == 0).all())


@pytest.mark.parametrize("rows,cin,cout", [(1000, 4, 16), (4096, 67, 64), (777, 131, 128), (512, 259, 256), (130, 512, 1024)])
def test_linear_bn_relu_vs_oracle(pkg, oracle_ops, cuda, rows, cin, cout):
    rng = np.random.default_rng(rows)
    x = rng.standard_normal((rows, cin)).astype(np.float32)
    w = (rng.standard_normal((cin, cout)) / np.sqrt(cin)).astype(np.float32)
    b = rng.standard_normal(cout).astype(np.float32)
    bn = (rng.uniform(0.5, 1.5, cout).astype(np.float32), rng.standard_normal(cout).astype(np.float32),
          rng.standard_normal(cout).astype(np.float32), rng.uniform(0.5, 1.5, cout).astype(np.float32))
    exp = oracle_ops.linear_bn_relu(x, w, b, bn, relu=True)
    P = importlib.import_module("3dssd_b200.params")
    params = {"s/weights": w, "s/biases": b, "s/bn/gamma": bn[0], "s/bn/beta": bn[1], "s/bn/moving_mean": bn[2],
              "s/bn/moving_variance": bn[3]}
    f = P.fold(params, "s", True, cuda)
    got = N(pkg.linear_bn_relu(T(x, cuda), f.w, f.scale, f.shift, relu=True))
    assert rel_err(got, exp) < 1e-4                                  # fp32 FMA path: far inside the 1e-3 budget


@pytest.mark.parametrize("pool", [16, 32, 64, 24])
def test_linear_pool_mask(pkg, oracle_ops, cuda, pool):
    rng = np.random.default_rng(pool)
    b, m, cin, cout = 2, 37, 35, 48
    x = rng.standard_normal((b, m, pool, cin)).astype(np.float32)
    w = rng.standard_normal((cin, cout)).astype(np.float32)
    cnt = rng.integers(0, 3, (b, m)).astype(np.int32)
    y = oracle_ops.linear_bn_relu(x, w, None, None, relu=True)
    exp = y.max(axis=2) * (cnt > 0)[..., None]
    one = torch.ones(cout, device=cuda); zero = torch.zeros(cout, device=cuda)
    got = N(pkg.linear_bn_relu(T(x, cuda), T(w, cuda), one, zero, relu=True, pool=pool, rowmask=T(cnt, cuda)))
    assert got.shape == (b, m, cout)
    assert rel_err(got, exp) < 1e-4


# ---------------------------------------------------------------------------------------------------------
# error behaviour (reference: OP_REQUIRES -> InvalidArgument)
# ---------------------------------------------------------------------------------------------------------
def test_argument_validation(pkg, cuda):
    xyz = torch.zeros((1, 10, 3), device=cuda)
    with pytest.raises(ValueError):
        pkg.query_ball_point(-1.0, 4, xyz, xyz)                      # tf_grouping.cpp:275
    with pytest.raises(ValueError):
        pkg.query_ball_point(1.0, 0, xyz, xyz)                       # tf_grouping.cpp:278
    with pytest.raises(ValueError):
        pkg.query_ball_point(1.0, 4, torch.zeros((1, 10, 4), device=cuda), xyz)   # last dim must be 3
    with pytest.raises(ValueError):
        pkg.farthest_point_sample(4, torch.zeros((10, 3), device=cuda))           # rank 3 (tf_sampling.cpp:142)
    with pytest.raises(ValueError):
        pkg.farthest_point_sample_with_distance(4, torch.zeros((1, 10, 9), device=cuda))  # square (cpp:175)
    with pytest.raises(ValueError):
        pkg.gather_point(xyz, torch.zeros((1, 4), dtype=torch.int64, device=cuda))  # int32 indices
    with pytest.raises(ValueError):
        pkg.farthest_point_sample(4, torch.zeros((1, 10, 3)))                     # CPU tensor: no CPU path
    # empty batch / zero samples are no-ops like the reference's early return
    assert pkg.farthest_point_sample(0, xyz).shape == (1, 0)


# ---------------------------------------------------------------------------------------------------------
# tensor-core path (tcgen05, bf16 hi/lo split, 3 MMAs): same 1e-3 budget, expected error ~1e-5
# ---------------------------------------------------------------------------------------------------------
def _fold(pkg, cuda, rng, cin, cout, bn=True):
    P = importlib.import_module("3dssd_b200.params")
    prm = {}
    P._conv_init(rng, prm, "s", cin, cout, bn)
    prm["s/biases"] = rng.standard_normal(cout).astype(np.float32)
    return prm, P.fold(prm, "s", bn, cuda)


def _oracle_conv(oracle_ops, prm, x, bn=True, relu=True):
    bnp = tuple(prm["s/bn/" + k] for k in ("gamma", "beta", "moving_mean", "moving_variance")) if bn else None
    return oracle_ops.linear_bn_relu(x, prm["s/weights"], prm["s/biases"], bnp, relu)


@pytest.mark.parametrize("rows,cin,cout", [(1000, 4, 16), (4096, 67, 64), (777, 131, 128), (512, 259, 256),
                                           (130, 512, 1024), (300, 64, 96), (2048, 128, 192), (256, 128, 3)])
def test_linear_tc_vs_oracle(pkg, oracle_ops, cuda, rows, cin, cout):
    rng = np.random.default_rng(rows + cin)
    prm, f = _fold(pkg, cuda, rng, cin, cout)
    x = rng.standard_normal((rows, cin)).astype(np.float32)
    exp = _oracle_conv(oracle_ops, prm, x)
    hi, lo = pkg.split_rows(T(x, cuda))
    assert hi.shape == (rows, f.kp) and rel_err(N(hi.float() + lo.float())[:, :cin], x) < 2e-5
    y, sp = pkg.linear_tc(hi, lo, f, want_f32=True, want_split=True)
    assert rel_err(N(y), exp) < 1e-4
    yh, yl = sp
    rec = N(yh.float() + yl.float())
    assert rel_err(rec[:, :cout], exp) < 1e-4 and (rec[:, cout:] == 0).all()     # padding columns are zero
    # single-output calls leave through the TMA-store epilogue: must equal the direct-store results bit for bit
    y2, none = pkg.linear_tc(hi, lo, f, want_f32=True, want_split=False)
    assert none is None and torch.equal(y2, y)
    none, (yh2, yl2) = pkg.linear_tc(hi, lo, f, want_f32=False, want_split=True)
    assert none is None and torch.equal(yh2, yh) and torch.equal(yl2, yl)


@pytest.mark.parametrize("pool", [8, 16, 32, 64, 128])
def test_linear_tc_pool_mask_and_concat_slices(pkg, oracle_ops, cuda, pool):
    rng = np.random.default_rng(pool)
    b, m, cin, cout = 2, 37, 67, 64
    prm, f = _fold(pkg, cuda, rng, cin, cout)
    x = rng.standard_normal((b, m, pool, cin)).astype(np.float32)
    cnt = rng.integers(0, 3, (b, m)).astype(np.int32)
    exp = _oracle_conv(oracle_ops, prm, x).max(axis=2) * (cnt > 0)[..., None]
    hi, lo = pkg.split_rows(T(x, cuda))
    concat = torch.full((b, m, 160), -7.0, device=cuda)
    ch = torch.zeros((b, m, 160), dtype=torch.bfloat16, device=cuda); cl = torch.zeros_like(ch)
    pkg.linear_tc(hi, lo, f, pool=pool, rowmask=T(cnt, cuda), out_f32=(concat, 32), out_split=(ch, cl, 32))
    got = N(concat)
    assert rel_err(got[..., 32:96], exp) < 1e-4
    assert (got[..., :32] == -7.0).all() and (got[..., 96:] == -7.0).all()      # neighbours of the slice untouched
    assert rel_err(N(ch.float() + cl.float())[..., 32:96], exp) < 1e-4


def test_linear_tc_three_layer_chain(pkg, oracle_ops, cuda):
    """A whole SA scale as the backbone runs it: gather+concat+split -> 2 split layers -> pooled layer."""
    rng = np.random.default_rng(77)
    b, n, c, m, k = 2, 600, 64, 50, 32
    xyz = rng.uniform(0, 1, (b, n, 3)).astype(np.float32)
    feats = rng.standard_normal((b, n, c)).astype(np.float32)
    new_xyz = np.array(xyz[:, :m], copy=True)
    idx = rng.integers(0, n, (b, m, k)).astype(np.int32)
    cnt = rng.integers(0, 2, (b, m)).astype(np.int32)
    dims = [c + 3, 64, 96, 128]
    g = np.concatenate([oracle_ops.group_point(feats, idx), oracle_ops.group_point(xyz, idx) - new_xyz[:, :, None]], -1)
    hi, lo = pkg.group_concat_split(T(xyz, cuda), T(feats, cuda), T(new_xyz, cuda), T(idx, cuda))
    assert rel_err(N(hi.float() + lo.float())[..., :c + 3], g) < 2e-5
    for li in range(3):
        prm, f = _fold(pkg, cuda, rng, dims[li], dims[li + 1])
        g = _oracle_conv(oracle_ops, prm, g)
        if li < 2:
            _, (hi, lo) = pkg.linear_tc(hi, lo, f, want_f32=False, want_split=True)
        else:
            y, _ = pkg.linear_tc(hi, lo, f, pool=k, rowmask=T(cnt, cuda))
    exp = g.max(axis=2) * (cnt > 0)[..., None]
    assert rel_err(N(y), exp) < 1e-4


def test_linear_tc_large_gemm_matches_fp32_path(pkg, cuda):
    """Layer-4-sized GEMM (65536 x 512 x 1024): tensor-core path vs the exact-fp32 FFMA kernel."""
    torch.manual_seed(0)
    x = torch.randn((8, 256, 32, 512), device=cuda)
    rng = np.random.default_rng(1)
    prm, f = _fold(pkg, cuda, rng, 512, 1024)
    ref = pkg.linear_bn_relu(x, f.w, f.scale, f.shift, relu=True, pool=32)
    hi, lo = pkg.split_rows(x)
    y, _ = pkg.linear_tc(hi, lo, f, pool=32)
    assert rel_err(N(y), N(ref)) < 1e-4


# ---------------------------------------------------------------------------------------------------------
# matrix-free F-FPS == calc_square_dist + farthest_point_sample_with_distance, index for index
# ---------------------------------------------------------------------------------------------------------
FFPS_CASES = [  # b, n, c_feat, m
    (8, 4096, 64, 512),     # 3DSSD layer 2 (cluster of 8, 2 points per thread)
    (8, 512, 128, 256),     # 3DSSD layer 3 (cluster of 2, 1 point per thread, 131 channels)
    (3, 3000, 29, 300),     # n not a multiple of anything, partial last CTA
    (2, 200, 64, 200),      # single CTA, every point picked (m == n)
    (2, 1500, 100, 64),     # 103 channels: the 132-wide variant with a cluster of 8
    (1, 700, 0, 40),        # xyz only
]


@pytest.mark.parametrize("b,n,c,m", FFPS_CASES)
def test_ffps_matrix_free_matches_matrix_route(pkg, oracle_ops, cuda, b, n, c, m):
    rng = np.random.default_rng(n + c)
    xyz = rng.uniform(-3, 3, (b, n, 3)).astype(np.float32)
    feats = np.maximum(rng.standard_normal((b, n, c)), 0).astype(np.float32) if c else None   # post-ReLU like the model's
    if c:
        feats[:, n // 2] = feats[:, n // 3]; xyz[:, n // 2] = xyz[:, n // 3]                   # exact duplicates: ties
    assert pkg.ffps_supported(n, c + 3)
    tx, tf = T(xyz, cuda), (T(feats, cuda) if c else None)
    got = pkg.farthest_point_sample_features(m, tx, tf)
    cat = torch.cat([tx, tf], -1).contiguous() if c else tx
    ref = pkg.farthest_point_sample_with_distance(m, pkg.calc_square_dist(cat))
    assert torch.equal(got, ref)
    if n <= 700:    # and against the CPU oracle's own two-step route
        exp = oracle_ops.farthest_point_sample_with_distance(m, oracle_ops.calc_square_dist(N(cat)))
        np.testing.assert_array_equal(N(got), exp)


def test_ffps_quantised_features_ties(pkg, cuda):
    """Heavily quantised features: many exactly equal distances, the tie-break must follow the matrix route."""
    rng = np.random.default_rng(5)
    xyz = (rng.integers(0, 4, (4, 2048, 3)) * 0.5).astype(np.float32)
    feats = rng.integers(0, 3, (4, 2048, 13)).astype(np.float32)
    tx, tf = T(xyz, cuda), T(feats, cuda)
    got = pkg.farthest_point_sample_features(256, tx, tf)
    ref = pkg.farthest_point_sample_with_distance(256, pkg.calc_square_dist(torch.cat([tx, tf], -1).contiguous()))
    assert torch.equal(got, ref)


def test_ffps_unsupported_shape_is_loud(pkg, cuda):
    assert not pkg.ffps_supported(8192, 67) and not pkg.ffps_supported(1024, 200)
    with pytest.raises(RuntimeError):
        pkg.farthest_point_sample_features(16, torch.zeros((1, 8192, 3), device=cuda), torch.zeros((1, 8192, 64), device=cuda))


# ---------------------------------------------------------------------------------------------------------
# whole SA scale in one kernel (gather + concat + conv stack + max-pool + mask)
# ---------------------------------------------------------------------------------------------------------
FUSED_CASES = [  # b, n, c, m, nsample, mlp
    (2, 700, 1, 96, 32, [16, 16, 32]),       # layer-1 scale 1 shape
    (2, 700, 1, 70, 64, [32, 32, 64]),       # layer-1 scale 3, rows not a multiple of 128 per scene
    (2, 500, 64, 64, 32, [64, 64, 128]),     # layer-2 scale 1
    (1, 500, 64, 50, 64, [64, 96, 128]),     # layer-2 scale 3 (K = 96: partial k-block)
    (3, 300, 29, 33, 16, [48, 32]),          # two layers, nsample 16, odd channel counts
    (2, 300, 5, 17, 8, [16]),                # one layer, nsample 8
    (1, 400, 8, 9, 128, [32, 32, 64]),       # nsample 128: group = whole tile
    (2, 900, 45, 130, 16, [112, 80, 64]),    # K = 48 / 112 / 80: every tail-block width (128 / 128 / 32-byte rows)
    (4, 2000, 64, 512, 32, [64, 64, 128]),   # layer-2 shape, several tiles per slot (3 slots per CTA)
    (2, 2000, 64, 300, 64, [64, 96, 128]),   # 2 slots per CTA, last tile partial
]


@pytest.mark.parametrize("b,n,c,m,k,mlp", FUSED_CASES)
def test_sa_mlp_fused_vs_oracle(pkg, oracle_ops, cuda, b, n, c, m, k, mlp):
    rng = np.random.default_rng(n + c + k)
    xyz = rng.uniform(0, 1, (b, n, 3)).astype(np.float32)
    feats = rng.standard_normal((b, n, c)).astype(np.float32)
    new_xyz = np.array(xyz[:, :m], copy=True)
    idx = rng.integers(0, n, (b, m, k)).astype(np.int32)
    cnt = rng.integers(0, 3, (b, m)).astype(np.int32)
    P = importlib.import_module("3dssd_b200.params")
    prm, scopes, cin = {}, [], c + 3
    for j, cout in enumerate(mlp):
        P._conv_init(rng, prm, "s/conv0_%d" % j, cin, cout, True)
        prm["s/conv0_%d/biases" % j] = rng.standard_normal(cout).astype(np.float32)
        scopes.append("s/conv0_%d" % j)
        cin = cout
    pp = P.prepare(prm, cuda)
    stack = pp.fused_stack(scopes, True, c + 3, limit=0)           # any stack that fits, regardless of the policy limit
    assert stack is not None
    g = np.concatenate([oracle_ops.group_point(feats, idx), oracle_ops.group_point(xyz, idx) - new_xyz[:, :, None]], -1)
    for sc in scopes:
        bnp = tuple(prm[sc + "/bn/" + kk] for kk in ("gamma", "beta", "moving_mean", "moving_variance"))
        g = oracle_ops.linear_bn_relu(g, prm[sc + "/weights"], prm[sc + "/biases"], bnp, True)
    exp = g.max(axis=2) * (cnt > 0)[..., None]
    y = pkg.sa_mlp_fused(T(xyz, cuda), T(feats, cuda), T(new_xyz, cuda), T(idx, cuda), T(cnt, cuda), stack)
    assert y.shape == (b, m, mlp[-1]) and rel_err(N(y), exp) < 1e-4
    # writing into slices of the concat buffers (fp32 + split bf16)
    ld = mlp[-1] + 48
    concat = torch.full((b, m, ld), -3.0, device=cuda)
    ch = torch.zeros((b, m, ld), dtype=torch.bfloat16, device=cuda); cl = torch.zeros_like(ch)
    pkg.sa_mlp_fused(T(xyz, cuda), T(feats, cuda), T(new_xyz, cuda), T(idx, cuda), T(cnt, cuda), stack,
                     out_f32=(concat, 16), out_split=(ch, cl, 16))
    got = N(concat)
    assert rel_err(got[..., 16:16 + mlp[-1]], exp) < 1e-4 and (got[..., :16] == -3.0).all() and (got[..., 16 + mlp[-1]:] == -3.0).all()
    assert rel_err(N(ch.float() + cl.float())[..., 16:16 + mlp[-1]], exp) < 1e-4


def test_sa_mlp_fused_rejects_oversized_stack(pkg, cuda):
    import ctypes
    nout = (ctypes.c_int * 3)(256, 512, 1024)
    assert pkg.lib().ssd3d_sa_fused_smem(256, 3, ctypes.cast(nout, ctypes.c_void_p)) == 0   # layer-4 does not fit
    nout = (ctypes.c_int * 3)(64, 64, 128)
    assert pkg.lib().ssd3d_sa_fused_smem(64, 3, ctypes.cast(nout, ctypes.c_void_p)) > 0


# ---------------------------------------------------------------------------------------------------------
# backward ops (row f3): vs the oracle, and the reference's own style of test (gradient error on random data,
# lib/utils/tf_ops/grouping/tf_grouping_op_test.py:9-25, interpolation/tf_interpolate_op_test.py:9-21)
# ---------------------------------------------------------------------------------------------------------
def test_backward_ops_vs_oracle(pkg, oracle_ops, cuda):
    rng = np.random.default_rng(11)
    feats = rng.standard_normal((2, 300, 13)).astype(np.float32)
    gi = rng.integers(0, 300, (2, 90)).astype(np.int32)
    og = rng.standard_normal((2, 90, 13)).astype(np.float32)
    got = pkg.gather_point_grad(torch.empty((2, 300, 13), device="meta"), T(gi, cuda), T(og, cuda))
    assert rel_err(N(got), oracle_ops.gather_point_grad((2, 300, 13), gi, og)) < 1e-5
    gidx = rng.integers(-1, 300, (2, 40, 6)).astype(np.int32)
    gg = rng.standard_normal((2, 40, 6, 13)).astype(np.float32)
    got = pkg.group_point_grad(torch.empty((2, 300, 13), device="meta"), T(gidx, cuda), T(gg, cuda))
    assert rel_err(N(got), oracle_ops.group_point_grad((2, 300, 13), gidx, gg)) < 1e-5
    idx3 = rng.integers(0, 50, (2, 200, 3)).astype(np.int32)
    w3 = rng.uniform(0, 1, (2, 200, 3)).astype(np.float32)
    go = rng.standard_normal((2, 200, 13)).astype(np.float32)
    got = pkg.three_interpolate_grad(torch.empty((2, 50, 13), device="meta"), T(idx3, cuda), T(w3, cuda), T(go, cuda))
    assert rel_err(N(got), oracle_ops.three_interpolate_grad((2, 50, 13), idx3, w3, go)) < 1e-5


def test_group_point_gradient_error_like_reference_test(pkg, cuda):
    """The reference's only test of this path: gradient error of group_point on random (1,128,16) points with
    query_ball_point(0.3, 32), asserted < 1e-4 (tf_grouping_op_test.py:9-25); same for three_interpolate."""
    torch.manual_seed(0)
    points = torch.rand((1, 128, 16), device=cuda, requires_grad=True)
    xyz1 = torch.rand((1, 128, 3), device=cuda)
    xyz2 = torch.rand((1, 8, 3), device=cuda)
    idx, _ = pkg.query_ball_point(0.3, 32, xyz1, xyz2)
    out = pkg.group_point(points, idx)
    wgt = torch.rand_like(out)
    (out * wgt).sum().backward()
    analytic = points.grad.clone()
    # the op is linear in `points`: the exact gradient is the scatter-add of the weights
    expected = torch.zeros_like(analytic)
    expected.index_put_((torch.zeros_like(idx, dtype=torch.long).flatten(), idx.flatten().long()),
                        wgt.reshape(-1, 16), accumulate=True)
    assert float((analytic - expected).abs().max()) < 1e-4
    # three_interpolate
    pts = torch.rand((1, 8, 16), device=cuda, requires_grad=True)
    dist, nidx = pkg.three_nn(xyz1, xyz2)
    w = torch.ones_like(dist) / 3.0
    y = pkg.three_interpolate(pts, nidx, w)
    wy = torch.rand_like(y)
    (y * wy).sum().backward()
    exp = torch.zeros_like(pts)
    for k in range(3):
        exp.index_put_((torch.zeros((128,), dtype=torch.long, device=cuda), nidx[0, :, k].long()), wy[0] * w[0, :, k:k + 1],
                       accumulate=True)
    assert float((pts.grad - exp).abs().max()) < 1e-4
    # gather_point
    src = torch.rand((2, 64, 5), device=cuda, requires_grad=True)
    gi = torch.randint(0, 64, (2, 20), device=cuda, dtype=torch.int32)
    g = pkg.gather_point(src, gi)
    g.sum().backward()
    cnt = torch.zeros((2, 64), device=cuda)
    cnt.scatter_add_(1, gi.long(), torch.ones((2, 20), device=cuda))
    assert torch.allclose(src.grad, cnt.unsqueeze(-1).expand(-1, -1, 5))


@pytest.mark.parametrize("b,n,c,m,k,cout,pooled", [(2, 600, 64, 50, 32, 64, False), (2, 500, 128, 33, 32, 128, False),
                                                   (1, 700, 256, 20, 16, 256, False), (2, 300, 29, 17, 16, 48, False),
                                                   (2, 300, 5, 40, 32, 16, True), (1, 256, 1, 9, 64, 32, False)])
def test_linear_tc_gather_equals_materialised_path(pkg, oracle_ops, cuda, b, n, c, m, k, cout, pooled):
    """Gather fused into the operand load == group_concat_split + linear_tc (bit for bit), and both match the oracle."""
    rng = np.random.default_rng(n + c)
    xyz = rng.uniform(0, 1, (b, n, 3)).astype(np.float32)
    feats = rng.standard_normal((b, n, c)).astype(np.float32)
    new_xyz = np.array(xyz[:, :m], copy=True)
    idx = rng.integers(0, n, (b, m, k)).astype(np.int32)
    cnt = rng.integers(0, 3, (b, m)).astype(np.int32)
    prm, f = _fold(pkg, cuda, rng, c + 3, cout)
    t = lambda a: T(a, cuda)
    hi, lo = pkg.group_concat_split(t(xyz), t(feats), t(new_xyz), t(idx))
    g = np.concatenate([oracle_ops.group_point(feats, idx), oracle_ops.group_point(xyz, idx) - new_xyz[:, :, None]], -1)
    exp = _oracle_conv(oracle_ops, prm, g)
    if pooled:
        y0, _ = pkg.linear_tc(hi, lo, f, pool=k, rowmask=t(cnt))
        y1, _ = pkg.linear_tc_gather(t(xyz), t(feats), t(new_xyz), t(idx), f, pool=k, rowmask=t(cnt), want_f32=True,
                                     want_split=False)
        assert torch.equal(y0, y1)
        assert rel_err(N(y1), exp.max(axis=2) * (cnt > 0)[..., None]) < 1e-4
    else:
        _, (h0, l0) = pkg.linear_tc(hi, lo, f, want_f32=False, want_split=True)
        _, (h1, l1) = pkg.linear_tc_gather(t(xyz), t(feats), t(new_xyz), t(idx), f)
        assert torch.equal(h0, h1) and torch.equal(l0, l1)
        assert rel_err(N(h1.float() + l1.float())[..., :cout], exp) < 1e-4


# ---------------------------------------------------------------------------------------------------------
# hoisted first conv: per-point table + second conv with the operand rebuilt per grouped row
# ---------------------------------------------------------------------------------------------------------
HOIST_CASES = [  # b, n, c, m, nsample, mlp
    (2, 600, 128, 70, 32, [128, 128, 256]),      # layer-3 shape, rows not a multiple of 128
    (2, 400, 256, 40, 16, [256, 512, 1024]),     # layer-4 scale: second conv has two 256-wide n-tiles
    (3, 300, 29, 33, 8, [48, 40]),               # two layers only (second conv pools), odd widths (n1 = 48 -> kp 48)
    (1, 500, 64, 50, 64, [72, 96, 64]),          # n1 = 72: K padded to 80, z row pitch not a multiple of 16 bytes... (72*4 ok)
]


@pytest.mark.parametrize("b,n,c,m,k,mlp", HOIST_CASES)
def test_hoisted_first_conv_matches_oracle_and_gather_path(pkg, oracle_ops, cuda, b, n, c, m, k, mlp):
    rng = np.random.default_rng(n + c + k)
    xyz = rng.uniform(0, 70, (b, n, 3)).astype(np.float32)          # KITTI-sized coordinates: the xyz part cancels
    feats = np.maximum(rng.standard_normal((b, n, c)), 0).astype(np.float32)
    new_xyz = np.array(xyz[:, :m], copy=True)
    idx = rng.integers(0, n, (b, m, k)).astype(np.int32)
    xyz[np.arange(b)[:, None, None], idx] = new_xyz[:, :, None, :] + rng.uniform(-2, 2, (b, m, k, 3)).astype(np.float32)
    cnt = rng.integers(0, 3, (b, m)).astype(np.int32)
    P = importlib.import_module("3dssd_b200.params")
    prm, scopes, cin = {}, [], c + 3
    for j, cout in enumerate(mlp):
        P._conv_init(rng, prm, "s/conv0_%d" % j, cin, cout, True)
        prm["s/conv0_%d/biases" % j] = rng.standard_normal(cout).astype(np.float32)
        scopes.append("s/conv0_%d" % j)
        cin = cout
    pp = P.prepare(prm, cuda)
    g = np.concatenate([oracle_ops.group_point(feats, idx), oracle_ops.group_point(xyz, idx) - new_xyz[:, :, None]], -1)
    for sc in scopes:
        bnp = tuple(prm[sc + "/bn/" + kk] for kk in ("gamma", "beta", "moving_mean", "moving_variance"))
        g = oracle_ops.linear_bn_relu(g, prm[sc + "/weights"], prm[sc + "/biases"], bnp, True)
    exp = g.max(axis=2) * (cnt > 0)[..., None]
    tx, tf, tn, ti, tc = T(xyz, cuda), T(feats, cuda), T(new_xyz, cuda), T(idx, cuda), T(cnt, cuda)
    zconv, wxs, n1s = pp.hoisted([scopes[0]], True, c)
    p_hi, p_lo = pkg.split_rows(tf)
    z, _ = pkg.linear_tc(p_hi, p_lo, zconv, relu=False, want_f32=True, want_split=False)
    f1 = pp.conv(scopes[1], True)
    if len(mlp) == 2:
        y, _ = pkg.linear_tc_hoisted(tx, z, 0, wxs[0], tn, ti, f1, pool=k, rowmask=tc, want_f32=True, want_split=False)
    else:
        _, (hi, lo) = pkg.linear_tc_hoisted(tx, z, 0, wxs[0], tn, ti, f1)
        y, _ = pkg.linear_tc(hi, lo, pp.conv(scopes[2], True), pool=k, rowmask=tc, want_f32=True, want_split=False)
    assert y.shape == (b, m, mlp[-1]) and rel_err(N(y), exp) < 1e-4
    # the materialised form of the same operand (wide layers take it): identical split operand -> identical GEMM result
    ehi, elo = pkg.tf_ops.hoist_expand_split(tx, z, 0, wxs[0], tn, ti)
    if len(mlp) == 2:
        y2, _ = pkg.linear_tc(ehi, elo, f1, pool=k, rowmask=tc, want_f32=True, want_split=False)
    else:
        _, (hi2, lo2) = pkg.linear_tc(ehi, elo, f1, want_f32=False, want_split=True)
        y2, _ = pkg.linear_tc(hi2, lo2, pp.conv(scopes[2], True), pool=k, rowmask=tc, want_f32=True, want_split=False)
    assert rel_err(N(y2), N(y)) < 1e-6


@pytest.mark.parametrize("b,n,c,m,k,mlp", [
    (2, 700, 1, 96, 32, [16, 16, 32]),       # layer-1 scale 1: one feature channel, n1 = 16
    (2, 700, 1, 70, 64, [32, 32, 64]),       # layer-1 scale 3
    (4, 2000, 64, 512, 32, [64, 64, 128]),   # layer-2 (3 slots per CTA)
    (2, 2000, 64, 300, 64, [64, 96, 128]),   # layer-2 scale 3
    (3, 300, 29, 33, 16, [48, 32]),          # two convs: the fused stack is a single conv
])
def test_sa_mlp_fused_hoisted_vs_oracle(pkg, oracle_ops, cuda, b, n, c, m, k, mlp):
    rng = np.random.default_rng(n + c + k + 1)
    xyz = rng.uniform(0, 70, (b, n, 3)).astype(np.float32)
    feats = np.maximum(rng.standard_normal((b, n, c)), 0).astype(np.float32)
    new_xyz = np.array(xyz[:, :m], copy=True)
    idx = rng.integers(0, n, (b, m, k)).astype(np.int32)
    cnt = rng.integers(0, 3, (b, m)).astype(np.int32)
    P = importlib.import_module("3dssd_b200.params")
    prm, scopes, cin = {}, [], c + 3
    for j, cout in enumerate(mlp):
        P._conv_init(rng, prm, "s/conv0_%d" % j, cin, cout, True)
        prm["s/conv0_%d/biases" % j] = rng.standard_normal(cout).astype(np.float32)
        prm["s/conv0_%d/bn/gamma" % j][1::3] *= -1.0                  # negative BatchNorm scales: the last layer's are
        scopes.append("s/conv0_%d" % j)                               # folded into its weights (pool-before-affine)
        cin = cout
    pp = P.prepare(prm, cuda)
    g = np.concatenate([oracle_ops.group_point(feats, idx), oracle_ops.group_point(xyz, idx) - new_xyz[:, :, None]], -1)
    for sc in scopes:
        bnp = tuple(prm[sc + "/bn/" + kk] for kk in ("gamma", "beta", "moving_mean", "moving_variance"))
        g = oracle_ops.linear_bn_relu(g, prm[sc + "/weights"], prm[sc + "/biases"], bnp, True)
    exp = g.max(axis=2) * (cnt > 0)[..., None]
    tx, tf, tn, ti, tc = T(xyz, cuda), T(feats, cuda), T(new_xyz, cuda), T(idx, cuda), T(cnt, cuda)
    zconv, wxs, n1s = pp.hoisted([scopes[0]], True, c)
    p_hi, p_lo = pkg.split_rows(tf)
    z, _ = pkg.linear_tc(p_hi, p_lo, zconv, relu=False, want_f32=True, want_split=False)
    stack = pp.fused_stack(scopes[1:], True, n1s[0], limit=0)
    assert stack is not None
    y = pkg.sa_mlp_fused_hoisted(tx, z, 0, wxs[0], tn, ti, tc, stack)
    # absolute coordinates up to 70 m: |(x_j - c_i) . Wx| is compared on the scale of the layer's outputs
    assert y.shape == (b, m, mlp[-1]) and rel_err(N(y), exp) < 1e-4


@pytest.mark.parametrize("c,ks,mlps,hoist", [
    (1, [32, 32, 64], [[16, 16, 32], [16, 16, 32], [32, 32, 64]], False),      # layer 1
    (64, [32, 32, 64], [[64, 64, 128], [64, 64, 128], [64, 96, 128]], True),   # layer 2 (first conv hoisted)
    (7, [16, 8, 128], [[48, 32], [16], [32, 32, 64]], False),                  # other group sizes
])
def test_sa_mlp_fused_unit_list_equals_dense(pkg, cuda, c, ks, mlps, hoist):
    """The unit-list route (only the 8-row units holding distinct neighbours are convolved, combined by atomicMax) gives
    the SAME BITS as the dense route: a group's skipped rows repeat its first neighbour (grouping/tf_grouping_g.cu:99-109),
    whose activation is already inside unit 0.  Dense clusters (cnt > nsample), isolated centres (cnt = 1) and empty
    dilated shells (cnt = 0) are all present; every third BatchNorm scale is negative."""
    rng = np.random.default_rng(c + sum(ks))
    b, n, m = 3, 4096, 600
    centres = rng.uniform(0, 40, (b, 40, 3))
    clustered = centres[np.arange(b)[:, None], rng.integers(0, 40, (b, 1500))] + rng.normal(0, 0.15, (b, 1500, 3))
    xyz = np.concatenate([clustered, rng.uniform(0, 40, (b, n - 1500, 3))], 1).astype(np.float32)
    perm = rng.permutation(n)
    xyz = np.ascontiguousarray(xyz[:, perm])
    feats = np.maximum(rng.standard_normal((b, n, c)), 0).astype(np.float32)
    tx, tf = T(xyz, cuda), T(feats, cuda)
    tn = tx[:, :m].contiguous()
    tn[:, -20:] += 500.0                                       # centres with no neighbour in any shell: cnt = 0
    lows, highs = [0.0, 0.2, 0.4], [0.2, 0.4, 0.8]
    idxs, cnts, units = pkg.query_ball_point_multi(lows, highs, ks, tx, tn, True, grid=True, return_units=True)
    i0, c0 = pkg.query_ball_point_multi(lows, highs, ks, tx, tn, True, grid=False)
    P = importlib.import_module("3dssd_b200.params")
    for s in range(3):
        assert units[s] is not None and torch.equal(idxs[s], i0[s]) and torch.equal(cnts[s], c0[s])
        cnt = N(cnts[s]); k = ks[s]
        u = N(units[s]); nu = int(u[0])
        assert nu == int(np.minimum((np.minimum(cnt, k) + 7) // 8, (k + 7) // 8)[cnt > 0].sum())   # ceil(min(cnt, K) / 8) per non-empty group
        grp, j = u[1:1 + nu] >> 4, u[1:1 + nu] & 15
        want = sorted((int(g), int(jj)) for g in np.flatnonzero(cnt.reshape(-1) > 0)
                      for jj in range((min(int(cnt.reshape(-1)[g]), k) + 7) // 8))
        assert sorted(zip(grp.tolist(), j.tolist())) == want
        assert (cnt == 0).any() and (cnt == 1).any() and (cnt >= min(k, 9)).any()
        prm, scopes, cin = {}, [], c + 3
        for jn, cout in enumerate(mlps[s]):
            P._conv_init(rng, prm, "s/conv%d_%d" % (s, jn), cin, cout, True)
            prm["s/conv%d_%d/bn/gamma" % (s, jn)][1::3] *= -1.0
            scopes.append("s/conv%d_%d" % (s, jn)); cin = cout
        pp = P.prepare(prm, cuda)
        ld = mlps[s][-1] + 32
        dense = torch.full((b, m, ld), -1.0, device=cuda)
        comp = torch.full((b, m, ld), -1.0, device=cuda)
        comp[..., 16:16 + mlps[s][-1]] = 0.0
        if hoist:
            zconv, wxs, n1s = pp.hoisted([scopes[0]], True, c)
            p_hi, p_lo = pkg.split_rows(tf)
            z, _ = pkg.linear_tc(p_hi, p_lo, zconv, relu=False, want_f32=True, want_split=False)
            stack = pp.fused_stack(scopes[1:], True, n1s[0], limit=0)
            assert stack is not None
            pkg.sa_mlp_fused_hoisted(tx, z, 0, wxs[0], tn, idxs[s], cnts[s], stack, out_f32=(dense, 16))
            pkg.sa_mlp_fused_hoisted(tx, z, 0, wxs[0], tn, idxs[s], cnts[s], stack, out_f32=(comp, 16), units=units[s])
        else:
            stack = pp.fused_stack(scopes, True, c + 3, limit=0)
            assert stack is not None
            pkg.sa_mlp_fused(tx, tf, tn, idxs[s], cnts[s], stack, out_f32=(dense, 16))
            pkg.sa_mlp_fused(tx, tf, tn, idxs[s], cnts[s], stack, out_f32=(comp, 16), units=units[s])
        assert torch.equal(dense, comp)
        assert float(dense[..., 16:16 + mlps[s][-1]].abs().max()) > 0
    with pytest.raises(ValueError):
        pkg.sa_mlp_fused(tx, tf, tn, idxs[0], cnts[0], stack, units=units[0])          # needs the zero-filled out_f32


@pytest.mark.parametrize("c,k,mlp,expand", [
    (64, 32, [64, 96, 128], False),      # hoisted second conv built inside the GEMM (layer-3 route), three convs
    (64, 64, [64, 128], False),          # two convs: the hoisted conv is the pooled one
    (256, 32, [256, 256, 320], True),    # operand materialised by hoist_expand_split (layer-4 route)
    (32, 16, [32, 40], True),
])
def test_linear_tc_unit_list_equals_dense(pkg, cuda, c, k, mlp, expand):
    """Layer-by-layer scales through the *_units kernels (compact rows, 8-row units pooled by atomicMax) give the same bits
    as the dense kernels.  Small candidate set: the unit list comes from group_units_kernel, in group order."""
    rng = np.random.default_rng(c + k)
    b, n, m = 3, 512, 200
    xyz = np.concatenate([rng.normal(0, 0.4, (b, 200, 3)) + 5.0, rng.uniform(0, 30, (b, n - 200, 3))], 1).astype(np.float32)
    xyz = np.ascontiguousarray(xyz[:, rng.permutation(n)])
    feats = np.maximum(rng.standard_normal((b, n, c)), 0).astype(np.float32)
    tx, tf = T(xyz, cuda), T(feats, cuda)
    tn = tx[:, :m].contiguous()
    tn[:, -10:] += 500.0
    (idx,), (cnt,), (units,) = pkg.query_ball_point_multi([0.0], [1.2], [k], tx, tn, False, return_units=True)
    cn = N(cnt).reshape(-1)
    assert (cn == 0).any() and (cn == 1).any() and (cn > 8).any()
    want = [(g << 4) | j for g in range(cn.size) for j in range((min(int(cn[g]), k) + 7) // 8)]
    u = N(units)
    assert int(u[0]) == len(want) and u[1:1 + len(want)].tolist() == want
    P = importlib.import_module("3dssd_b200.params")
    prm, scopes, cin = {}, [], c + 3
    for jn, cout in enumerate(mlp):
        P._conv_init(rng, prm, "s/conv0_%d" % jn, cin, cout, True)
        prm["s/conv0_%d/bn/gamma" % jn][1::3] *= -1.0
        scopes.append("s/conv0_%d" % jn); cin = cout
    pp = P.prepare(prm, cuda)
    zconv, wxs, n1s = pp.hoisted([scopes[0]], True, c)
    p_hi, p_lo = pkg.split_rows(tf)
    z, _ = pkg.linear_tc(p_hi, p_lo, zconv, relu=False, want_f32=True, want_split=False)
    ld = mlp[-1] + 32
    dense = torch.full((b, m, ld), -1.0, device=cuda)
    comp = torch.full((b, m, ld), -1.0, device=cuda)
    comp[..., 16:16 + mlp[-1]] = 0.0

    def run(out, ukw, last_kw):
        f1 = pp.conv(scopes[1], True)
        if len(mlp) == 2:
            if expand:
                hi, lo = pkg.tf_ops.hoist_expand_split(tx, z, 0, wxs[0], tn, idx, **ukw)
                pkg.linear_tc(hi, lo, f1, out_f32=(out, 16), **last_kw)
            else:
                pkg.linear_tc_hoisted(tx, z, 0, wxs[0], tn, idx, f1, want_split=False, out_f32=(out, 16), **last_kw)
            return
        if expand:
            hi, lo = pkg.tf_ops.hoist_expand_split(tx, z, 0, wxs[0], tn, idx, **ukw)
            _, (hi, lo) = pkg.linear_tc(hi, lo, f1, want_f32=False, want_split=True, **ukw)
        else:
            _, (hi, lo) = pkg.linear_tc_hoisted(tx, z, 0, wxs[0], tn, idx, f1, **ukw)
        pkg.linear_tc(hi, lo, pp.conv(scopes[2], True), out_f32=(out, 16), **last_kw)

    run(dense, {}, dict(pool=k, rowmask=cnt))
    run(comp, dict(units=units), dict(units=units, unit_pool=True))
    assert torch.equal(dense, comp)
    assert float(dense[..., 16:16 + mlp[-1]].max()) > 0
    with pytest.raises(ValueError):
        pkg.linear_tc(p_hi, p_lo, zconv, units=units, pool=8)


def test_peer_allgather_protocol_three_simulated_ranks(pkg, cuda):
    """csrc/peer_gather.cu on ONE device: three "ranks" are three streams, each with its own symmetric buffer (here plain
    allocations of the same process -- the kernel only sees addresses).  Several replays: parity reuse, the device-side
    replay counter and the flag protocol; every rank ends with everybody's slice of that replay."""
    dist_mod = pkg.dist
    world, slice_bytes = 3, 28832
    recv_off, flag_off, total = dist_mod.peer_layout(world, slice_bytes)
    assert recv_off[1] == world * slice_bytes and flag_off[0] == 2 * world * slice_bytes and total >= flag_off[1] + world * 4
    sym = [torch.zeros((total,), dtype=torch.uint8, device=cuda) for _ in range(world)]
    peers = torch.tensor([t.data_ptr() for t in sym], dtype=torch.int64, device=cuda)
    send = [torch.zeros((slice_bytes,), dtype=torch.uint8, device=cuda) for _ in range(world)]
    out = [torch.zeros((world * slice_bytes,), dtype=torch.uint8, device=cuda) for _ in range(world)]
    state = [torch.zeros((4,), dtype=torch.int32, device=cuda) for _ in range(world)]
    streams = [torch.cuda.Stream(device=cuda) for _ in range(world)]
    gen = torch.Generator(device="cpu").manual_seed(5)
    for replay in range(1, 6):
        payload = [torch.randint(0, 256, (slice_bytes,), dtype=torch.uint8, generator=gen) for _ in range(world)]
        for r in range(world):
            send[r].copy_(payload[r])
        torch.cuda.synchronize()
        for r in (2, 0, 1):                                      # launch order != rank order: early ranks wait for late ones
            with torch.cuda.stream(streams[r]):
                pkg.tf_ops.peer_allgather(send[r], peers, world, r, slice_bytes, recv_off, flag_off, state[r], out[r])
        torch.cuda.synchronize()
        want = torch.cat(payload)
        for r in range(world):
            assert torch.equal(out[r].cpu(), want), "rank %d replay %d" % (r, replay)
            assert state[r].cpu().tolist()[:3] == [replay, 0, 0]


# ---------------------------------------------------------------------------------------------------------
# training-mode BatchNorm (row f3)
# ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("rows,c", [(5000, 48), (131072, 256), (7, 3)])
def test_bn_train_vs_float64(pkg, cuda, rows, c):
    rng = np.random.default_rng(rows)
    x = (rng.standard_normal((rows, c)) * rng.uniform(0.1, 5, c) + rng.uniform(-3, 3, c) + 100.0 * (np.arange(c) % 5 == 0)).astype(np.float32)
    g, be = rng.uniform(0.5, 1.5, c).astype(np.float32), rng.normal(0, 0.2, c).astype(np.float32)
    mm, mv = rng.normal(0, 1, c).astype(np.float32), rng.uniform(0.5, 2, c).astype(np.float32)
    tmm, tmv = T(mm, cuda), T(mv, cuda)
    y, scale, shift, bm, bv = pkg.tf_ops.bn_train(T(x, cuda), T(g, cuda), T(be, cuda), tmm, tmv, decay=0.9, relu=True)
    xd = x.astype(np.float64)
    mean, var = xd.mean(0), xd.var(0)
    inv = g / np.sqrt(var + 1e-3)
    exp = np.maximum(xd * inv + (be - mean * inv), 0)
    assert rel_err(N(bm), mean.astype(np.float32), atol_frac=1e-6) < 1e-6
    assert rel_err(N(bv), var.astype(np.float32), rtol=1e-4, atol_frac=1e-6) < 1e-4      # offset channels: E[x^2]-E[x]^2 in double
    assert rel_err(N(y), exp.astype(np.float32)) < 1e-4
    np.testing.assert_allclose(N(tmm), mm - (mm - mean) * 0.1, rtol=1e-5, atol=1e-5)
    np.testing.assert_allclose(N(tmv), mv - (mv - var) * 0.1, rtol=1e-4, atol=1e-5)
    np.testing.assert_allclose(N(scale), inv, rtol=1e-5)
