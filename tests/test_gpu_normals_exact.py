"""The default (fast) radius normals, bit for bit against the oracle, on scenes whose float sums are exact.

k_normals<0> sums a point's neighbours in cell-run order with fused multiply-adds; the oracle sums them in FLANN's
(d2, index) order with separately rounded products.  Only the order and the fusing differ: the neighbour predicate and
everything after the nine sums are the same operations.  On a dyadic scene (synth.dyadic: coordinates on a 2^-e lattice)
with every partial sum below 2^24 lattice units, each add and fma is exact, so the fast normals must equal the oracle's
exactly -- and so must everything computed from them.  Each test proves that precondition for its scene
(oracle/exact_sums.check) before it compares; a scene that violates it fails the test.

Elsewhere the fast mode is held to statistical bars only (tests/test_gpu_chain.py, tests/test_gpu_parity.py), which a
neighbour counted but left out of the sums, or a sum predicate that differs from the count predicate, can pass when it
touches few points.  Here such a fault changes bits.
"""
import numpy as np
import pytest

from geometric_mapping_b200 import capi, synth
from oracle import chain
from oracle import exact_sums as X
from oracle import oracle as O
from test_gpu_chain import TAU, _assert_canonical
from test_gpu_parity import _fuzz_cloud, _scan_with_junk

pytestmark = pytest.mark.gpu


def _assert_normals_exact(ctx, pts, bound, radius, e, is_dense=True, tag=""):
    """After crop + normals on `ctx`: counts, normals and curvature (NaN rows included), the valid map and the compacted
    cloud and normals equal the oracle's bit for bit.  -> the oracle's neighbour counts."""
    cropped, _ = O.crop(pts, bound, is_dense)
    ref, ref_cnt, _ = O.normals(cropped, radius)
    X.check(cropped, ref_cnt, radius, e, n_sample=1000)
    ref_cloud, ref_nc, ref_vmap = O.compact(cropped, ref)
    assert ctx.counts().device_error == 0, tag
    assert np.array_equal(chain._bits(ctx.download_cloud(0)), chain._bits(cropped)), tag
    assert np.array_equal(ctx.download_neighbor_counts(), ref_cnt), tag + " neighbour counts"
    assert np.array_equal(chain._bits(ctx.download_normals(0)), chain._bits(ref)), tag + " normals"
    assert np.array_equal(ctx.download_valid_map(), ref_vmap), tag + " valid map"
    assert np.array_equal(chain._bits(ctx.download_cloud(1)), chain._bits(ref_cloud)), tag + " compacted cloud"
    assert np.array_equal(chain._bits(ctx.download_normals(1)), chain._bits(ref_nc)), tag + " compacted normals"
    return ref_cnt


def _run_chain(pts, Hp, Hc, radius, leaf, e, f=None):
    """The whole chain on the fast path against the oracle alone: every output compare() checks exactly in canonical
    mode (cylinder hypotheses, test parameters, counts and argmax included) and the canonical bars for the rest."""
    if f is None:
        f = chain.front(pts, radius=radius, leaf=leaf)
    X.check(f["cropped"], f["nbr_count"], radius, e)
    assert f["n_valid"] > 0.5 * len(pts)
    ps = synth.sample_indices(f["n_valid"], Hp, 3, seed=3)
    cs = synth.sample_indices(f["n_valid"], Hc, 2, seed=4)
    b = chain.back(f, ps, cs, tau=TAU)
    assert b["plane_best"] >= 0 and b["cyl_best"] >= 0
    g = chain.gpu_chain(pts, ps, cs, False, radius, leaf)
    _assert_canonical(chain.compare(g, f, b, exact_normals=True))
    return f, b, ps, cs


# ---- the BASELINE scenes, rounded to a lattice, end to end ----------------------------------------------------------
C1_E, C1_R, C1_LEAF = 6, 0.05, 0.1


@pytest.fixture(scope="module")
def c1():
    """C1 (1M-point curved tunnel) on the 2^-6 m lattice and the oracle's front half of the chain for it."""
    pts = synth.dyadic(synth.curved_tunnel(1_000_000, seed=2), C1_E)
    return pts, chain.front(pts, radius=C1_R, leaf=C1_LEAF)


@pytest.mark.parametrize("H", [1024, 4096])
def test_c1_c2_fast_path_is_bit_exact_end_to_end(c1, H):
    """BASELINE configs[1] / [2] on the timed path: r = 0.05 over the 1/64 m lattice (~41 neighbours, worst partial-sum
    bound 0.52 of 2^24)."""
    pts, f = c1
    _run_chain(pts, H // 2, H - H // 2, C1_R, C1_LEAF, C1_E, f)


def test_c0_fast_path_is_bit_exact_end_to_end():
    """BASELINE configs[0]: the 100k straight cylinder on the 1/32 m lattice, r = 0.15."""
    _run_chain(synth.dyadic(synth.straight_cylinder(100_000, seed=1), 5), 512, 512, 0.15, 0.1, 5)


def test_junk_scan_fast_path_is_bit_exact_end_to_end():
    """NaN / inf / out-of-box points, isolated points (NaN normals) and exact duplicates (more of them on the lattice)."""
    pts = synth.curved_tunnel(40_000, seed=5, outlier_frac=0.05)
    pts[100] = [np.nan, 0, 0, 1]
    pts[101] = [0, np.inf, 0, 1]
    pts[102] = [9.0, 0, 0, 1]
    pts[200:210] = pts[300:310]
    _run_chain(synth.dyadic(pts, 6), 128, 128, 0.12, 0.2, 6)


def test_graph_replay_and_a_reused_context_give_the_plain_launch_bits(c1):
    """The dyadic C1 scan through captured-graph replays (graph mode 1) on a context that first processed another scan:
    every exact output equals the oracle's, as the plain launches of test_c1_c2_fast_path_is_bit_exact_end_to_end do."""
    pts, f = c1
    X.check(f["cropped"], f["nbr_count"], C1_R, C1_E)
    ps = synth.sample_indices(f["n_valid"], 512, 3, seed=3)
    cs = synth.sample_indices(f["n_valid"], 512, 2, seed=4)
    b = chain.back(f, ps, cs, tau=TAU)
    other = synth.curved_tunnel(len(pts) - 4321, seed=9)
    with chain.gpu_context(len(pts), ps, cs, C1_R, C1_LEAF) as ctx:
        ctx.set_graph_mode(1)
        ctx.upload_scan(other)
        ctx.process_scan(ps, cs)
        for rep in range(3):   # captured, then replayed
            ctx.upload_scan(pts)
            ctx.process_scan(ps, cs)
            _assert_canonical(chain.compare(chain.gpu_outputs(ctx, ps, cs), f, b, exact_normals=True))
        captures, replays = ctx.graph_stats()
    assert captures >= 1 and replays >= 2


# ---- the neighbour-grid shapes of test_neighbour_grid_shapes_keep_exact_neighbour_sets ------------------------------
@pytest.mark.parametrize("bound,radius,box,e", [
    (5.0, 0.5, None, 5),                                      # the launch-file radius
    (2.6, 2.5, None, 3),                                      # radius ~ the whole cloud
    (50.0, 0.03, None, 7),                                    # crop cube too large for 4-cell blocks of r: enlarged cells
    (5.0, 0.11, ((-5.0, -3.0, -1.7), (5.0, 3.0, 0.2)), 6),    # flat grid box
    (5.0, 0.11, ((-0.5, -0.5, -0.5), (0.5, 0.5, 0.5)), 6),    # box much smaller than the data
    (40.0, 0.2, ((-30.0, -2.0, -2.0), (30.0, 2.0, 2.0)), 5),  # long thin box
])
def test_neighbour_grid_shapes_keep_exact_normals(bound, radius, box, e):
    """Whatever the grid looks like, the fast normals of a dyadic scene are the oracle's; the far-out boxes need a
    coarse lattice for the sums of their distant points to stay exact."""
    pts = _scan_with_junk(25_000, seed=88)
    if bound > 10:
        pts = pts.copy()
        pts[::7, 0] *= 5.0
    pts = synth.dyadic(pts, e)
    with capi.Context(capi.default_params(boxFilterBound=bound, neighborRadius=radius), max_points=len(pts), max_hypotheses=4) as ctx:
        if box is not None:
            ctx.set_grid_box(box[0], box[1])
        ctx.upload_scan(pts)
        ctx.crop()
        ctx.normals()
        _assert_normals_exact(ctx, pts, bound, radius, e, tag=f"bound {bound} r {radius}")


# ---- radii on the lattice: pairs at d2 == r2 exactly ----------------------------------------------------------------
@pytest.mark.parametrize("m", [2, 3, 5])
def test_lattice_radius_and_one_ulp_above(m):
    """r = m * q puts hundreds of thousands of pairs at d2 == r2, which the strict < leaves out; one float ulp above
    r takes them all in.  Between lattice distances a sum predicate that differed from the count predicate near the
    boundary would go unseen; here it changes the sums of most points."""
    e = 5
    pts = synth.dyadic(synth.curved_tunnel(200_000, seed=7, outlier_frac=0.02), e)
    r = m * 2.0 ** -e
    up = float(np.nextafter(np.float32(r), np.float32(np.inf)))
    cnt = {}
    with capi.Context(capi.default_params(neighborRadius=r), max_points=len(pts), max_hypotheses=4) as ctx:
        for radius in (r, up):
            ctx.set_params(capi.default_params(neighborRadius=radius))
            ctx.upload_scan(pts)
            ctx.crop()
            ctx.normals()
            cnt[radius] = _assert_normals_exact(ctx, pts, 5.0, radius, e, tag=f"r {radius!r}")
    assert int((cnt[up] - cnt[r]).sum()) > 100_000       # the boundary pairs exist


# ---- small clouds -----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("seed", [1, 2, 3, 4])
def test_fuzz_small_dyadic_clouds_bit_exact(seed):
    """Small random clouds (degenerate shapes, NaN / inf, lattice points on cell faces), random radius (some on the
    lattice or one ulp above it), bound, is_dense and grid box: runs of length 1, odd run ends and the slack element
    past the last point all occur.  The finest lattice of 2^-7 .. 2^-2 on which the precondition holds is used."""
    g = np.random.Generator(np.random.Philox(2000 + seed))
    with capi.Context(capi.default_params(), max_points=4096, max_hypotheses=4) as ctx:
        for case in range(12):
            n = int(g.choice([0, 1, 2, 3, 7, 33, 200, 1000, 4000]))
            raw = _fuzz_cloud(g, n)
            bound = float(g.choice([0.75, 2.0, 5.0]))
            dense = bool(g.integers(0, 2))
            radius = float(g.choice([0.05, 0.13, 0.4, 1.1, 0.1875, 0.25]))
            if g.integers(0, 2):
                radius = float(np.nextafter(np.float32(radius), np.float32(np.inf)))
            box = None
            if g.integers(0, 2):
                lo = g.uniform(-bound, 0.0, 3)
                box = (lo, lo + g.uniform(0.1, 2.0 * bound, 3))
            for e in range(7, 1, -1):
                pts = synth.dyadic(raw, e)
                cropped, _ = O.crop(pts, bound, dense)
                _, cnt, _ = O.normals(cropped, radius)
                if X.sum_bound(cropped, cnt, radius, e)[0] < X.LIMIT:
                    break
            tag = f"seed {seed} case {case} n {n} bound {bound} r {radius!r} e {e} dense {dense} box {box}"
            ctx.set_params(capi.default_params(boxFilterBound=bound, neighborRadius=radius, is_dense=int(dense)))
            if box is None:
                ctx.set_grid_box()
            else:
                ctx.set_grid_box(box[0], box[1])
            ctx.upload_scan(pts)
            ctx.crop()
            ctx.normals()
            _assert_normals_exact(ctx, pts, bound, radius, e, dense, tag)
