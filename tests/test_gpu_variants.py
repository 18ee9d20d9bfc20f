"""Every kernel variant that frame size and the PREVIOUS frame on a context select, against the oracle.

Which instantiation of the radix sort runs (`radix_coop_kernel<ITEMS, MASK_TABLE>`, grid, waves), how many digit passes
the pair sort makes, how the binning splits its large-footprint queue and which blend kernel writes the pixels are all
picked at launch time from the frame's size and from counts the previous frame left behind (`n_vis_hint`,
`n_pairs_hint`).  Each case here runs on a FRESH context and sets that hint on purpose with a primer frame, then holds the
frame to the oracle: sorted (key, index) entries, tile ranges and per-tile slices bit-exact, pixels within 1e-3.

The first half of the file restates the selection arithmetic in Python (each function cites what it restates) and a
CPU-only test checks that the case table below reaches every instantiation, pass count and `part_shift`.  The GPU tests
re-derive the variant of every frame and put it in their assertion messages, so a change of the heuristics shows up as
a coverage failure rather than as silently lost coverage.
"""
from __future__ import annotations

import dataclasses

import numpy as np
import pytest

import bevy_gaussian_splatting_b200 as B

PIXEL_TOL = 1e-3
B200_SMS = 148

# ---------------------------------------------------------------------------------------------------------------------
# A. mirror of the selection arithmetic
# ---------------------------------------------------------------------------------------------------------------------
RS_THREADS = 512                      # radix.cu:27
RS_ITEM_SIZES = (2, 4, 6, 8, 10, 12, 16)
SORT_VARIANTS = tuple(f"<{i},MASK_TABLE>" for i in RS_ITEM_SIZES) + ("<16,MATCH.ANY>",)
SORT_CTAS_PER_SM, SORT_CTAS_PER_SM_QUEUED = 2, 1      # api.cu:373-375 (DESIGN §5: 2 co-resident, queued pair sort 1)
BIN_CTAS_PER_SM, BIN_CTAS_PER_SM_QUEUED = 4, 1        # api.cu:364-372
BIN_WARPS_PER_CTA = 256 // 32                         # bin.cu:13
BIN_BIG = 128                                         # bin.cu:18: larger footprints go to the large queue


@dataclasses.dataclass(frozen=True)
class SortLaunch:
    items: int
    mask_table: bool
    grid: int
    waves: int

    @property
    def variant(self) -> str:
        return f"<{self.items},{'MASK_TABLE' if self.mask_table else 'MATCH.ANY'}>"

    def __str__(self):
        return f"{self.variant} grid={self.grid} waves={self.waves}"


def radix_num_tiles(capacity: int) -> int:
    """radix.cu:329-332: look-back status rows of a sort of up to `capacity` entries."""
    return max(capacity // (RS_THREADS * 16) + 1, 4096)


def radix_launch(sm_count: int, coop_per_sm: int, capacity: int, status_capacity: int, hint: int) -> SortLaunch:
    """radix.cu:374-404 (`launch_radix_sort`): items per thread and grid from the hint, clamped to the capacity;
    `status_capacity` is what the status rows were sized for (api.cu:282-298, grow-only)."""
    hint = min(hint, capacity)
    want = hint + hint // 32 + 1024

    def items_for(g):
        per_wave = g * RS_THREADS * 16
        waves = -(-want // per_wave)
        return -(-want // (g * RS_THREADS * waves)), waves

    grid = sm_count
    items, waves = items_for(grid)
    if waves > 1 and coop_per_sm >= 2:
        grid = 2 * sm_count
        items, waves = items_for(grid)
    if waves > 3:
        items = 17
    rows = radix_num_tiles(status_capacity)
    items = max(items, -(-capacity // (rows * RS_THREADS)))
    for it in RS_ITEM_SIZES:
        if items <= it:
            return SortLaunch(it, True, grid, waves)
    return SortLaunch(16, False, grid, waves)


def pair_passes(num_tiles: int) -> int:
    """api.cu:209-213: 8-bit digit passes of the tile-id sort."""
    bits = 1
    while (1 << bits) < num_tiles:
        bits += 1
    return (bits + 7) // 8


def part_shift(big_count: int, grid_ctas: int) -> int:
    """bin.cu:349-351: the large-footprint queue is dealt as big_count << part_shift tickets over the grid's warps."""
    total_warps = grid_ctas * BIN_WARPS_PER_CTA
    ps = 0
    while ps < 4 and (big_count << (ps + 2)) <= total_warps:
        ps += 1
    return ps


def tile_count(xlo, xhi, ylo, yhi):
    """bin.cu:203-204: tiles a pixel bbox (inclusive) touches; 0 for an empty bbox."""
    xlo, xhi, ylo, yhi = (np.asarray(a, np.int64) for a in (xlo, xhi, ylo, yhi))
    return np.where((xlo <= xhi) & (ylo <= yhi), ((xhi >> 4) - (xlo >> 4) + 1) * ((yhi >> 4) - (ylo >> 4) + 1), 0)


class ContextMirror:
    """What a context remembers between frames and what it launches from it (api.cu:534-577 finish_frame,
    api.cu:711-852 render_impl): the hints, the grow-only pair capacity and status rows."""

    def __init__(self, sm_count: int):
        self.sm = sm_count
        self.n_vis_hint = self.n_pairs_hint = self.cap_pairs = self.status_n = self.status_np = 0

    def frame(self, n: int, n_vis: int, n_pairs: int, num_tiles: int, sort_all: bool = False, queued: bool = False,
              big_count: int = 0) -> dict:
        """One frame (a queued one must fit the pair buffer: sizing it is a synchronous frame's job here)."""
        if self.cap_pairs == 0:
            self.cap_pairs = max(n, 1 << 20)                                     # api.cu:711-715
        if n_pairs > self.cap_pairs:
            assert not queued, "a queued frame overflowing the pair buffer is re-rendered after bgs_sync"
            self.cap_pairs = n_pairs + n_pairs // 4 + 1024                       # api.cu:543-552, the frame is redone
        self.status_n = max(self.status_n, n)
        self.status_np = max(self.status_np, self.cap_pairs)
        d_hint = n if sort_all else (self.n_vis_hint or n)                       # api.cu:788-789
        depth = radix_launch(self.sm, SORT_CTAS_PER_SM, n, self.status_n, d_hint)
        p_hint = min(self.n_pairs_hint or self.cap_pairs, self.cap_pairs)        # api.cu:847-849
        pair = radix_launch(self.sm, SORT_CTAS_PER_SM_QUEUED if queued else SORT_CTAS_PER_SM, self.cap_pairs, self.status_np, p_hint)
        large_fp = self.n_vis_hint > 0 and self.n_pairs_hint >= 8 * self.n_vis_hint   # api.cu:827
        bin_grid = self.sm * (BIN_CTAS_PER_SM_QUEUED if queued else BIN_CTAS_PER_SM)
        out = dict(depth=depth, pair=pair, passes=pair_passes(num_tiles), blend="raster2_kernel" if large_fp else "raster_kernel<0>",
                   part_shift=part_shift(big_count, bin_grid), queued=queued)
        self.n_vis_hint, self.n_pairs_hint = n_vis, n_pairs
        return out


# ---------------------------------------------------------------------------------------------------------------------
# the case table (B to E); the GPU tests run exactly these
# ---------------------------------------------------------------------------------------------------------------------
FRONT = (480, 272)            # 30 x 17 = 510 tiles: 2 pair-sort passes
SIDE = (256, 256)             # 256 tiles: 1 pair-sort pass
BASE_N = 2_090_000            # the sort cases' cloud (<= 2^21 entries: the capacity does not raise the tile size)
SIDE_N = 300                  # splats only the side camera sees (the "stale large hint" frames)
SMALL_PRIMER = 1000


@dataclasses.dataclass(frozen=True)
class SortCase:
    name: str
    m: int                    # visible splats (= pairs: each covers one tile) of the test frame
    bits: int
    primer: str               # "count": the same frame first; "small": a 1 000-splat frame; "p<count>": a frame of that many


SORT_CASES = [
    # hint = count: one instantiation each (and the side frame after it: the same hint, a few hundred entries)
    SortCase("count-2", 100_000, 16, "count"), SortCase("count-4", 250_000, 24, "count"),
    SortCase("count-6", 400_000, 32, "count"), SortCase("count-8", 550_000, 16, "count"),
    SortCase("count-10", 700_000, 24, "count"), SortCase("count-12", 850_000, 32, "count"),
    SortCase("count-16", 1_100_000, 16, "count"),
    SortCase("count-10-2cta", 1_300_000, 24, "count"), SortCase("count-16-2cta", 2_000_000, 32, "count"),
    # stale small hint (1 000): 1 024-entry tiles, one wave exactly +- 1, tile edges k * 1024 +- 1, many tiles per CTA
    SortCase("small-wave-1", 148 * 1024 - 1, 32, "small"), SortCase("small-wave", 148 * 1024, 16, "small"),
    SortCase("small-wave+1", 148 * 1024 + 1, 32, "small"),
    SortCase("small-tile-1", 400 * 1024 - 1, 16, "small"), SortCase("small-tile", 400 * 1024, 32, "small"),
    SortCase("small-tile+1", 400 * 1024 + 1, 24, "small"), SortCase("small-2M", 2_000_000, 16, "small"),
    # hint from a 400 000-splat frame: <6> (3 072-entry tiles, grid 148): one wave +- 1, tile edges with idle CTAs
    SortCase("p400k-wave-1", 148 * 3072 - 1, 16, "p400000"), SortCase("p400k-wave", 148 * 3072, 32, "p400000"),
    SortCase("p400k-wave+1", 148 * 3072 + 1, 16, "p400000"),
    SortCase("p400k-tile-1", 100 * 3072 - 1, 32, "p400000"), SortCase("p400k-tile", 100 * 3072, 16, "p400000"),
    SortCase("p400k-tile+1", 100 * 3072 + 1, 24, "p400000"),
]

BIG_N, BIG_FRONT = 8_000_000, 7_400_000     # the multi-wave sorts: MATCH.ANY ranking
PASS_VIEWPORTS = [(256, 256), (4112, 16), (4096, 4096), (4112, 4096)]   # 256 / 257 / 65 536 / 65 792 tiles
BIG_QUEUE_TARGETS = [1, 50, 300, 3000]


def sort_case_frames(case: SortCase, sm: int):
    """The frames of one SortCase on a fresh context -> list of (label, mirror result)."""
    ctx = ContextMirror(sm)
    front_tiles, side_tiles = (FRONT[0] // 16) * (FRONT[1] // 16), (SIDE[0] // 16) * (SIDE[1] // 16)
    out = []
    if case.primer == "count":
        ctx.frame(BASE_N, case.m, case.m, front_tiles)
    elif case.primer == "small":
        ctx.frame(SMALL_PRIMER + SIDE_N, SMALL_PRIMER, SMALL_PRIMER, front_tiles)
    else:
        p = int(case.primer[1:])
        ctx.frame(BASE_N, p, p, front_tiles)
    if case.primer in ("count", "small"):
        regime = "hint=count" if case.primer == "count" else "stale small hint"
    else:
        regime = "stale hint > count" if int(case.primer[1:]) > case.m else "stale small hint"
    out.append((regime, ctx.frame(BASE_N, case.m, case.m, front_tiles)))
    out.append(("hint=count", ctx.frame(BASE_N, case.m, case.m, front_tiles)))
    if case.primer == "count":
        out.append(("stale large hint", ctx.frame(BASE_N, SIDE_N, SIDE_N, side_tiles)))
    return out


def big_cloud_frames(sm: int):
    """test_match_any_sorts: the 8 M cloud (7.4 M in front, 300 at the side)."""
    front_tiles, side_tiles = (1920 // 16) * (1088 // 16), (SIDE[0] // 16) * (SIDE[1] // 16)
    ctx = ContextMirror(sm)
    out = [("hint=count (sort_all)", ctx.frame(BIG_N, BIG_FRONT, BIG_FRONT, front_tiles, sort_all=True))]
    out.append(("hint=count", ctx.frame(BIG_N, BIG_FRONT, BIG_FRONT, front_tiles)))
    out.append(("stale large hint", ctx.frame(BIG_N, SIDE_N, SIDE_N, side_tiles)))
    small = ContextMirror(sm)
    small.frame(SMALL_PRIMER + SIDE_N, SMALL_PRIMER, SMALL_PRIMER, front_tiles)
    out.append(("stale small hint", small.frame(BIG_N, BIG_FRONT, BIG_FRONT, front_tiles)))
    return out


def queued_frames(sm: int):
    """Queued frames of the tests: the > 3.7 M-pair scene (after a synchronous frame sized the buffer), the large-queue
    scenes and C3 (721 340 visible, 1 392 163 pairs, DESIGN §5) round-robin."""
    out = []
    ctx = ContextMirror(sm)
    ctx.frame(400_000, 360_000, 3_900_000, 8160)
    out.append(("queued, hint=count", ctx.frame(400_000, 360_000, 3_900_000, 8160, queued=True)))
    for k in BIG_QUEUE_TARGETS:
        for queued in (False, True):
            c = ContextMirror(sm)
            out.append((f"large queue {k}", c.frame(20_000, 20_000, 200_000, 8160, queued=queued, big_count=k)))
    c3 = ContextMirror(sm)
    c3.frame(6_000_000, 721_340, 1_392_163, 8160)
    out.append(("C3 queued", c3.frame(6_000_000, 721_340, 1_392_163, 8160, queued=True)))
    return out


def pass_count_frames(sm: int):
    return [("passes", ContextMirror(sm).frame(20_000, 10_000, 40_000, ((w + 15) // 16) * ((h + 15) // 16))) for w, h in PASS_VIEWPORTS]


def table_coverage(sm: int = B200_SMS):
    frames = []
    for case in SORT_CASES:
        frames += sort_case_frames(case, sm)
    frames += big_cloud_frames(sm) + queued_frames(sm) + pass_count_frames(sm)
    cov = dict(depth=set(), pair=set(), pair_queued=set(), passes=set(), part_shift_sync=set(), part_shift_queued=set(),
               depth_regimes=set(), pair_regimes=set())
    for regime, f in frames:
        cov["depth"].add(f["depth"].variant)
        cov["depth_regimes"].add((f["depth"].variant, regime))
        cov["pair_queued" if f["queued"] else "pair"].add(f["pair"].variant)
        cov["pair_regimes"].add((f["pair"].variant, regime + (" queued" if f["queued"] else "")))
        cov["passes"].add(f["passes"])
        cov["part_shift_queued" if f["queued"] else "part_shift_sync"].add(f["part_shift"])
    return cov


def test_selection_mirror_reaches_every_variant():
    """CPU: the case table reaches every sort instantiation (depth and pair sort), 1 / 2 / 3 pair passes and part_shift
    0, 4 and values in between under both binning grids."""
    cov = table_coverage(B200_SMS)
    summary = "\n".join(f"{k}: {sorted(v)}" for k, v in cov.items())
    assert cov["depth"] == set(SORT_VARIANTS), summary
    assert cov["pair"] == set(SORT_VARIANTS), summary
    assert "<16,MATCH.ANY>" in cov["pair_queued"], summary
    assert cov["passes"] == {1, 2, 3}, summary
    for k in ("part_shift_sync", "part_shift_queued"):
        assert {0, 4} <= cov[k] and cov[k] & {1, 2, 3}, summary
    print(summary)


def test_selection_mirror_spot_values():
    """CPU: hand-checked values of the mirror (DESIGN §5's C3 frame: 721 340 entries -> <10> on 148 CTAs; the
    multi-wave thresholds; the pass counts at 2^8 / 2^16 tiles)."""
    assert str(radix_launch(148, 2, 6_000_000, 6_000_000, 721_340)) == "<10,MASK_TABLE> grid=148 waves=1"
    assert radix_launch(148, 2, 8_000_000, 8_000_000, 7_400_000).variant == "<16,MATCH.ANY>"
    assert radix_launch(148, 2, 8_000_000, 8_000_000, 6_900_000).variant == "<16,MASK_TABLE>"
    assert radix_launch(148, 1, 5_000_000, 5_000_000, 3_700_000).variant == "<16,MATCH.ANY>"
    assert radix_launch(148, 2, 8_000_000, 8_000_000, 1000).variant == "<4,MASK_TABLE>"       # min_items from capacity
    assert [pair_passes(t) for t in (1, 256, 257, 65536, 65537)] == [1, 1, 2, 2, 3]
    assert [part_shift(k, 592) for k in (1, 50, 300, 1200)] == [4, 4, 2, 0]
    assert [part_shift(k, 148) for k in (1, 50, 300)] == [4, 3, 0]
    assert list(tile_count([0, 0, 5], [15, 16, 4], [0, 0, 0], [15, 40, 0])) == [1, 6, 0]


# ---------------------------------------------------------------------------------------------------------------------
# scene construction (fixed seeds)
# ---------------------------------------------------------------------------------------------------------------------
def front_view(w=FRONT[0], h=FRONT[1]):
    return B.perspective_view((0.0, 1.5, 5.0), (0.0, 1.5, 4.0), w, h)


def side_view():
    """Same eye, looking along +x: sees only the side group (the front group lies >= 50 degrees off its axis)."""
    return B.perspective_view((0.0, 1.5, 5.0), (1.0, 1.5, 5.0), SIDE[0], SIDE[1])


def tile_centred(view, m, rng, dmin=2.0, dmax=30.0):
    """m points whose projections are tile centres of `view` (W, H multiples of 16), at depths U(dmin, dmax)."""
    W, H = view.width, view.height
    tx, ty = W // 16, H // 16
    t = rng.integers(0, tx * ty, m)
    nx = ((t % tx) * 16 + 8.0) / W * 2.0 - 1.0
    ny = 1.0 - ((t // tx) * 16 + 8.0) / H * 2.0
    ndc = np.stack([nx, ny, 0.1 / rng.uniform(dmin, dmax, m), np.ones(m)], 1)
    w = ndc @ np.linalg.inv(view.clip_from_world.astype(np.float64)).T
    return (w[:, :3] / w[:, 3:]).astype(np.float32)


def attribute_planes(n, seed, scale=1e-3):
    """SH / rotation / scale+opacity from a 64 K pool (tiled: cheap at 8 M): tiny splats (~1 pixel) by default."""
    rng = np.random.default_rng(seed)
    pool = min(n, 1 << 16)
    sh = rng.uniform(-1, 1, (pool, 48)).astype(np.float32)
    rot = rng.uniform(-1, 1, (pool, 4)).astype(np.float32)
    so = np.concatenate([rng.uniform(0.3, 1.0, (pool, 3)) * scale, rng.uniform(0.2, 0.8, (pool, 1))], 1).astype(np.float32)
    idx = np.arange(n) % pool
    return sh[idx], rot[idx], so[idx]


def sort_scene_positions(n, m, seed, front=None):
    """[0, m): tile-centred in the front view; [n - SIDE_N, n): tile-centred in the side view; the rest behind the eye."""
    rng = np.random.default_rng(seed)
    pos = np.ones((n, 4), np.float32)
    pos[:m, :3] = tile_centred(front or front_view(), m, rng)
    nb = n - m - SIDE_N
    pos[m:n - SIDE_N, 0] = rng.uniform(-0.3, 0.3, nb)
    pos[m:n - SIDE_N, 1] = 1.5 + rng.uniform(-0.3, 0.3, nb)
    pos[m:n - SIDE_N, 2] = rng.uniform(6.0, 30.0, nb)
    pos[n - SIDE_N:, :3] = tile_centred(side_view(), SIDE_N, rng)
    return pos


def sort_scene(n, m, planes, seed=1, front=None):
    sh, rot, so = planes
    return B.PlanarGaussian3d(sort_scene_positions(n, m, seed, front), sh, rot, so)


@pytest.fixture(scope="module")
def base_planes():
    return attribute_planes(BASE_N, 7)


@pytest.fixture(scope="module")
def sm_count():
    import torch

    return torch.cuda.get_device_properties(0).multi_processor_count


def fresh():
    return B.GaussianSplattingPlugin(0)


def check_frame(p, oracle, cloud, settings, view, img, what, transform=None, pixels=True, aabb=None):
    """The frame just rendered on `p` against the oracle: sorted entries, counts, tile ranges and slices bit-exact,
    pixels (rgba32f) within PIXEL_TOL.  `what` goes into every message."""
    u = p.cloud_uniform(settings, transform, aabb)
    bits = int(settings.radix_sort_depth_bits)
    keys = oracle.keygen(cloud.position_visibility, view.to_abi(), u, bits)
    sk, si = oracle.radix_sort(keys, bits)
    got = p.sorted_entries()
    assert np.array_equal(got[:, 0], sk), f"sorted keys differ: {what}"
    assert np.array_equal(got[:, 1], si), f"sort permutation differs: {what}"
    til = oracle.render_tiles(cloud, view.to_abi(), u, settings.to_abi(), want_image=pixels)
    fs = p.frame_stats()
    assert fs.rounds == 1, what
    assert (fs.n_visible, fs.n_pairs) == (til["n_vis"], til["n_pairs"]), what
    assert np.array_equal(p.tile_ranges(), til["tile_ranges"]), f"tile ranges differ: {what}"
    assert np.array_equal(p.tile_entries(), til["tile_entries"]), f"per-tile slices differ: {what}"
    if pixels:
        err = float(np.abs(img - til["image"]).max())
        assert err <= PIXEL_TOL, f"pixel L-inf {err}: {what}"
    return til


# ---------------------------------------------------------------------------------------------------------------------
# B / C. depth sort and pair sort: instantiation x hint regime, tile and wave edges
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("case", SORT_CASES, ids=[c.name for c in SORT_CASES])
def test_sort_variants_vs_oracle(oracle, base_planes, sm_count, case):
    """Every splat covers exactly one tile, so the pair sort sorts as many entries as the depth sort: both run the
    variant the mirror names, at the counts the case sets (tile edges, wave edges, several tiles per CTA)."""
    frames = sort_case_frames(case, sm_count)
    s = B.CloudSettings(global_scale=1.0, radix_sort_depth_bits=B.RadixSortDepthBits(case.bits))
    view = front_view()
    cloud = sort_scene(BASE_N, case.m, base_planes, seed=case.m)
    p = fresh()
    handles = []
    try:
        h = p.add_cloud(cloud)
        handles.append(h)
        if case.primer == "count":
            p.render_view(h, s, view, to_host=False)
        elif case.primer == "small":
            sp = attribute_planes(SMALL_PRIMER + SIDE_N, 3)
            hp = p.add_cloud(sort_scene(SMALL_PRIMER + SIDE_N, SMALL_PRIMER, sp, seed=3))
            handles.append(hp)
            p.render_view(hp, s, view, to_host=False)
            assert p.frame_stats().n_visible == SMALL_PRIMER
        else:
            pc = int(case.primer[1:])
            hp = p.add_cloud(sort_scene(BASE_N, pc, base_planes, seed=pc))
            handles.append(hp)
            p.render_view(hp, s, view, to_host=False)
            assert p.frame_stats().n_visible == pc
        (regime, f), (_, f2) = frames[0], frames[1]
        what = f"{case.name}, {regime}: depth sort {f['depth']}, pair sort {f['pair']} ({f['passes']} passes)"
        img = p.render_view(h, s, view)
        til = check_frame(p, oracle, cloud, s, view, img, what)
        assert til["n_vis"] == case.m and til["n_pairs"] == case.m, f"construction: one tile per splat ({what})"
        ent = p.sorted_entries()
        again = p.render_view(h, s, view)
        what2 = f"{case.name}, re-render (hint=count): depth sort {f2['depth']}, pair sort {f2['pair']}"
        assert np.array_equal(img.view(np.uint32), again.view(np.uint32)), what2
        assert np.array_equal(p.sorted_entries(), ent), what2
        assert np.array_equal(p.tile_ranges(), til["tile_ranges"]), what2
        if len(frames) > 2:
            regime3, f3 = frames[2]
            sv = side_view()
            what3 = f"{case.name}, side view, {regime3}: depth sort {f3['depth']}, pair sort {f3['pair']} ({f3['passes']} pass)"
            side = p.render_view(h, s, sv)
            st = check_frame(p, oracle, cloud, s, sv, side, what3)
            assert st["n_vis"] == SIDE_N, what3
            assert np.array_equal(side.view(np.uint32), p.render_view(h, s, sv).view(np.uint32)), what3
    finally:
        for hh in handles:
            hh.destroy()
        p.destroy()


@pytest.fixture(scope="module")
def big_cloud():
    """8 M gaussians: 7.4 M one-tile splats in a 1920x1088 front view, 300 at the side, the rest behind the eye."""
    return sort_scene(BIG_N, BIG_FRONT, attribute_planes(BIG_N, 11), seed=12, front=front_view(1920, 1088))


@pytest.mark.gpu
def test_match_any_sorts_and_stale_hints_at_8m(oracle, big_cloud, sm_count):
    """The multi-wave sorts (<16, MATCH.ANY>): sort_all over 8 M entries; 7.4 M visible (depth and pair sort); a few
    hundred entries after a 7.4 M hint on the SAME cloud (the hint is clamped to the cloud's size: a smaller cloud would
    hide it); and 7.4 M entries after a 1 000-entry hint (capacity-bounded tiles, ~25 tiles per CTA)."""
    frames = big_cloud_frames(sm_count)
    view, sv = front_view(1920, 1088), side_view()
    s_all = B.CloudSettings(global_scale=1.0, sort_all=True, radix_sort_depth_bits=B.RadixSortDepthBits(16))
    s = B.CloudSettings(global_scale=1.0, radix_sort_depth_bits=B.RadixSortDepthBits(16))
    p = fresh()
    try:
        h = p.add_cloud(big_cloud)
        regime, f = frames[0]
        img_all = p.render_view(h, s_all, view)
        what = f"8M sort_all, {regime}: depth sort {f['depth']}"
        u = p.cloud_uniform(s_all)
        keys = oracle.keygen(big_cloud.position_visibility, view.to_abi(), u, 16)
        sk, si = oracle.radix_sort(keys, 16)
        ent = p.sorted_entries()
        assert np.array_equal(ent[:, 0], sk) and np.array_equal(ent[:, 1], si), what
        assert int((sk == 0xFFFF).sum()) == BIG_N - BIG_FRONT and np.diff(sk[:BIG_FRONT].astype(np.int64)).min() == 0
        regime, f = frames[1]
        what = f"8M, 7.4M visible, {regime}: depth sort {f['depth']}, pair sort {f['pair']}"
        img = p.render_view(h, s, view)
        assert np.array_equal(img, img_all), what
        til = check_frame(p, oracle, big_cloud, s, view, img, what, pixels=False)
        assert BIG_FRONT <= til["n_pairs"] < BIG_FRONT + BIG_FRONT // 1000, what      # (a few near splats straddle two tiles)
        regime, f = frames[2]
        what = f"8M cloud, side view, {regime}: depth sort {f['depth']}, pair sort {f['pair']}"
        side = p.render_view(h, s, sv)
        assert check_frame(p, oracle, big_cloud, s, sv, side, what)["n_vis"] == SIDE_N
        assert np.array_equal(side, p.render_view(h, s, sv)), what
        h.destroy()
    finally:
        p.destroy()
    regime, f = frames[3]
    what = f"8M cloud after a 1 000-splat frame, {regime}: depth sort {f['depth']}, pair sort {f['pair']}"
    p = fresh()
    try:
        hp = p.add_cloud(sort_scene(SMALL_PRIMER + SIDE_N, SMALL_PRIMER, attribute_planes(SMALL_PRIMER + SIDE_N, 3), seed=3))
        p.render_view(hp, s, view, to_host=False)
        h = p.add_cloud(big_cloud)
        again = p.render_view(h, s, view)
        assert np.array_equal(again, img), what
        assert np.array_equal(p.sorted_entries(), ent), what
        assert np.array_equal(p.tile_ranges(), til["tile_ranges"]), what
        assert np.array_equal(p.tile_entries(), til["tile_entries"]), what
        h.destroy(); hp.destroy()
    finally:
        p.destroy()


# ---------------------------------------------------------------------------------------------------------------------
# C. pair-sort passes, footprint classes, the large-footprint queue
# ---------------------------------------------------------------------------------------------------------------------
def mixed_cloud(n, seed, scale_lo=1e-3, scale_hi=0.05):
    """A random cloud in front of the headless camera with log-uniform scales: footprints from one tile to thousands."""
    c = B.random_gaussians_3d_seeded(n, seed)
    rng = np.random.default_rng(seed)
    c.position_visibility[:, 2] = np.float32(-rng.uniform(0.0, 25.0, n))
    c.position_visibility[:, :2] *= np.float32(0.4)
    c.scale_opacity[:, :3] = np.exp(rng.uniform(np.log(scale_lo), np.log(scale_hi), (n, 3))).astype(np.float32)
    c.scale_opacity[:, 3] = rng.uniform(0.2, 0.8, n).astype(np.float32)
    return c


@pytest.mark.gpu
@pytest.mark.parametrize("w,h", PASS_VIEWPORTS, ids=[f"{w}x{h}" for w, h in PASS_VIEWPORTS])
def test_pair_sort_passes_vs_oracle(oracle, sm_count, w, h):
    """1 / 2 / 3 digit passes of the tile-id sort: 256 tiles, 257 tiles, 65 536 tiles (the largest frame that may be
    binned in rounds) and 65 792 tiles (3 passes, never in rounds)."""
    cloud = mixed_cloud(20000, 5, 1e-3, 0.02)
    view = B.headless_view(w, h)
    s = B.CloudSettings()
    p = fresh()
    try:
        hd = p.add_cloud(cloud)
        img = p.render_view(hd, s, view)
        fs = p.frame_stats()
        what = f"{w}x{h}: {fs.tiles_x * fs.tiles_y} tiles, {pair_passes(fs.tiles_x * fs.tiles_y)} pair-sort passes"
        til = check_frame(p, oracle, cloud, s, view, img, what)
        assert til["n_pairs"] > til["n_vis"] > 1000, what
        assert np.array_equal(img, p.render_view(hd, s, view)), what
        hd.destroy()
    finally:
        p.destroy()


def footprint_sweep(view, seed):
    """Axis-aligned splats centred in tiles, their pixel extents swept finely in x and y: every tile width x height up
    to the view, including 1 x (> 128) columns and footprints that are no multiple of 32 or of 16."""
    rng = np.random.default_rng(seed)
    sx = np.concatenate([np.full(40, 1e-4), np.exp(np.linspace(np.log(1e-3), np.log(0.3), 24))])
    sy = np.exp(np.linspace(np.log(1e-3), np.log(3.0), 90))
    gx, gy = np.meshgrid(sx, sy)
    k = gx.size
    pos = np.ones((k, 4), np.float32)
    pos[:, :3] = tile_centred(view, k, rng, 4.0, 8.0)
    so = np.stack([gx.ravel(), gy.ravel(), np.full(k, 1e-3), rng.uniform(0.2, 0.8, k)], 1).astype(np.float32)
    rot = np.tile(np.array([1, 0, 0, 0], np.float32), (k, 1))
    return B.PlanarGaussian3d(pos, rng.uniform(-1, 1, (k, 48)).astype(np.float32), rot, so)


def concat(*clouds):
    return B.PlanarGaussian3d(*(np.concatenate([getattr(c, f) for c in clouds]) for f in
                                ("position_visibility", "spherical_harmonic", "rotation", "scale_opacity")))


def projected_tile_counts(oracle, cloud, view, s, u=None):
    u = u if u is not None else B.GaussianSplattingPlugin.cloud_uniform(s)
    til = oracle.render_tiles(cloud, view.to_abi(), u, s.to_abi(), want_image=False)
    rec = oracle.project(cloud, view.to_abi(), u, s.to_abi(), til["rank_to_id"])
    return rec, tile_count(rec["xlo"], rec["xhi"], rec["ylo"], rec["yhi"])


@pytest.mark.gpu
def test_binning_footprint_classes_vs_oracle(oracle):
    """Splats of exactly 4 / 5 / 128 / 129 tiles (the thread / medium-queue / large-queue bounds), one-tile-wide columns
    taller than 128 tiles and large footprints that are no multiple of 32, synchronously and queued."""
    view = B.perspective_view((0.0, 1.5, 5.0), (0.0, 1.5, 4.0), 768, 2304)
    s = B.CloudSettings(opacity_adaptive_radius=False)
    cloud = concat(footprint_sweep(view, 21), mixed_cloud(4000, 22, 1e-3, 0.03))
    rec, cnt = projected_tile_counts(oracle, cloud, view, s)
    w = (rec["xhi"].astype(np.int64) >> 4) - (rec["xlo"].astype(np.int64) >> 4) + 1
    hgt = (rec["yhi"].astype(np.int64) >> 4) - (rec["ylo"].astype(np.int64) >> 4) + 1
    have = set(cnt.tolist())
    assert {4, 5, 128, 129} <= have, "the construction must straddle the footprint-class bounds"
    assert np.any((cnt > 0) & (w == 1) & (hgt > BIN_BIG)), "a one-tile-wide column taller than 128 tiles"
    big = cnt[cnt > BIN_BIG]
    assert np.any(big % 32 != 0) and np.any(big % 16 != 0) and len(big) > 20
    p = fresh()
    try:
        hd = p.add_cloud(cloud)
        img = p.render_view(hd, s, view)
        check_frame(p, oracle, cloud, s, view, img, f"footprint classes, sync, large queue {len(big)}")
        out = np.empty_like(img)
        p.render_view(hd, s, view, out=out, asynchronous=True)
        assert p.sync()
        assert np.array_equal(out, img), "footprint classes, queued"
        hd.destroy()
    finally:
        p.destroy()


def big_queue_scene(k, seed):
    """k splats of several hundred tiles each (a 1920x1088 view) over 20 000 one-tile splats."""
    view = front_view(1920, 1088)
    rng = np.random.default_rng(seed)
    small = sort_scene(20_000 + SIDE_N, 20_000, attribute_planes(20_000 + SIDE_N, seed), seed=seed, front=view)
    pos = np.ones((k, 4), np.float32)
    pos[:, :3] = tile_centred(view, k, rng, 5.0, 9.0)
    so = np.stack([rng.uniform(0.6, 0.8, k), rng.uniform(0.6, 0.8, k), rng.uniform(0.1, 0.3, k), rng.uniform(0.2, 0.8, k)], 1)
    big = B.PlanarGaussian3d(pos, rng.uniform(-1, 1, (k, 48)).astype(np.float32), rng.uniform(-1, 1, (k, 4)).astype(np.float32),
                             so.astype(np.float32))
    return concat(small, big), view


@pytest.mark.gpu
@pytest.mark.parametrize("k", BIG_QUEUE_TARGETS, ids=[f"big{k}" for k in BIG_QUEUE_TARGETS])
def test_large_footprint_queue_parts_vs_oracle(oracle, sm_count, k):
    """The large-footprint queue with 1, 50, 300 and thousands of splats, synchronously (4 CTAs per SM) and queued
    (1 CTA per SM): part_shift from 4 down to 0 under both grids; queued frames equal the synchronous ones byte for
    byte, and the last one's tiles equal the oracle's."""
    cloud, view = big_queue_scene(k, 40 + k)
    s = B.CloudSettings()
    _, cnt = projected_tile_counts(oracle, cloud, view, s)
    nbig = int((cnt > BIN_BIG).sum())
    # (a splat centred in a border tile is clipped to the viewport: a few of the larger sets drop below 129 tiles)
    assert nbig == k if k <= 50 else abs(nbig - k) <= k // 100, f"the construction must put {k} splats in the large queue, not {nbig}"
    shifts = {q: part_shift(nbig, sm_count * (BIN_CTAS_PER_SM_QUEUED if q else BIN_CTAS_PER_SM)) for q in (False, True)}
    what = f"large queue {nbig}: part_shift {shifts[False]} (sync), {shifts[True]} (queued)"
    p = fresh()
    try:
        hd = p.add_cloud(cloud)
        img = p.render_view(hd, s, view)
        check_frame(p, oracle, cloud, s, view, img, what + ", sync")
        outs = [np.empty_like(img) for _ in range(2)]
        for o in outs:
            p.render_view(hd, s, view, out=o, asynchronous=True)
        assert p.sync(), what
        for o in outs:
            assert np.array_equal(o, img), what + ", queued"
        check_frame(p, oracle, cloud, s, view, outs[-1], what + ", queued")
        hd.destroy()
    finally:
        p.destroy()


@pytest.mark.gpu
def test_queued_match_any_pair_sort_vs_oracle(oracle, sm_count):
    """A queued frame of > 3.7 M pairs sorts them with <16, MATCH.ANY> on one CTA per SM (a synchronous frame sized the
    pair buffer and set the hint first)."""
    cloud = mixed_cloud(400_000, 61, 0.02, 0.1)
    view = front_view(1920, 1088)
    s = B.CloudSettings()
    p = fresh()
    try:
        hd = p.add_cloud(cloud)
        ref = p.render_view(hd, s, view)
        fs = p.frame_stats()
        assert fs.rounds == 1 and fs.n_pairs > 3_700_000, (fs.n_pairs, fs.rounds)
        m = ContextMirror(sm_count)
        m.frame(len(cloud), fs.n_visible, fs.n_pairs, fs.tiles_x * fs.tiles_y)
        f = m.frame(len(cloud), fs.n_visible, fs.n_pairs, fs.tiles_x * fs.tiles_y, queued=True)
        what = f"queued, {fs.n_pairs} pairs: pair sort {f['pair']}"
        assert f["pair"].variant == "<16,MATCH.ANY>", what
        out = np.empty_like(ref)
        p.render_view(hd, s, view, out=out, asynchronous=True)
        assert p.sync(), what
        assert np.array_equal(out, ref), what
        check_frame(p, oracle, cloud, s, view, out, what)
        hd.destroy()
    finally:
        p.destroy()


# ---------------------------------------------------------------------------------------------------------------------
# D. the two blend kernels give the same bytes
# ---------------------------------------------------------------------------------------------------------------------
def srgb_enc(c):
    c = np.clip(c, 0, 1)
    return np.where(c <= 0.0031308, 12.92 * c, 1.055 * np.power(c, 1 / 2.4) - 0.055)


def srgb_dec(c):
    return np.where(c <= 0.04045, c / 12.92, np.power((c + 0.055) / 1.055, 2.4))


def close_to(got, want, fmt, what):
    """`want`: the oracle's f32 frame.  rgba32f within PIXEL_TOL; rgba16f within PIXEL_TOL plus its own rounding; rgba8:
    the sRGB encoding of the oracle within half a step (+ the 1e-3 scaled to the encoding: never reached)."""
    if fmt == "rgba32f":
        err = float(np.abs(got - want).max())
        assert err <= PIXEL_TOL, f"{what}: L-inf {err}"
    elif fmt == "rgba16f":
        err = np.abs(got.astype(np.float32) - want) - np.abs(want) * 2.0 ** -11
        assert float(err.max()) <= PIXEL_TOL, f"{what}: L-inf {float(err.max())}"
    else:
        enc = np.concatenate([srgb_enc(want[..., :3]), np.clip(want[..., 3:4], 0, 1)], 2) * 255.0
        err = float(np.abs(got.astype(np.float32) - enc).max())
        assert err <= 0.51, f"{what}: {err} steps"


@pytest.mark.gpu
@pytest.mark.parametrize("gm", [B.GaussianMode.Gaussian3d, B.GaussianMode.Gaussian2d], ids=["3dgs-obb", "2dgs-obb"])
def test_blend_variants_identical_vs_oracle(oracle, gm):
    """After a small-footprint frame the blend runs raster_kernel<0>, after a large-footprint one (>= 8 pairs per
    visible splat) raster2_kernel: the same frame must come out byte for byte the same, in every format and output mode."""
    view = B.orbit_view(1, 8, 384, 224)
    s = B.CloudSettings(global_scale=0.2, gaussian_mode=gm)
    cloud = B.random_gaussians_3d_seeded(20000, 31)
    small_s = B.CloudSettings(global_scale=1.0, gaussian_mode=gm)
    small_c = sort_scene(2000 + SIDE_N, 2000, attribute_planes(2000 + SIDE_N, 32), seed=32, front=front_view(384, 224))
    large_s = B.CloudSettings(global_scale=1.0, gaussian_mode=gm)
    large_c = B.random_gaussians_3d_seeded(3000, 33)
    u = B.GaussianSplattingPlugin.cloud_uniform(s)
    tiles_img = oracle.render_tiles(cloud, view.to_abi(), u, s.to_abi())["image"]
    layer_img = oracle.render_ref(cloud, view.to_abi(), u, s.to_abi(), dst=np.zeros_like(tiles_img))
    p = fresh()
    try:
        hc, hs, hl = p.add_cloud(cloud), p.add_cloud(small_c), p.add_cloud(large_c)
        ratios = {}
        for name, hp, sp in (("small", hs, small_s), ("large", hl, large_s)):
            p.render_view(hp, sp, view, to_host=False)
            fs = p.frame_stats()
            ratios[name] = fs.n_pairs / max(fs.n_visible, 1)
        assert ratios["small"] < 8 <= ratios["large"], ratios
        for fmt in ("rgba32f", "rgba16f", "rgba8_srgb"):
            for mode in ("opaque", "premultiplied"):
                got = {}
                for name, hp, sp in (("small", hs, small_s), ("large", hl, large_s)):
                    p.render_view(hp, sp, view, to_host=False)
                    kernel = "raster2_kernel" if name == "large" else "raster_kernel<0>"
                    got[name] = p.render_view(hc, s, view, fmt=fmt, premultiplied=mode == "premultiplied")
                    close_to(got[name], tiles_img if mode == "opaque" else layer_img, fmt, f"{gm.name} {fmt} {mode} via {kernel}")
                assert np.array_equal(got["small"].view(np.uint8), got["large"].view(np.uint8)), \
                    f"{gm.name} {fmt} {mode}: raster_kernel<0> and raster2_kernel differ"
            # blend-over: the target layer is itself the primer (small or large footprints)
            for name, hp, sp in (("small", hs, small_s), ("large", hl, large_s)):
                kernel = "raster2_kernel" if name == "large" else "raster_kernel<0>"
                held = p.render_view(hp, sp, view, fmt=fmt, premultiplied=True)
                got = p.render_view(hc, s, view, fmt=fmt, blend_over=True).astype(np.float32)
                what = f"{gm.name} {fmt} blend-over via {kernel}"
                if fmt == "rgba8_srgb":
                    h8 = held.astype(np.float32) / 255.0
                    dst = np.concatenate([srgb_dec(h8[..., :3]), h8[..., 3:4]], axis=2).astype(np.float32)
                    want = oracle.render_ref(cloud, view.to_abi(), u, s.to_abi(), dst=dst)
                    want = np.concatenate([srgb_enc(want[..., :3]), np.clip(want[..., 3:4], 0, 1)], axis=2)
                    assert np.abs(got / 255.0 - want).max() <= 1.01 / 255.0, what
                else:
                    want = oracle.render_ref(cloud, view.to_abi(), u, s.to_abi(), dst=held.astype(np.float32))
                    tol = PIXEL_TOL if fmt == "rgba32f" else 4e-3 * max(1.0, float(np.abs(want).max()))
                    assert np.abs(got - want).max() <= tol, what
        for hh in (hc, hs, hl):
            hh.destroy()
    finally:
        p.destroy()


# ---------------------------------------------------------------------------------------------------------------------
# E. the benchmark's regime at full size: C3, three contexts, queued frames, a different view per frame
# ---------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def c3_cloud():
    return B.random_gaussians_3d_seeded(6_000_000, 0)


@pytest.mark.gpu
def test_c3_queued_round_robin_distinct_views_vs_oracle(oracle, c3_cloud, sm_count):
    """bench.py's regime (C3: 6 M f16, 1920x1080, global_scale 0.02; three contexts sharing one cloud, frames queued
    round-robin to host memory) with a DIFFERENT view for every frame, so a mix-up of frame slot, toggle or copy event
    cannot hide behind identical frames: every host frame equals the synchronous render of its view, each context's
    last frame matches the oracle, and a heavier second frame that outgrows the pair buffer while the first is in
    flight is reported and re-rendered exactly."""
    views = [B.orbit_view(i, 9, 1920, 1080) for i in range(9)]
    s = B.CloudSettings(global_scale=0.02)
    oc = c3_cloud.rounded_to_f16()
    ctxs = [fresh() for _ in range(3)]
    ref_ctx = fresh()
    try:
        h = ctxs[0].add_cloud(c3_cloud, f16=True)
        for c in ctxs:
            c.render_view(h, s, views[0], fmt="rgba8_srgb", to_host=False)        # sizes buffers, sets the hints
        outs = [np.empty((1080, 1920, 4), np.uint8) for _ in views]
        for i, v in enumerate(views):
            ctxs[i % 3].render_view(h, s, v, fmt="rgba8_srgb", out=outs[i], asynchronous=True)
        for c in ctxs:
            assert c.sync()
        for k, c in enumerate(ctxs):
            i = 6 + k                                   # the context's last frame
            fs = c.frame_stats()
            m = ContextMirror(sm_count)
            m.frame(fs.n, fs.n_visible, fs.n_pairs, fs.tiles_x * fs.tiles_y)
            f = m.frame(fs.n, fs.n_visible, fs.n_pairs, fs.tiles_x * fs.tiles_y, queued=True)
            check_frame(c, oracle, oc, s, views[i], None, f"C3 context {k}, queued view {i}: depth sort {f['depth']}, "
                        f"pair sort {f['pair']}", pixels=False)
        firsts = []
        for i, v in enumerate(views):
            want = ref_ctx.render_view(h, s, v, fmt="rgba8_srgb")
            firsts.append(want)
            assert np.array_equal(outs[i], want), f"queued frame {i} (context {i % 3}) differs from the synchronous render"
        assert len({f.tobytes() for f in firsts}) == len(views)
        # a heavier second frame: outgrows the pair buffer while the first is still in flight
        heavy = B.CloudSettings(global_scale=0.1)
        c = ctxs[1]
        want_heavy = ref_ctx.render_view(h, heavy, views[4], fmt="rgba8_srgb")
        needed = ref_ctx.frame_stats().n_pairs
        assert ref_ctx.frame_stats().rounds == 1 and needed > len(c3_cloud), "the heavy frame must outgrow the 6 M-pair buffer"
        light_out, heavy_out = np.empty_like(outs[0]), np.empty_like(outs[0])
        c.render_view(h, s, views[3], fmt="rgba8_srgb", out=light_out, asynchronous=True)
        c.render_view(h, heavy, views[4], fmt="rgba8_srgb", out=heavy_out, asynchronous=True)
        assert not c.sync(), "the heavy frame overflowed the pair buffer: bgs_sync must say so"
        c.render_view(h, s, views[3], fmt="rgba8_srgb", out=light_out, asynchronous=True)
        c.render_view(h, heavy, views[4], fmt="rgba8_srgb", out=heavy_out, asynchronous=True)
        assert c.sync()
        assert np.array_equal(light_out, firsts[3]) and np.array_equal(heavy_out, want_heavy)
        h.destroy()
    finally:
        for c in ctxs + [ref_ctx]:
            c.destroy()


# ---------------------------------------------------------------------------------------------------------------------
# F. BGS_LAYOUT=planar: the reference's planes, no gaussian-major repack
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("f16", [False, True], ids=["f32", "f16"])
def test_planar_layout_identical_vs_oracle(oracle, monkeypatch, f16):
    from test_gpu_parity import check_against_oracle

    cloud = B.random_gaussians_3d_seeded(30000, 51)
    view = B.orbit_view(2, 8, 416, 240)
    variants = [dict(), dict(aabb=True), dict(gaussian_mode=B.GaussianMode.Gaussian2d, aabb=True),
                dict(rasterize_mode=B.RasterizeMode.Depth)]
    p = fresh()
    try:
        blocked = p.add_cloud(cloud, f16=f16)
        monkeypatch.setenv("BGS_LAYOUT", "planar")
        planar = p.add_cloud(cloud, f16=f16)
        for kw in variants:
            s = B.CloudSettings(global_scale=0.15, **kw)
            for fmt in ("rgba32f", "rgba8_srgb"):
                a = p.render_view(blocked, s, view, fmt=fmt)
                b = p.render_view(planar, s, view, fmt=fmt)
                assert np.array_equal(a.view(np.uint8), b.view(np.uint8)), (kw, fmt)
        s = B.CloudSettings(global_scale=0.15)
        for a, b in zip(p.render_view_aux(blocked, s, view), p.render_view_aux(planar, s, view)):
            assert np.array_equal(a, b), "render_view_aux"
        blocked.destroy(); planar.destroy()
        check_against_oracle(p, oracle, cloud, s, view, f16=f16)          # uploads under BGS_LAYOUT=planar
        if f16:
            cov = B.random_gaussians_3d_seeded(20000, 52)
            cov.scale_opacity[:, :3] *= np.float32(0.15)
            check_against_oracle(p, oracle, cov, B.CloudSettings(), view, f16=True, cov=True)
            hp = p.add_cloud(cov, precompute_covariance=True)
            monkeypatch.delenv("BGS_LAYOUT")
            hb = p.add_cloud(cov, precompute_covariance=True)
            assert np.array_equal(p.render_view(hp, B.CloudSettings(), view), p.render_view(hb, B.CloudSettings(), view))
            hp.destroy(); hb.destroy()
    finally:
        p.destroy()
