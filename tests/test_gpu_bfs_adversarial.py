"""The BFS_3D wavefront kernels on adversarial grids (tests/bfs_mazes.py): one-cell corridors across tile seams and
through tile corners, mazes longer than a stepwise launch chunk, fronts meeting head-on, sealed pockets, and stacked
banks over a field whose slot faces are free.  Every path of run_grid (smplgpu.cu) is compared, int32 for int32, with
the CPU oracle's BFS_3D over the whole grid or every cell of every slot:

  single grid   TILES / AUTO: bfs_tiles_kernel<1> (< 4096 tiles), <4> (>= 4096 tiles); LEVELS: bfs_levels_kernel
  bank, sync    TILES: the cooperative tile kernel (<1> / <4>); LEVELS: the cooperative level kernel
  bank, async   TILES: one tile-kernel launch per super-step, queued in chunks (bfs_bank_run_done / _wait queue the
                rest); LEVELS: the cooperative level kernel on the bank stream
  environment   test_environment_variants re-runs the quick tests of this file in a child process under each switch
                that the library reads once per process: SMPLGPU_BANK_TILE_CHUNK (the continuation path in chunks of
                1 and 5 super-steps), SMPLGPU_BANK_COOPERATIVE (async tile runs as one cooperative launch),
                SMPLGPU_BANK_STEPWISE (async level runs one launch per level), SMPLGPU_BFS_TILE_RPT = 1 / 4 / 2 / 32
                (bfs_tiles_kernel<1>, <4>, <2> and bfs_warp_tiles_kernel whatever the grid size).
"""
import functools
import os
import re
import subprocess
import sys
import time

import numpy as np
import pytest

import bfs_mazes as M
from conftest import ROOT
from helpers import make_oracle
from oracle_api import OracleBfs
from smpl_b200 import api, scenes

pytestmark = pytest.mark.gpu
WALL = 0x7FFFFFFF
MODES = {"tiles": api.GpuContext.BFS_TILES, "levels": api.GpuContext.BFS_LEVELS, "auto": api.GpuContext.BFS_AUTO}
RES, DMAX_SQ = 0.02, 400          # the synthetic fields: d2 = 0 on walls, DMAX_SQ elsewhere
SMALL = {m.name: m for m in M.small_mazes()}


@pytest.fixture(scope="module")
def ctx():
    c = api.GpuContext(0)
    yield c
    c.close()


def oracle_grid(walls, seeds):
    """BFS_3D over walls[z, y, x] from seeds: the padded int32 grid.  Fresh walls per call."""
    nz, ny, nx = walls.shape
    b = OracleBfs(nx, ny, nz)
    b.set_walls(walls)
    if len(seeds) == 1:
        b.run(*seeds[0])
    else:
        b.run_multi(list(seeds) + [(0, 0, 0)])   # the reference's iterator drops the last triple: a sentinel
    return b.grid()


@functools.lru_cache(maxsize=None)
def large_maze():
    m = M.large()
    return m, oracle_grid(m.walls, m.seeds)


@functools.lru_cache(maxsize=None)
def small_oracle(name):
    m = SMALL[name]
    return oracle_grid(m.walls, m.seeds)


def assert_same(got, want, what, padded=False):
    """Exact equality; on failure the first differing cell (x, y, z of the unpadded grid or slot), its tile and the
    tile kernel's super-step that should have found it."""
    if np.array_equal(got, want):
        return
    bad = np.argwhere(got != want)
    first = tuple(int(v) for v in bad[0])
    z, y, x = (v - 1 if padded else v for v in first[-3:])
    slot = "slot %d, " % first[0] if len(first) == 4 else ""
    w, g = int(want[first]), int(got[first])
    raise AssertionError("%s: %d cells differ; first at %s(x, y, z) = (%d, %d, %d), tile %s of its grid: got %d, want %d "
                         "(super-step %s)" % (what, len(bad), slot, x, y, z, M.tile_of(x, y, z), g, w,
                                              w // 8 if 0 <= w < WALL else "-"))


def max_distance(grid):
    return int(grid[(grid >= 0) & (grid != WALL)].max())


# ---- single grids ----

def run_single(ctx, maze, mode):
    ctx.bfs_set_mode(MODES[mode])
    try:
        ctx.bfs_set_walls(maze.walls)
        assert ctx.bfs_run(maze.seeds) == len(maze.seeds)
        return ctx.bfs_download(), ctx.bfs_last_levels()
    finally:
        ctx.bfs_set_mode(ctx.BFS_AUTO)


@pytest.mark.parametrize("name", list(SMALL))
@pytest.mark.parametrize("mode", list(MODES))
def test_single_grid_mazes(ctx, mode, name):
    m = SMALL[name]
    nx, ny, nz = m.dims
    assert M.n_tiles(nx, ny, nz) < 4096                       # bfs_tiles_kernel<1> unless a size is forced
    got, levels = run_single(ctx, m, mode)
    want = small_oracle(name)
    assert_same(got, want, "%s, %s" % (name, mode), padded=True)
    assert levels >= max_distance(want)


@pytest.mark.parametrize("mode", list(MODES))
def test_single_grid_large(ctx, mode):
    m, want = large_maze()
    assert M.n_tiles(*m.dims) >= 4096                         # bfs_tiles_kernel<4> unless a size is forced
    got, levels = run_single(ctx, m, mode)
    assert_same(got, want, "%s, %s" % (m.name, mode), padded=True)
    assert levels >= max_distance(want)


# ---- stacked banks over a field with free faces ----

def set_field(ctx, walls):
    ctx.set_distance_field(M.field_from_walls(walls, DMAX_SQ), (0.0, 0.0, 0.0), RES, DMAX_SQ)


def create_bank(ctx, walls, n_slots):
    """inflation radius 0: only the d2 = 0 cells are walls, so the grid faces can be free"""
    assert ctx.bfs_bank_create(n_slots, 0.0) == int((walls != 0).sum())


def bank_read(ctx, walls, n_slots, chunk_cells=1 << 22):
    """Every cell of every slot: [slot, z, y, x] through bfs_bank_distances."""
    nz, ny, nx = walls.shape
    cells = np.argwhere(np.ones((nz, ny, nx), bool))[:, ::-1].astype(np.int32)     # (x, y, z), z-major like [z, y, x]
    per = max(1, chunk_cells // len(cells))
    out = np.empty((n_slots, nz, ny, nx), np.int32)
    for s0 in range(0, n_slots, per):
        k = min(per, n_slots - s0)
        sl = np.repeat(np.arange(s0, s0 + k, dtype=np.int32), len(cells))
        out[s0:s0 + k] = ctx.bfs_bank_distances(sl, np.tile(cells, (k, 1))).reshape(k, nz, ny, nx)
    return out


def bank_run(ctx, how, slots, seeds):
    if how == "sync":
        assert ctx.bfs_bank_run_slots(slots, seeds) == len(slots)
    else:
        assert ctx.bfs_bank_run_slots_async(slots, seeds) == len(slots)
        ctx.bfs_bank_run_wait()


def bank_paths():
    return [(k, h) for k in ("tiles", "levels") for h in ("sync", "async")]


def slots_for_large(nx, ny, nz):
    """The fewest slots whose stacked bank has >= 4096 tiles."""
    n = 1
    while M.n_tiles(nx, ny, n * (nz + 2) - 2) < 4096:
        n += 1
    return n


# nz = 14: slot_dz = 16, slot boundaries on the z seams; 13, 29, 45: inside tiles at different offsets
BANKS = [(14, "small"), (13, "small"), (29, "small"), (45, "small"), (14, "large"), (13, "large")]


@pytest.mark.parametrize("nz,size", BANKS, ids=["nz%d-%s" % b for b in BANKS])
@pytest.mark.parametrize("kind,how", bank_paths(), ids=["%s-%s" % p for p in bank_paths()])
def test_bank_open_faces(ctx, kind, how, nz, size):
    nx, ny = (40, 20) if size == "small" else (30, 14)
    w = M.open_face_walls(nx, ny, nz)
    n = 6 if size == "small" else slots_for_large(nx, ny, nz)
    assert (M.n_tiles(nx, ny, n * (nz + 2) - 2) >= 4096) == (size == "large")
    seeds = M.top_face_seeds(w, 6)
    want = np.stack([oracle_grid(w, [s])[1:-1, 1:-1, 1:-1] for s in seeds])
    set_field(ctx, w)
    ctx.bfs_set_mode(MODES[kind])
    try:
        create_bank(ctx, w, n)
        # every slot, seeded on its top face at one of six places
        first = np.arange(n) % 6
        bank_run(ctx, how, np.arange(n), [seeds[i] for i in first])
        got = bank_read(ctx, w, n)
        assert_same(got, want[first], "bank %s %s nz %d, %d slots" % (kind, how, nz, n))
        # a third of the slots again from other seeds; the others keep their distances
        sub = np.arange(1, n, 3)
        again = (sub + 1) % 6
        bank_run(ctx, how, sub, [seeds[i] for i in again])
        expect = got.copy()
        expect[sub] = want[again]
        assert_same(bank_read(ctx, w, n), expect, "bank %s %s nz %d, slots re-run" % (kind, how, nz))
    finally:
        ctx.bfs_set_mode(ctx.BFS_AUTO)


@pytest.mark.parametrize("finish", ["wait", "poll"])
@pytest.mark.parametrize("kind", ["tiles", "levels"])
def test_bank_serpentine_continuation(ctx, kind, finish):
    """A ~2 000-level maze in every slot: the stepwise runs span many launch chunks.  bfs_bank_run_done() may only
    report a run complete once its last chunk has run, so distances read right after it returns 1 are final."""
    nx, ny, nz = 64, 64, 4
    path = M.serpentine_cells(nx, ny, nz - 1)
    w = M.solid(nx, ny, nz)
    M.carve(w, path)
    seeds = [path[0], path[len(path) // 3], path[-1], path[len(path) // 2]]
    want = np.stack([oracle_grid(w, [s])[1:-1, 1:-1, 1:-1] for s in seeds])
    assert max_distance(want) >= 1500
    set_field(ctx, w)
    ctx.bfs_set_mode(MODES[kind])
    try:
        create_bank(ctx, w, 4)
        assert ctx.bfs_bank_run_slots_async(np.arange(4), seeds) == 4
        if finish == "wait":
            ctx.bfs_bank_run_wait()
        else:
            t0 = time.time()
            while not ctx.bfs_bank_run_done():
                assert time.time() - t0 < 60.0, "bank run not done after 60 s"
        assert_same(bank_read(ctx, w, 4), want, "serpentine bank %s, %s" % (kind, finish))
    finally:
        ctx.bfs_set_mode(ctx.BFS_AUTO)


@pytest.mark.parametrize("kind", ["tiles", "levels"])
def test_bank_refill_async(ctx, kind):
    """Slots 1 and 3 refilled asynchronously from new seeds; slots 0 and 2 keep the distances of the run before."""
    nx, ny, nz = 40, 20, 13
    w = M.open_face_walls(nx, ny, nz)
    seeds = M.top_face_seeds(w, 6)
    want = np.stack([oracle_grid(w, [s])[1:-1, 1:-1, 1:-1] for s in seeds])
    set_field(ctx, w)
    ctx.bfs_set_mode(MODES[kind])
    try:
        create_bank(ctx, w, 4)
        assert ctx.bfs_bank_run_slots(np.arange(4), seeds[:4]) == 4
        assert_same(bank_read(ctx, w, 4), want[:4], "bank %s before the refill" % kind)
        assert ctx.bfs_bank_run_slots_async([1, 3], [seeds[4], seeds[5]]) == 2
        t0 = time.time()
        while not ctx.bfs_bank_run_done():
            assert time.time() - t0 < 60.0
        assert_same(bank_read(ctx, w, 4), want[[0, 4, 2, 5]], "bank %s after refilling slots 1 and 3" % kind)
    finally:
        ctx.bfs_set_mode(ctx.BFS_AUTO)


@pytest.mark.parametrize("wait", [True, False], ids=["sync", "async"])
@pytest.mark.parametrize("kind", ["tiles", "levels"])
def test_bank_goal_sets(ctx, kind, wait):
    """bfs_bank_run_slots_multi: up to SMPLGPU_MAX_GOAL_SET seeds per slot, some out of bounds, some on walls (a seed on
    a wall frees it for that run only), one empty set; each slot equals the oracle's multi-seed run on fresh walls."""
    nx, ny, nz = 40, 20, 13
    w = M.open_face_walls(nx, ny, nz)
    rng = np.random.default_rng(41)
    free = np.argwhere(w == 0)[:, ::-1]
    wall = np.argwhere(w != 0)[:, ::-1]

    def goal_set(k, n_wall, n_out):
        s = [free[i] for i in rng.choice(len(free), k - n_wall - n_out, replace=False)]
        s += [wall[i] for i in rng.choice(len(wall), n_wall, replace=False)]
        s += [(-1, 3, 3), (nx, 0, 0), (0, ny, 2), (1, 1, nz), (0, -5, 0)][:n_out]
        s = np.array(s, np.int32).reshape(-1, 3)
        return s[rng.permutation(len(s))]

    set_field(ctx, w)
    ctx.bfs_set_mode(MODES[kind])
    try:
        create_bank(ctx, w, 5)
        for round_ in range(2):
            sets = [goal_set(api.MAX_GOAL_SET, 6, 5), goal_set(1, 0, 0), np.zeros((0, 3), np.int32),
                    goal_set(20, 3, 2), goal_set(api.MAX_GOAL_SET, 0, 0)]
            order = np.array([3, 0, 4, 1, 2]) if round_ else np.arange(5)
            slots = np.arange(5)[order]
            sets = [sets[i] for i in order]
            n_in = ctx.bfs_bank_run_slots_multi(slots, sets, wait=wait)
            if wait:
                assert n_in == sum(int(((s >= 0) & (s < (nx, ny, nz))).all(axis=1).sum()) for s in sets)
            else:
                assert n_in == 5
                ctx.bfs_bank_run_wait()
            got = bank_read(ctx, w, 5)
            for sl, s in zip(slots, sets):
                b = OracleBfs(nx, ny, nz)
                b.set_walls(w)
                b.run_multi([tuple(c) for c in s] + [(0, 0, 0)])
                assert_same(got[sl], b.grid()[1:-1, 1:-1, 1:-1], "goal sets %s round %d slot %d" % (kind, round_, sl))
    finally:
        ctx.bfs_set_mode(ctx.BFS_AUTO)


# ---- the wall threshold at its boundaries ----

def test_wall_threshold_boundaries(ctx):
    """Walls are cells with res * sqrt(d2) <= radius (the reference's m_sqrt_table[d2] <= radius).  For every k up to
    dmax_sq, at radius exactly res * sqrt(k) (cells with d2 = k are walls) and at the next double below (they are
    not), the single grid and the bank count the walls the oracle counts; the walls themselves are compared at some."""
    scene = scenes.pr2_tabletop_scene()
    o = make_oracle(scene, with_kdl=False)
    dims, origin, res, dmax_sq = o.grid_info()
    d2 = o.df_d2()
    ctx.set_distance_field(d2.astype(np.uint16), origin, res, dmax_sq)
    # the reference's rule, restated: count(radius) = #cells with table[d2] <= radius, table[k] = res * sqrt(k)
    table = res * np.sqrt(np.arange(dmax_sq + 1, dtype=np.float64))
    cum = np.cumsum(np.bincount(d2.ravel(), minlength=dmax_sq + 1))

    def count(r):
        i = int(np.searchsorted(table, r, side="right")) - 1
        return int(cum[i]) if i >= 0 else 0

    present = np.unique(d2)
    anchors = set(present[:16].tolist()) | {int(present[len(present) // 2]), int(present[-1]), dmax_sq}
    for k in range(dmax_sq + 1):
        for r in (table[k], np.nextafter(table[k], -np.inf)):
            want = count(r)
            if k in anchors:
                assert o.heur_init(r, scene.cost_per_cell) == want, (k, r)
            assert ctx.bfs_set_walls_from_df(r) == want, (k, r)
            assert ctx.bfs_bank_create(1, r) == want, (k, r)
    # the walls themselves: a run without seeds leaves WALL on walls and -1 elsewhere
    nx, ny, nz = (int(v) for v in dims)
    for k in (1, 2, int(present[17])):
        for r in (table[k], np.nextafter(table[k], -np.inf)):
            o.heur_init(r, scene.cost_per_cell)
            want = o.heur_grid() == WALL
            ctx.bfs_set_walls_from_df(r)
            assert ctx.bfs_run(np.zeros((0, 3), np.int32)) == 0
            assert np.array_equal(ctx.bfs_download() == WALL, want), (k, r)
            ctx.bfs_bank_create(1, r)
            assert ctx.bfs_bank_run_slots([0], [(-1, 0, 0)]) == 0
            cells = np.argwhere(np.ones((nz, ny, nx), bool))[:, ::-1].astype(np.int32)
            bank = ctx.bfs_bank_distances(np.zeros(len(cells), np.int32), cells).reshape(nz, ny, nx)
            assert np.array_equal(bank == WALL, want[1:-1, 1:-1, 1:-1]), (k, r)
    o.close()


# ---- the switches the library reads once per process, in child processes ----

QUICK = "single_grid_mazes or bank_serpentine or (bank_open_faces and small) or bank_refill or bank_goal_sets"
VARIANTS = [
    {"SMPLGPU_BANK_TILE_CHUNK": "1"},
    {"SMPLGPU_BANK_TILE_CHUNK": "5"},
    {"SMPLGPU_BANK_COOPERATIVE": "1"},
    {"SMPLGPU_BFS_MODE": "1", "SMPLGPU_BANK_STEPWISE": "1"},
    {"SMPLGPU_BFS_TILE_RPT": "1"},
    {"SMPLGPU_BFS_TILE_RPT": "4"},
    {"SMPLGPU_BFS_TILE_RPT": "2"},
    {"SMPLGPU_BFS_TILE_RPT": "32"},
]


@pytest.mark.parametrize("env", VARIANTS, ids=[",".join("%s=%s" % kv for kv in v.items()) for v in VARIANTS])
def test_environment_variants(env):
    e = dict(os.environ)
    e.update(env)
    cmd = [sys.executable, "-m", "pytest", os.path.abspath(__file__), "-m", "gpu", "-k", QUICK, "-q", "-x",
           "-p", "no:cacheprovider"]
    t0 = time.time()
    r = subprocess.run(cmd, cwd=ROOT, env=e, capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, "%s\n%s\n%s" % (env, r.stdout[-6000:], r.stderr[-3000:])
    summary = r.stdout.strip().splitlines()[-1]
    ran = re.match(r"(\d+) passed", summary)
    assert ran and int(ran.group(1)) >= 50 and "skipped" not in summary, summary   # the quick tests ran, all of them
    print("%s: %.1f s, %s" % (env, time.time() - t0, summary))
