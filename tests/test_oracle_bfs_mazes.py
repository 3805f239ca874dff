"""The adversarial BFS grids (tests/bfs_mazes.py) do what they claim, checked with the CPU oracle's BFS_3D: a GPU test
on them cannot pass because its grid turned out trivial.  No GPU needed."""
import numpy as np
import pytest

import bfs_mazes as M
from oracle_api import OracleBfs

WALL = 0x7FFFFFFF


def oracle(maze):
    nx, ny, nz = maze.dims
    b = OracleBfs(nx, ny, nz)
    b.set_walls(maze.walls)
    if len(maze.seeds) == 1:
        b.run(*maze.seeds[0])
    else:
        b.run_multi(list(maze.seeds) + [(0, 0, 0)])   # the reference's iterator drops the last triple: a sentinel
    return b.grid()


def at(grid, c):
    return int(grid[c[2] + 1, c[1] + 1, c[0] + 1])


def check_claims(maze):
    g = oracle(maze)
    got = [at(g, c) for c, _ in maze.expect]
    want = [d for _, d in maze.expect]
    assert got == want, maze.name
    assert all(at(g, c) == -1 for c in maze.pockets), maze.name
    for s in maze.seeds:
        assert at(g, s) == 0
    return g


@pytest.mark.parametrize("signs", M.SIGNS, ids=["%+d%+d%+d" % s for s in M.SIGNS])
def test_staircase_is_one_cell_per_level_through_a_tile_corner(signs):
    m = M.staircase(signs)
    g = check_claims(m)
    a, b = m.corner
    ta, tb = np.array(M.tile_of(*a)), np.array(M.tile_of(*b))
    # one unit step that changes the tile on all three axes: it passes through the corner where the three seams meet,
    # into the diagonal neighbour tile
    assert np.abs(np.array(b) - np.array(a)).tolist() == [1, 1, 1]
    assert (tb - ta).tolist() == list(signs)
    assert {a[0], b[0]} == {62, 63} and {a[1], b[1]} == {a[2], b[2]} == {30, 31}
    assert len(m.expect) == int((m.walls == 0).sum())          # nothing but the path is free
    # one cell per level: every level 0 .. max holds exactly one cell
    d = g[(g >= 0) & (g != WALL)]
    assert np.array_equal(np.sort(d), np.arange(len(m.expect)))


def test_axis_corridors_cross_seams_and_come_back():
    m = M.axis_corridors()
    g = check_claims(m)
    tiles_x = {M.tile_of(x, 18, 18)[0] for x in range(96)}
    assert tiles_x == {0, 1, 2, 3}
    # the main corridor re-enters tiles of its first leg, many levels after it left them
    for x in (94, 20):
        t_first = M.tile_of(x, 18, 18)
        assert M.tile_of(x, 22, 24) == t_first
        assert at(g, (x, 22, 24)) - at(g, (x, 18, 18)) > 3 * 8
    assert len(m.pockets) > 30


def test_serpentine_spans_eight_stepwise_chunks():
    m = M.serpentine()
    g = check_claims(m)
    free = m.walls == 0
    d = g[1:-1, 1:-1, 1:-1][free]
    assert (d >= 0).all() and d.max() >= 1500 and d.max() > 8 * 24 * 8   # > 8 chunks of 24 super-steps of 8 levels


def test_head_on_fronts_have_equidistant_cells():
    m = M.head_on()
    g = check_claims(m)
    assert len(m.seeds) >= 4
    # equidistant cells in the middle of a tile and a pair straddling each seam
    assert at(g, (47, 5, 5)) == 31 and M.tile_of(46, 5, 5) == M.tile_of(48, 5, 5)
    assert at(g, (30, 10, 5)) == at(g, (31, 10, 5)) == 19 and M.tile_of(30, 10, 5)[0] + 1 == M.tile_of(31, 10, 5)[0]
    assert at(g, (104, 14, 10)) == at(g, (104, 15, 10))
    assert at(g, (64, 20, 14)) == at(g, (64, 20, 15))


def test_large_grid_has_4096_tiles_and_stays_cheap():
    m = M.large()
    nx, ny, nz = m.dims
    assert M.n_tiles(nx, ny, nz) >= 4096
    assert (m.walls == 0).mean() < 0.001
    g = check_claims(m)
    a, b = m.corner
    assert np.abs(np.array(M.tile_of(*a)) - np.array(M.tile_of(*b))).tolist() == [1, 1, 1]
    assert int(g[(g != WALL)].max()) > 800


@pytest.mark.parametrize("nz", [13, 14, 29, 45])
def test_open_face_field_reaches_both_faces(nz):
    nx, ny = 40, 20
    w = M.open_face_walls(nx, ny, nz)
    seeds = M.top_face_seeds(w, 6)
    assert len(set(seeds)) == 6
    for s in seeds:
        b = OracleBfs(nx, ny, nz)
        b.set_walls(w)
        b.run(*s)
        g = b.grid()[1:-1, 1:-1, 1:-1]
        for z in (0, nz - 1):                                   # free cells on both faces, all of them reached
            face = g[z][w[z] == 0]
            assert len(face) > 20 and (face >= 0).all()
    f = M.field_from_walls(w, 400)
    assert f.shape == (nx, ny, nz) and int((f == 0).sum()) == int(w.sum())
    assert np.array_equal(f.transpose(2, 1, 0) == 0, w != 0)
