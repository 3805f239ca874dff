"""Adversarial grids for the BFS_3D wavefront kernels: one-cell corridors that cross the tile seams, mazes longer than
a stepwise launch chunk, fronts that meet head-on, sealed pockets, and fields with free faces for the stacked banks.

Coordinates follow the device layout (smpl_b200/csrc/bfs_tiles.cuh): padded cell = cell + 1, a tile is 32 padded
cells in x and 16 in y and z.  In unpadded coordinates the first cell of a tile is therefore at x = 31 (mod 32) and
y, z = 15 (mod 16); `tile_of` maps a cell to its tile.

Every generator returns a Maze: walls[z, y, x] (uint8, nonzero = wall), the seeds (x, y, z), and what the grid claims
about itself -- `expect` (cells with their exact BFS distance), `pockets` (free cells that no seed reaches), `corner`
(the pair of path cells that step diagonally across a 3-D tile corner).  tests/test_oracle_bfs_mazes.py checks those
claims against the CPU oracle, so a GPU test cannot pass on a grid that is easier than it looks.
"""
from dataclasses import dataclass, field
import itertools

import numpy as np

TILE_X, TILE_YZ = 32, 16
SIGNS = list(itertools.product((1, -1), repeat=3))


@dataclass
class Maze:
    name: str
    walls: np.ndarray                                  # [nz, ny, nx] uint8
    seeds: list                                        # [(x, y, z)]
    expect: list = field(default_factory=list)         # [((x, y, z), distance)]
    pockets: list = field(default_factory=list)        # [(x, y, z)] free, unreachable
    corner: tuple = None                               # (cell before, cell after) crossing a tile corner

    @property
    def dims(self):
        nz, ny, nx = self.walls.shape
        return nx, ny, nz


def tile_of(x, y, z):
    """(tx, ty, tz) of an unpadded cell."""
    return (x + 1) // TILE_X, (y + 1) // TILE_YZ, (z + 1) // TILE_YZ


def n_tiles(nx, ny, nz):
    """Tiles of the padded grid: ceil((nx+2)/32) * ceil((ny+2)/16) * ceil((nz+2)/16)."""
    return -(-(nx + 2) // TILE_X) * (-(-(ny + 2) // TILE_YZ)) * (-(-(nz + 2) // TILE_YZ))


def solid(nx, ny, nz):
    return np.ones((nz, ny, nx), np.uint8)


def carve(walls, cells):
    for x, y, z in cells:
        walls[z, y, x] = 0


def polyline(points):
    """The cells of axis-aligned segments between consecutive points (each pair differs in one coordinate), in order."""
    out = [tuple(points[0])]
    for a, b in zip(points, points[1:]):
        axis = [i for i in range(3) if a[i] != b[i]]
        assert len(axis) == 1, (a, b)
        i = axis[0]
        step = 1 if b[i] > a[i] else -1
        for v in range(a[i] + step, b[i] + step, step):
            c = list(a)
            c[i] = v
            out.append(tuple(c))
    return out


def box(x0, x1, y0, y1, z0, z1):
    return [(x, y, z) for z in range(z0, z1 + 1) for y in range(y0, y1 + 1) for x in range(x0, x1 + 1)]


# ---- diagonal staircases ----

def staircase_cells(signs, corner, t_cross, length):
    """A 26-connected path p(t) = p0 + signs * t (t = 0 .. length-1) whose step t_cross -> t_cross + 1 goes from one tile
    into its diagonal neighbour through the 3-D tile corner at `corner` (the first cell of the upper tile on every
    axis): on an axis with sign +1 the path is at corner - 1 at t_cross, with sign -1 at corner."""
    p0 = [(c - 1 if s > 0 else c) - s * t_cross for c, s in zip(corner, signs)]
    return [tuple(p0[i] + signs[i] * t for i in range(3)) for t in range(length)]


def staircase(signs, corner=(63, 31, 31), t_cross=30, length=60, dims=(96, 64, 64)):
    """One-cell-wide diagonal staircase, walls everywhere else; seeded at t = 0, so the frontier is ONE cell per level
    and the distance of p(t) is exactly t (cells two steps apart differ by 2 on every axis: no short cuts)."""
    path = staircase_cells(signs, corner, t_cross, length)
    w = solid(*dims)
    carve(w, path)
    return Maze("staircase%+d%+d%+d" % tuple(signs), w, [path[0]], expect=[(c, t) for t, c in enumerate(path)],
                corner=(path[t_cross], path[t_cross + 1]))


# ---- axis corridors ----

def axis_corridors():
    """One-cell corridors along x, y and z across several tiles.  The main corridor runs +x through four tiles (the
    front moves TILE_K = 8 cells per super-step in x, the halo width), turns at the x seam into +y, at the y seam into +z,
    comes back -y and then -x through the tiles of its first leg -- re-entering tiles it left 4 and 15 super-steps
    earlier -- and ends in a +z run across two z seams.  Two straight corridors along y and z have seeds of their own.
    Free pockets lie two cells (one wall) away from the corridors, across seams too."""
    nx, ny, nz = 160, 48, 48
    w = solid(nx, ny, nz)
    main = polyline([(0, 18, 18), (95, 18, 18), (95, 31, 18), (95, 31, 24), (95, 22, 24), (2, 22, 24), (2, 22, 47)])
    ycor = polyline([(140, 0, 5), (140, ny - 1, 5)])
    zcor = polyline([(150, 5, 0), (150, 5, nz - 1)])
    for c in (main, ycor, zcor):
        carve(w, c)
    pockets = (polyline([(40, 18, 20), (50, 18, 20)])         # beside the first leg, in z
               + polyline([(28, 16, 18), (35, 16, 18)])       # beside the first leg, in y, across the x seam
               + polyline([(97, 18, 18), (97, 25, 18)])       # beside the turn into +y, in the next tile in x
               + polyline([(142, 13, 5), (142, 18, 5)])       # beside the y corridor, across the y seam
               + box(152, 154, 3, 7, 13, 17))                 # beside the z corridor, across the z seam
    carve(w, pockets)
    expect = [((x, 18, 18), x) for x in range(96)] + [((140, y, 5), y) for y in range(ny)] + \
             [((150, 5, z), z) for z in range(nz)]
    return Maze("axis_corridors", w, [(0, 18, 18), (140, 0, 5), (150, 5, 0)], expect=expect, pockets=pockets)


# ---- serpentine ----

def serpentine_cells(nx, ny, z, y0=0):
    """Boustrophedon in the plane z: lanes along x at y = y0, y0+2, ..., joined at alternating ends."""
    pts = []
    lanes = list(range(y0, ny, 2))
    for i, y in enumerate(lanes):
        a, b = (0, nx - 1) if i % 2 == 0 else (nx - 1, 0)
        pts += [(a, y, z), (b, y, z)]
    return polyline(pts)


def serpentine(nx=64, ny=64, nz=3, z=1):
    """One-cell-wide boustrophedon in one slab of the grid; seeded at its start.  64 x 64: 32 lanes, about 2 000 levels
    (250 super-steps of the tile kernel, 11 stepwise chunks of 24 super-steps)."""
    cells = serpentine_cells(nx, ny, z)
    w = solid(nx, ny, nz)
    carve(w, cells)
    return Maze("serpentine", w, [cells[0]], expect=[(cells[0], 0)])


# ---- head-on fronts ----

def head_on():
    """Corridors seeded at both ends, so that the two fronts meet head-on: in the middle of a tile (odd length: one
    cell equidistant from both seeds) and on a seam (even length: the two middle cells are equidistant, one on each
    side of the seam), along x, y and z; plus an open box across three seams seeded at two opposite corners."""
    nx, ny, nz = 128, 48, 48
    w = solid(nx, ny, nz)
    lines = [
        polyline([(16, 5, 5), (78, 5, 5)]),      # 63 cells, middle x = 47 inside tile 1 (x 31..62)
        polyline([(11, 10, 5), (50, 10, 5)]),    # 40 cells, middle pair x = 30 | 31 on the x seam
        polyline([(100, 0, 10), (100, 30, 10)]),  # 31 cells, middle y = 15: the first cell of tile 1
        polyline([(104, 3, 10), (104, 26, 10)]),  # 24 cells, middle pair y = 14 | 15 on the y seam
        polyline([(60, 20, 0), (60, 20, 30)]),   # 31 cells along z, middle z = 15
        polyline([(64, 20, 3), (64, 20, 26)]),   # 24 cells along z, middle pair z = 14 | 15
    ]
    seeds, expect = [], []
    for cells in lines:
        carve(w, cells)
        seeds += [cells[0], cells[-1]]
        n = len(cells)
        expect += [(c, min(i, n - 1 - i)) for i, c in enumerate(cells)]
    room = box(80, 120, 28, 46, 28, 46)          # across the x seam at 95 and the y, z seams at 31
    carve(w, room)
    seeds += [(80, 28, 28), (120, 46, 46)]
    expect += [((x, y, z), min(max(x - 80, y - 28, z - 28), max(120 - x, 46 - y, 46 - z))) for x, y, z in room[::97]]
    return Maze("head_on", w, seeds, expect=expect)


# ---- large grid (the 256-thread tile kernel) ----

def large(n=320):
    """n^3, mostly walls: ntiles >= 4096 from n = 286 up (320^3: 11 * 21 * 21 = 4851), so the single-grid run takes
    bfs_tiles_kernel<4>.  A corridor along x across every x tile, turning at the seam x = 319 into +y and at y = 303 into
    +z (about 900 levels); a diagonal staircase through the tile corner (159, 159, 159); pockets beside both."""
    w = solid(n, n, n)
    main = polyline([(0, 15, 15), (n - 1, 15, 15), (n - 1, n - 17, 15), (n - 1, n - 17, n - 17)])
    stair = staircase_cells((1, -1, 1), (159, 159, 159), 60, 120)
    carve(w, main)
    carve(w, stair)
    pockets = polyline([(100, 15, 17), (140, 15, 17)]) + [(c[0] + 2, c[1], c[2] - 2) for c in stair[10:20]]
    carve(w, pockets)
    expect = [((x, 15, 15), x) for x in range(n)] + [(c, t) for t, c in enumerate(stair)]
    return Maze("large%d" % n, w, [(0, 15, 15), stair[0]], expect=expect, pockets=pockets,
                corner=(stair[60], stair[61]))


def small_mazes():
    """Every small generator's grid."""
    return [staircase(s) for s in SIGNS] + [axis_corridors(), serpentine(), head_on()]


# ---- stacked banks: a field whose slot faces are free ----

def open_face_walls(nx, ny, nz):
    """walls[z, y, x] whose corridors end on the free z = 0 and z = nz - 1 faces: a serpentine on the top face, a patch
    of free cells directly below it on the bottom face, and two shafts from face to face.  In a bank the top face of
    slot s and the bottom face of slot s + 1 are free cells three padded rows apart (two border rows between them)."""
    w = solid(nx, ny, nz)
    top = serpentine_cells(nx, ny - 2, nz - 1, y0=1)
    carve(w, top)
    carve(w, box(2, nx - 3, 1, ny - 2, 0, 0))                         # the bottom face, open
    carve(w, polyline([(0, ny - 1, nz - 1), (0, ny - 1, 0)]))          # shafts at two far corners
    carve(w, polyline([(nx - 1, 0, nz - 1), (nx - 1, 0, 0)]))
    carve(w, [(0, ny - 2, nz - 1), (nx - 1, 1, nz - 1), (1, ny - 1, 0), (nx - 2, 0, 0)])   # their ends joined
    return w


def top_face_seeds(walls, k):
    """k distinct free cells of the top face (z = nz - 1), spread along it."""
    nz = walls.shape[0]
    free = np.argwhere(walls[nz - 1] == 0)                              # (y, x)
    pick = free[np.linspace(0, len(free) - 1, k).astype(int)]
    return [(int(x), int(y), nz - 1) for y, x in pick]


def field_from_walls(walls, dmax_sq):
    """The uint16 distance field [x, y, z] (z fastest) whose d2 = 0 cells are exactly the walls: d2 = 0 on walls,
    dmax_sq elsewhere."""
    return np.where(np.transpose(walls, (2, 1, 0)) != 0, 0, dmax_sq).astype(np.uint16)
