"""Synthetic scenes for the BASELINE.json configs (seeded; see SURVEY.md 8(d) / BASELINE.md table).

ball_pile(n_balls, ...) : jittered lattice of tetrahedral balls with surface gaps of U(0.3,1.2)*sqrt(dHat) and a
                          search direction toward the pile centre -- the "1M-tet ball pile, heavy CCD pair count".
twisted_mat(...)        : the "mat-twist ~100K tets, FixedCoRot, no contact" case.
"""
import numpy as np

from . import mesh as M
from . import msh


def ball_pile(n_balls, res=10, radius=0.5, seed=5, energy=0, dhat_rel=1e-3, gap_lo=0.3, gap_hi=1.2, q=6.0, height=5):
    """Columns of stacked L_q "balls" (rounded, nearly flat poles).  Returns (mesh, info).

    Balls of one column are separated along z by gaps g ~ U(gap_lo, gap_hi) * sqrt(dHat) (pole to pole), rotated about z
    by a random angle (so facing edges are generically not parallel) and shifted laterally by a small jitter; columns
    are far enough apart not to interact.  info = dict(dHat, p, ...): dHat = (dhat_rel)^2 * bboxDiag^2
    (Optimizer.cpp:274-281) and p is a search direction that squeezes every column toward its middle with
    |p| ~ 2-4 sqrt(dHat), i.e. alpha_CFL < 1: the full-CCD branch of Optimizer.cpp:1961 is taken.
    """
    rng = np.random.default_rng(seed)
    n_cols = int(np.ceil(n_balls / height))
    side = int(np.ceil(np.sqrt(n_cols)))
    col_pitch = 2.0 * radius + 0.5
    ext = np.array([side * col_pitch, side * col_pitch, height * 2.0 * radius])
    dHat = dhat_rel ** 2 * float((ext ** 2).sum())
    sq = np.sqrt(dHat)
    Vb, Tb = M.superball_tets(res, radius, q)
    parts, centers, col_mid = [], [], []
    k = 0
    for ci in range(n_cols):
        cx, cy = (ci % side) * col_pitch, (ci // side) * col_pitch
        z = 0.0
        zs = []
        for l in range(height):
            if k >= n_balls:
                break
            th = rng.uniform(0, 2 * np.pi)
            R = np.array([[np.cos(th), -np.sin(th), 0.0], [np.sin(th), np.cos(th), 0.0], [0.0, 0.0, 1.0]])
            c = np.array([cx + rng.normal(0, 0.02), cy + rng.normal(0, 0.02), z])
            parts.append((Vb @ R.T + c, Tb))
            centers.append(c)
            zs.append(z)
            z += 2.0 * radius + rng.uniform(gap_lo, gap_hi) * sq
            k += 1
        col_mid += [0.5 * (zs[0] + zs[-1])] * len(zs)
    m = M.merge_meshes(parts, energy=energy)
    centers = np.array(centers)
    col_mid = np.array(col_mid)
    # mild smooth volumetric deformation (keeps every tet positive and leaves the poles' gaps almost untouched)
    X = m.V_rest
    nVb = Vb.shape[0]
    ball_of = np.repeat(np.arange(len(centers)), nVb)
    local = X - centers[ball_of]
    m.V = X + 0.01 * radius * np.stack([np.sin(2 * np.pi * local[:, 1]), np.sin(2 * np.pi * local[:, 0]), 0 * local[:, 2]], axis=1)
    # search direction: every ball moves toward its column's middle
    dz = col_mid[ball_of] - centers[ball_of, 2]
    p = np.zeros((m.nV, 3))
    p[:, 2] = np.sign(dz) * 3.0 * sq * rng.uniform(0.6, 1.0, m.nV)
    p += rng.normal(0, 0.1 * sq, (m.nV, 3))
    info = dict(dHat=dHat, p=np.ascontiguousarray(p).ravel(), centers=centers, radius=radius, n_balls=len(centers))
    return m, info


def twisted_mat(nx=26, ny=26, nz=25, seed=2, energy=1, invert_frac=0.001):
    V, T = M.grid_tets(nx, ny, nz)
    m = M.Mesh(V, T, energy=energy)
    M.deform(m, seed, twist=np.pi, amp=0.02, noise=0.02)
    if invert_frac > 0 and energy == 1:
        rng = np.random.default_rng(seed)
        k = max(1, int(invert_frac * m.nV))
        m.V[rng.integers(0, m.nV, k)] += 0.8 * m.avgEdgeLen * rng.standard_normal((k, 3))
    return m


def ball_on_mat(nx=40, res=6, seed=3, energy=0, dhat_rel=1e-3, gap_lo=0.2, gap_hi=1.5):
    """BASELINE config C3 ("ball-on-mat, barrier contact + CCD line search"): a one-cell-thick mat of nx x nx x 1 cells (all surface, as
    the reference's thin mats are) and a ball hovering over its middle at a gap of U(gap_lo, gap_hi)*sqrt(dHat); the search direction
    pushes the ball down by up to 2 sqrt(dHat) (BASELINE.md C3: nx=200 -> 240,000 mat tets).  Returns (mesh, info) like ball_pile."""
    rng = np.random.default_rng(seed)
    h = 1.0 / nx
    Vm, Tm = M.grid_tets(nx, nx, 1, h=h)
    radius = 0.15
    Vb, Tb = M.superball_tets(res, radius, 2.0)
    ext = np.array([1.0, 1.0, h + 2 * radius])
    dHat = dhat_rel ** 2 * float((ext ** 2).sum())
    sq = np.sqrt(dHat)
    gap = rng.uniform(gap_lo, gap_hi) * sq
    nVm = Vm.shape[0]
    Vm_def = Vm + 0.02 * h * rng.standard_normal((nVm, 3)) * np.array([1.0, 1.0, 0.2])
    # the ball's lowest vertex sits `gap` above the highest mat vertex; off the lattice so that no feature pair is exactly degenerate
    c = np.array([0.5 + 0.31 * h, 0.5 - 0.17 * h, Vm_def[:, 2].max() + gap - Vb[:, 2].min()])
    m = M.merge_meshes([(Vm, Tm), (Vb + c, Tb)], energy=energy)
    m.V = m.V_rest.copy()
    m.V[:nVm] = Vm_def
    p = np.zeros((m.nV, 3))
    p[nVm:, 2] = -rng.uniform(0.0, 2.0, m.nV - nVm) * sq
    p += rng.normal(0, 0.05 * sq, (m.nV, 3))
    return m, dict(dHat=dHat, p=np.ascontiguousarray(p).ravel(), n_mat_verts=nVm, gap=gap)


# ---------------------------------------------------------------------------------------------------------------------------------
# scenes built from the reference's own assets (assets/_ref cache, see msh.py); BASELINE.md table, configs C3 / C4 / C5
# ---------------------------------------------------------------------------------------------------------------------------------
def shape_transform(V, translate=(0, 0, 0), rotate_deg=(0, 0, 0), scale=(1, 1, 1)):
    """Placement of an input shape exactly as the reference applies a `shapes input` line: x' = R (x * scale) + t with
    R = Rx(a) Ry(b) Rz(c) (Config.cpp:218-224, main.cpp:1074-1077)."""
    a, b, c = np.deg2rad(rotate_deg)
    Rx = np.array([[1, 0, 0], [0, np.cos(a), -np.sin(a)], [0, np.sin(a), np.cos(a)]])
    Ry = np.array([[np.cos(b), 0, np.sin(b)], [0, 1, 0], [-np.sin(b), 0, np.cos(b)]])
    Rz = np.array([[np.cos(c), -np.sin(c), 0], [np.sin(c), np.cos(c), 0], [0, 0, 1]])
    return (V * np.asarray(scale, dtype=float)) @ (Rx @ Ry @ Rz).T + np.asarray(translate, dtype=float)


def affine_prestrain(m, about=None):
    """Multiply the CURRENT state by a small fixed strain (I + E), |E| ~ 1e-3, about a point: no tet is left exactly at rest.
    Why the parity scenes need it: IglUtils::makePD2d (IglUtils.hpp:138-177) is DISCONTINUOUS at L2 = 0 -- for L2 < 0 it returns
    (L1 - d)^2 / L1 etc., which is not the limit of the untouched matrix as L2 -> 0- (at F = I the twist block [[mu, mu], [mu, mu]] comes
    back halved) -- and at an exact rest state L2 = +-1e-17 is pure rounding noise of the SVD, in the reference as much as here.  Two
    correct implementations of the same formulas (the oracle's implicit-QR SVD, the kernels' Jacobi SVD) then disagree per tet on the
    branch.  Gaps between bodies change by a relative 1e-3, i.e. not at all at the resolution of the U(lo, hi) sqrt(dHat) placement."""
    E = np.array([[1.0e-3, 2.0e-4, -1.0e-4], [2.0e-4, -7.0e-4, 3.0e-4], [-1.0e-4, 3.0e-4, 4.0e-4]])
    c = m.V.mean(0) if about is None else np.asarray(about, dtype=float)
    m.V = (m.V - c) @ (np.eye(3) + E).T + c
    return m


def _fcc_points(n):
    """the n points of the FCC lattice (nearest-neighbour distance 1) closest to the origin, ordered by distance then lexicographically"""
    k = int(np.ceil((n / 4.0) ** (1.0 / 3.0))) + 2
    g = np.arange(-k, k + 1)
    I, J, K = np.meshgrid(g, g, g, indexing="ij")
    keep = (I + J + K) % 2 == 0
    P = np.stack([I[keep], J[keep], K[keep]], axis=1).astype(np.float64) / np.sqrt(2.0)
    r2 = (P ** 2).sum(1)
    order = np.lexsort((P[:, 2], P[:, 1], P[:, 0], np.round(r2, 9)))
    return P[order[:n]]


def _random_rotations(rng, n):
    q = rng.standard_normal((n, 4))
    q /= np.linalg.norm(q, axis=1)[:, None]
    w, x, y, z = q.T
    return np.stack([np.stack([1 - 2 * (y * y + z * z), 2 * (x * y - z * w), 2 * (x * z + y * w)], 1),
                     np.stack([2 * (x * y + z * w), 1 - 2 * (x * x + z * z), 2 * (y * z - x * w)], 1),
                     np.stack([2 * (x * z - y * w), 2 * (y * z + x * w), 1 - 2 * (x * x + y * y)], 1)], 1)


def sphere_pile_fcc(n_balls=146, seed=5, energy=0, dhat_rel=1e-3, gap_lo=0.3, gap_hi=1.2, ball=None):
    """BASELINE config C5 as specified (BASELINE.md / SURVEY 8(d)): `n_balls` copies of input/tetMeshes/sphere1K.msh (146 copies =
    1,000,246 tets, 256,960 verts, 180,894 surface verts) on a jittered FCC lattice -- every ball has up to 12 neighbours at
    surface gaps of U(gap_lo, gap_hi)*sqrt(dHat) -- each ball randomly rotated; the search direction moves every ball toward the pile
    centre with |p| ~ 2-3 sqrt(dHat), so alpha_CFL = sqrt(dHat)/(2 max|p|) < 1 and the full-CCD branch of Optimizer.cpp:1961 is taken.
    `ball` = (V, T, SF) overrides the asset (used when the asset cache is absent: a synthetic ball of similar size)."""
    rng = np.random.default_rng(seed)
    if ball is None:
        ball = msh.load_asset("sphere1K")
    Vb, Tb, SFb = ball
    Vb = Vb - 0.5 * (Vb.max(0) + Vb.min(0))
    # contact radius of the faceted ball: the mean radius of its surface vertices (sphere1K: 0.4992; vertices range over 0.4966-0.5018,
    # facet centres sit ~0.001 lower), so that the surface-to-surface gaps -- not the gaps of the circumscribed spheres -- follow U(lo, hi)
    sv = np.unique(SFb) if len(SFb) else np.arange(len(Vb))
    R = float(np.linalg.norm(Vb[sv], axis=1).mean())
    lat = _fcc_points(n_balls)
    ext = (lat.max(0) - lat.min(0)) * 2.0 * R + 2.0 * R
    dHat = dhat_rel ** 2 * float((ext ** 2).sum())
    sq = np.sqrt(dHat)
    # centre distance 2R + mid gap; a jitter of <= 0.2 sqrt(dHat) per centre moves every gap by at most 0.4 sqrt(dHat)
    mid, half = 0.5 * (gap_lo + gap_hi), 0.5 * (gap_hi - gap_lo)
    D = 2.0 * R + mid * sq
    jit = rng.standard_normal((n_balls, 3))
    jit *= (rng.uniform(0, 1, n_balls) ** (1 / 3) / np.maximum(np.linalg.norm(jit, axis=1), 1e-300))[:, None]
    centers = lat * D + jit * (0.5 * half * sq * 0.95)
    Rm = _random_rotations(rng, n_balls)
    parts = [(Vb @ Rm[k].T + centers[k], Tb, SFb) for k in range(n_balls)]
    m = M.merge_meshes(parts, energy=energy)
    nVb = Vb.shape[0]
    ball_of = np.repeat(np.arange(n_balls), nVb)
    local = m.V_rest - centers[ball_of]
    # smooth internal strain that vanishes on the sphere r = R (surface gaps stay as placed, every tet stays positive)
    r2 = (local ** 2).sum(1) / (R * R)
    bump = np.clip(1.0 - r2, 0.0, None)
    m.V = m.V_rest + (0.03 * R) * bump[:, None] * np.stack([np.sin(2 * np.pi * local[:, 1]), np.sin(2 * np.pi * local[:, 2]), np.sin(2 * np.pi * local[:, 0])], axis=1)
    c0 = centers.mean(0)
    to_c = c0 - centers
    nrm = np.linalg.norm(to_c, axis=1)
    dirn = np.where(nrm[:, None] > 1e-12, to_c / np.maximum(nrm, 1e-300)[:, None], 0.0)
    p = dirn[ball_of] * (3.0 * sq * rng.uniform(0.6, 1.0, m.nV))[:, None]
    p += rng.normal(0, 0.1 * sq, (m.nV, 3))
    info = dict(dHat=dHat, p=np.ascontiguousarray(p).ravel(), centers=centers, radius=R, n_balls=n_balls, ball_verts=nVb)
    return m, info


def ball_on_mat_c3(nx=200, seed=3, energy=0, dhat_rel=1e-3, gap_lo=0.2, gap_hi=1.5):
    """BASELINE config C3 at its full size: mat grid nx x nx x 1 cells (nx = 200 -> 240,000 tets, all surface like the reference's thin
    mats) + input/tetMeshes/sphere1K.msh (6,851 tets) hovering over the middle at a gap of U(gap_lo, gap_hi)*sqrt(dHat), dHat relative
    1e-3, ball pushed down by up to 2 sqrt(dHat) (12_sphereOnMat.txt:2-3 is the same pair of bodies at 16K tets)."""
    rng = np.random.default_rng(seed)
    h = 1.0 / nx
    Vm, Tm = M.grid_tets(nx, nx, 1, h=h)
    Vb, Tb, SFb = msh.load_asset("sphere1K")
    radius = 0.15
    Vb = shape_transform(Vb - 0.5 * (Vb.max(0) + Vb.min(0)), rotate_deg=(90, 0, 45), scale=(2 * radius,) * 3)
    ext = np.array([1.0, 1.0, h + 2 * radius])
    dHat = dhat_rel ** 2 * float((ext ** 2).sum())
    sq = np.sqrt(dHat)
    gap = rng.uniform(gap_lo, gap_hi) * sq
    nVm = Vm.shape[0]
    Vm_def = Vm + 0.02 * h * rng.standard_normal((nVm, 3)) * np.array([1.0, 1.0, 0.2])
    c = np.array([0.5 + 0.31 * h, 0.5 - 0.17 * h, Vm_def[:, 2].max() + gap - Vb[:, 2].min()])
    m = M.merge_meshes([(Vm, Tm, M.boundary_faces(Tm)), (Vb + c, Tb, SFb)], energy=energy)
    m.V = m.V_rest.copy()
    m.V[:nVm] = Vm_def
    affine_prestrain(m)  # the ball would otherwise sit exactly at rest (see affine_prestrain)
    p = np.zeros((m.nV, 3))
    p[nVm:, 2] = -rng.uniform(0.0, 2.0, m.nV - nVm) * sq
    p += rng.normal(0, 0.05 * sq, (m.nV, 3))
    return m, dict(dHat=dHat, p=np.ascontiguousarray(p).ravel(), n_mat_verts=nVm, gap=gap)


# the four tet bodies of input/paperExamples/1_squeezeOut.txt:12-15 with their script placement (translate, rotate, scale)
SQUEEZE_OUT_BODIES = [("alien", (0, -1.05, 0), (0, 0, 0), 0.45), ("hollowCat7.5K", (1.2, 0.2, -0.1), (-90, 0, 0), 0.22),
                      ("monkey8K", (-0.03, 1.05, 0), (-90, 0, 0), 0.012), ("32770_octocat", (0, 1.9, 0), (-90, 0, 0), 0.01)]


def have_squeeze_out_meshes():
    """the C4 meshes are too large to store in the repository: they exist only where the build cached them (msh.build_asset_cache)"""
    return all(msh.have_asset(name) for name, *_ in SQUEEZE_OUT_BODIES)


def _vertex_normals(V, SF):
    n = np.cross(V[SF[:, 1]] - V[SF[:, 0]], V[SF[:, 2]] - V[SF[:, 0]])
    N = np.zeros_like(V)
    for k in range(3):
        np.add.at(N, SF[:, k], n)
    ln = np.linalg.norm(N, axis=1)
    return N / np.maximum(ln, 1e-300)[:, None]


def squeeze_out_tiled(seed=4, energy=0, dhat_rel=1e-3, gap_lo=0.3, gap_hi=1.2, contact_frac=0.05, far=2.5, slide=0.15, bodies=None):
    """BASELINE config C4: the tet bodies of 1_squeezeOut.txt:12-15 (180,569 tets) tiled x3 (541,707 tets) with dense self-contact.

    No simulation is available to press the bodies together, so the squeezed state is manufactured per body from three copies:
      copy 0  the body at its script placement;
      copy 1  the same body with every SURFACE vertex pushed out along its vertex normal: by U(gap_lo, gap_hi)*sqrt(dHat) (plus a random
              tangential slide of <= 0.15 local edge lengths) inside smooth patches that cover ~`contact_frac` of the surface, by `far` sqrt(dHat)
              elsewhere -- its surface hovers over copy 0's surface like a squeezed neighbour would, giving patches of PT / EE / PE / PP
              and nearly-parallel (mollified) pairs; the two solids overlap in volume, which the surface-based contact path does not see;
      copy 2  a free copy moved aside by a seeded offset (jittered tile).
    dHat = (dhat_rel * bboxDiag)^2.  The search direction pushes copy 1's contact patches inward (toward copy 0) by up to 2 sqrt(dHat) and
    shakes everything else by 0.05 sqrt(dHat).  Returns (mesh, info) like ball_pile."""
    rng = np.random.default_rng(seed)
    if bodies is None:
        bodies = [(msh.load_asset(name), tr, rot, sc) for name, tr, rot, sc in SQUEEZE_OUT_BODIES]
    placed = []
    for (V, T, SF), tr, rot, sc in bodies:
        if len(SF) == 0:
            SF = M.boundary_faces(T)
        placed.append((shape_transform(V, tr, rot, (sc,) * 3), T, SF))
    allV = np.concatenate([b[0] for b in placed])
    ext = allV.max(0) - allV.min(0)
    tile = np.array([ext[0] * 1.25, 0.0, 0.0])
    ext3 = ext + 2 * tile
    dHat = dhat_rel ** 2 * float((ext3 ** 2).sum())
    sq = np.sqrt(dHat)
    parts, push = [], []
    for bi, (V, T, SF) in enumerate(placed):
        sv = np.unique(SF)
        N = _vertex_normals(V, SF)
        e = np.concatenate([np.linalg.norm(V[SF[:, i]] - V[SF[:, (i + 1) % 3]], axis=1) for i in range(3)])
        el = np.zeros(len(V)); cnt = np.zeros(len(V))
        for i in range(3):
            np.add.at(el, SF[:, i], e[i * len(SF):(i + 1) * len(SF)]); np.add.at(cnt, SF[:, i], 1.0)
        el = el / np.maximum(cnt, 1.0)
        # smooth patch mask: low-frequency field thresholded at the quantile that leaves `contact_frac` of the surface vertices inside
        c, L = V.mean(0), float(np.linalg.norm(V.max(0) - V.min(0)))
        ph = rng.uniform(0, 2 * np.pi, 3)
        fld = np.sin(7.0 * (V[:, 0] - c[0]) / L * 2 * np.pi + ph[0]) + np.sin(5.0 * (V[:, 1] - c[1]) / L * 2 * np.pi + ph[1]) + np.sin(6.0 * (V[:, 2] - c[2]) / L * 2 * np.pi + ph[2])
        thr = np.quantile(fld[sv], 1.0 - contact_frac)
        inside = np.zeros(len(V), dtype=bool)
        inside[sv] = fld[sv] >= thr
        off = np.zeros(len(V))
        off[sv] = far * sq
        off[inside] = rng.uniform(gap_lo, gap_hi, int(inside.sum())) * sq
        tang = rng.standard_normal(V.shape)
        tang -= (tang * N).sum(1)[:, None] * N
        tang *= (slide * el * rng.uniform(0, 1, len(V)) / np.maximum(np.linalg.norm(tang, axis=1), 1e-300))[:, None]
        tang[~inside] = 0.0
        disp = N * off[:, None] + tang
        # repair: where pushing along diverse normals (concave creases, slivers) would invert or crush a tet, replace the displacements
        # of its vertices by their mean (locally rigid translation), repeated until every tet keeps >= 30 % of its rest volume
        x0 = V[T]
        vol0 = np.linalg.det(np.stack([x0[:, 1] - x0[:, 0], x0[:, 2] - x0[:, 0], x0[:, 3] - x0[:, 0]], axis=2))
        for _ in range(200):
            x = (V + disp)[T]
            ratio = np.linalg.det(np.stack([x[:, 1] - x[:, 0], x[:, 2] - x[:, 0], x[:, 3] - x[:, 0]], axis=2)) / vol0
            bad = np.nonzero(ratio < 0.3)[0]
            if len(bad) == 0:
                break
            mean = disp[T[bad]].mean(axis=1)
            acc, cnt2 = np.zeros_like(disp), np.zeros(len(V))
            for k in range(4):
                np.add.at(acc, T[bad, k], mean)
                np.add.at(cnt2, T[bad, k], 1.0)
            touched = cnt2 > 0
            disp[touched] = acc[touched] / cnt2[touched, None]
        V1 = V + disp
        V2 = V + tile * (1 if bi % 2 == 0 else -1) + rng.normal(0, 0.01 * L, 3)
        parts += [(V, T, SF), (V1, T, SF), (V2, T, SF)]
        pv = np.zeros((len(V), 3))
        pv[inside] = -N[inside] * (rng.uniform(0.0, 2.0, int(inside.sum())) * sq)[:, None]
        push += [np.zeros((len(V), 3)), pv, np.zeros((len(V), 3))]
    # rest shapes: copies 0 and 2 rest where they are; copy 1 rests on the undeformed body (its pushed-out surface is a strained state)
    rest = [(parts[k - 1][0] if k % 3 == 1 else parts[k][0], parts[k][1], parts[k][2]) for k in range(len(parts))]
    m = M.merge_meshes(rest, energy=energy)
    m.V = np.concatenate([b[0] for b in parts])
    affine_prestrain(m)  # copies 0 and 2 would otherwise sit exactly at rest (see affine_prestrain)
    p = np.concatenate(push) + rng.normal(0, 0.05 * sq, (m.nV, 3))
    return m, dict(dHat=dHat, p=np.ascontiguousarray(p).ravel(), n_bodies=len(placed), tile=tile)


# ---------------------------------------------------------------------------------------------------------------------------------
# a mesh next to a kinematic obstacle (row f3: MeshCO) -- test scene, seeded
# ---------------------------------------------------------------------------------------------------------------------------------
def surface_of(V, T):
    """(V, E, F) of the boundary surface of a tet mesh with compact vertex numbering: what MeshCO loads from an .obj
    (MeshCO.cpp:37-80: Base::V, Base::F, edges collected from F like Mesh::SFEdges)."""
    SF = M.boundary_faces(np.asarray(T, dtype=np.int32))
    used = np.unique(SF)
    remap = -np.ones(len(V), dtype=np.int64)
    remap[used] = np.arange(len(used))
    F = remap[SF].astype(np.int32)
    return np.ascontiguousarray(V[used], dtype=np.float64), M.surface_edges(F), F


def balls_on_obstacle(n_balls=3, res=4, plate=12, seed=7, energy=0, dhat_rel=1e-3, gap_lo=0.3, gap_hi=1.2, plate_angle=0.37):
    """A short column of rounded balls (self contact between them) whose lowest ball hovers U(gap_lo, gap_hi) sqrt(dHat) over an obstacle
    plate, with a second obstacle body -- a rotated ball surface -- just beside the column.  The obstacle is ONE triangle mesh with two
    components.  The search direction pushes the column down and toward the side body by 2-4 sqrt(dHat), so both step bounds bite.
    Returns (mesh, info) with info["obstacle"] = dict(V, E, F) in the obstacle's own numbering."""
    rng = np.random.default_rng(seed)
    radius = 0.5
    Vb, Tb = M.superball_tets(res, radius, 6.0)
    ext = np.array([3.0, 3.0, n_balls * 2.0 * radius + 0.2])
    dHat = dhat_rel ** 2 * float((ext ** 2).sum())
    sq = np.sqrt(dHat)
    parts, z = [], 0.0
    for _ in range(n_balls):
        th = rng.uniform(0, 2 * np.pi)
        R = np.array([[np.cos(th), -np.sin(th), 0.0], [np.sin(th), np.cos(th), 0.0], [0.0, 0.0, 1.0]])
        parts.append((Vb @ R.T + np.array([rng.normal(0, 0.01), rng.normal(0, 0.01), z]), Tb))
        z += 2.0 * radius + rng.uniform(gap_lo, gap_hi) * sq
    m = M.merge_meshes(parts, energy=energy)
    local = m.V_rest - np.array([0.0, 0.0, 0.0])
    m.V = m.V_rest + 0.004 * radius * np.stack([np.sin(5 * local[:, 1]), np.sin(5 * local[:, 0]), 0 * local[:, 2]], axis=1)
    # obstacle 1: a plate under the column, slightly bumpy and rotated about z so that its edges are generically not parallel to the balls'
    h = 3.0 / plate
    Vp, Tp = M.grid_tets(plate, plate, 1, h=h, origin=(-1.5, -1.5, -h))
    th = plate_angle  # 0: the plate's edges are parallel to the grid edges of the balls' flat poles (mollified entries)
    Rz = np.array([[np.cos(th), -np.sin(th), 0.0], [np.sin(th), np.cos(th), 0.0], [0.0, 0.0, 1.0]])
    Vp = Vp @ Rz.T
    if plate_angle != 0.0:
        Vp[:, 2] += 0.2 * sq * np.sin(3.1 * Vp[:, 0]) * np.cos(2.3 * Vp[:, 1])
    Vp[:, 2] += m.V[:, 2].min() - rng.uniform(gap_lo, gap_hi) * sq - Vp[:, 2].max()
    # obstacle 2: a ball surface beside the lowest ball of the column
    th2 = 0.9
    Ry = np.array([[np.cos(th2), 0.0, np.sin(th2)], [0.0, 1.0, 0.0], [-np.sin(th2), 0.0, np.cos(th2)]])
    Vs = Vb @ Ry.T
    low = m.V[: Vb.shape[0]]
    Vs += np.array([low[:, 0].max() - Vs[:, 0].min() + rng.uniform(gap_lo, gap_hi) * sq, 0.013, low[:, 2].mean() - Vs[:, 2].mean() + 0.021])
    V1, E1, F1 = surface_of(Vp, Tp)
    V2, E2, F2 = surface_of(Vs, Tb)
    Vo = np.concatenate([V1, V2])
    Fo = np.concatenate([F1, F2 + len(V1)]).astype(np.int32)
    Eo = M.surface_edges(Fo)
    p = np.zeros((m.nV, 3))
    p[:, 2] = -3.0 * sq * rng.uniform(0.6, 1.0, m.nV)
    p[:, 0] = 2.0 * sq * rng.uniform(0.6, 1.0, m.nV)
    p += rng.normal(0, 0.1 * sq, (m.nV, 3))
    info = dict(dHat=dHat, p=np.ascontiguousarray(p).ravel(), obstacle=dict(V=Vo, E=Eo, F=Fo))
    return m, info


def ball_on_obstacle_mat(nx=200, seed=3, energy=0, dhat_rel=1e-3, gap_lo=0.2, gap_hi=1.5):
    """BASELINE config C3's pair of bodies with the mat as a kinematic OBSTACLE (what 12_sphereOnMat.txt would be with the mat loaded through
    `meshCO`): the mesh is input/tetMeshes/sphere1K.msh alone, the obstacle is the surface of the nx x nx x 1 mat (nx = 200: 80,802 vertices,
    160,800 triangles).  Same placement, gap and search direction as ball_on_mat_c3.  Returns (mesh, info) with info["obstacle"]."""
    rng = np.random.default_rng(seed)
    h = 1.0 / nx
    Vm, Tm = M.grid_tets(nx, nx, 1, h=h)
    Vb, Tb, SFb = msh.load_asset("sphere1K")
    radius = 0.15
    Vb = shape_transform(Vb - 0.5 * (Vb.max(0) + Vb.min(0)), rotate_deg=(90, 0, 45), scale=(2 * radius,) * 3)
    ext = np.array([1.0, 1.0, h + 2 * radius])
    dHat = dhat_rel ** 2 * float((ext ** 2).sum())
    sq = np.sqrt(dHat)
    gap = rng.uniform(gap_lo, gap_hi) * sq
    Vm_def = Vm + 0.02 * h * rng.standard_normal((Vm.shape[0], 3)) * np.array([1.0, 1.0, 0.2])
    c = np.array([0.5 + 0.31 * h, 0.5 - 0.17 * h, Vm_def[:, 2].max() + gap - Vb[:, 2].min()])
    m = M.merge_meshes([(Vb + c, Tb, SFb)], energy=energy)
    affine_prestrain(m)
    Vo, Eo, Fo = surface_of(Vm_def, Tm)
    p = np.zeros((m.nV, 3))
    p[:, 2] = -rng.uniform(0.0, 2.0, m.nV) * sq
    p += rng.normal(0, 0.05 * sq, (m.nV, 3))
    return m, dict(dHat=dHat, p=np.ascontiguousarray(p).ravel(), gap=gap, obstacle=dict(V=Vo, E=Eo, F=Fo))
