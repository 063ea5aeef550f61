"""Reader for the reference's tet-mesh files (`input/tetMeshes/*.msh`) and the build-time asset cache.

Format: Gmsh MSH 4.1 ASCII with ONE node block and ONE element block, followed by the reference's custom `$Surface` section
(1-based surface triangles) -- what `IglUtils::readTetMesh` / `readTetMesh_msh4` consume (src/Utils/IglUtils.cpp:440-570).
In a 4.1 node block the node tags come first and the coordinates after them; element lines are `tag v0 v1 v2 v3` (1-based).

The meshes are scene INPUT DATA, not source.  sphere1K (C3 / C5 and the bench.py workload) is stored in the repository as
`tests/golden/sphere1K.npz`.  The larger meshes of the other BASELINE configs are too big to store: `build_asset_cache()` (called by
`__graft_entry__.build()` wherever the reference tree is present) converts them into `assets/_ref/<name>.npz`, a git-ignored cache, and
the tests that need them skip without it.  Nothing on the hot path reads either: they feed the scene generators of the tests and of bench.py.
"""
import os

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CACHE_DIR = os.path.join(ROOT, "assets", "_ref")
STORED_DIR = os.path.join(ROOT, "tests", "golden")
REFERENCE_MESH_DIR = "/root/reference/input/tetMeshes"
# meshes named by the BASELINE configs and not stored in the repository: C3 mat40x40 (12_sphereOnMat.txt:3), C2 mat150x150t40
# (14_matTwist.txt:2), C4 the four tet bodies of 1_squeezeOut.txt:12-15, C1 cube (tutorialExamples/2cubesFall.txt)
ASSETS = ["cube", "mat40x40", "mat150x150t40", "alien", "hollowCat7.5K", "monkey8K", "32770_octocat"]


def read_msh(path):
    """Returns V (nV,3) float64, T (nT,4) int32 0-based, SF (nSF,3) int32 0-based (empty if the file has no $Surface)."""
    with open(path, "r") as f:
        tok = f.read().split()
    pos = {}
    for k, t in enumerate(tok):
        if t and t[0] == "$":
            pos.setdefault(t, k)
    k = pos["$Nodes"] + 1
    n_blocks, nV = int(tok[k]), int(tok[k + 1])
    k += 4
    V = np.empty((nV, 3))
    tags = np.empty(nV, dtype=np.int64)
    got = 0
    for _ in range(n_blocks):
        n = int(tok[k + 3])
        k += 4
        tags[got:got + n] = np.array(tok[k:k + n], dtype=np.int64)
        k += n
        V[got:got + n] = np.array(tok[k:k + 3 * n], dtype=np.float64).reshape(n, 3)
        k += 3 * n
        got += n
    assert got == nV and tok[k] == "$EndNodes"
    assert np.array_equal(tags, np.arange(1, nV + 1)), "node tags are expected to be 1..N in order"
    k = pos["$Elements"] + 1
    n_blocks, nT = int(tok[k]), int(tok[k + 1])
    k += 4
    T = np.empty((nT, 4), dtype=np.int64)
    got = 0
    for _ in range(n_blocks):
        etype, n = int(tok[k + 2]), int(tok[k + 3])
        assert etype == 4, "only 4-node tetrahedra are expected"
        k += 4
        blk = np.array(tok[k:k + 5 * n], dtype=np.int64).reshape(n, 5)
        T[got:got + n] = blk[:, 1:] - 1
        k += 5 * n
        got += n
    assert got == nT
    SF = np.empty((0, 3), dtype=np.int64)
    if "$Surface" in pos:
        k = pos["$Surface"] + 1
        n = int(tok[k])
        SF = np.array(tok[k + 1:k + 1 + 3 * n], dtype=np.int64).reshape(n, 3) - 1
    return V, T.astype(np.int32), SF.astype(np.int32)


def write_msh(path, V, T, SF=None):
    """Same layout as the reference's files, so that a real reference build elsewhere can consume generated scenes."""
    with open(path, "w") as f:
        nV, nT = len(V), len(T)
        f.write("$MeshFormat\n4.1 0 8\n$EndMeshFormat\n$Nodes\n1 %d 1 %d\n3 0 0 %d\n" % (nV, nV, nV))
        f.write("\n".join(str(i + 1) for i in range(nV)) + "\n")
        f.write("\n".join("%.17e %.17e %.17e" % tuple(v) for v in V) + "\n$EndNodes\n")
        f.write("$Elements\n1 %d 1 %d\n3 0 4 %d\n" % (nT, nT, nT))
        f.write("\n".join("%d %d %d %d %d" % (i + 1, *(t + 1)) for i, t in enumerate(np.asarray(T))) + "\n$EndElements\n")
        if SF is not None and len(SF):
            f.write("$Surface\n%d\n" % len(SF))
            f.write("\n".join("%d %d %d" % tuple(s + 1) for s in np.asarray(SF)) + "\n$EndSurface\n")


def build_asset_cache(force=False):
    """Convert the reference meshes named in ASSETS to assets/_ref/*.npz (no-op where the reference tree is absent)."""
    if not os.path.isdir(REFERENCE_MESH_DIR):
        return []
    os.makedirs(CACHE_DIR, exist_ok=True)
    made = []
    for name in ASSETS:
        src, dst = os.path.join(REFERENCE_MESH_DIR, name + ".msh"), os.path.join(CACHE_DIR, name + ".npz")
        if not os.path.exists(src) or (os.path.exists(dst) and not force):
            continue
        V, T, SF = read_msh(src)
        np.savez_compressed(dst, V=V, T=T, SF=SF)
        made.append(name)
    return made


def _asset_path(name):
    stored = os.path.join(STORED_DIR, name + ".npz")
    return stored if os.path.exists(stored) else os.path.join(CACHE_DIR, name + ".npz")


def have_asset(name):
    return os.path.exists(_asset_path(name))


def load_asset(name):
    """(V, T, SF) of a stored or cached reference mesh; raises FileNotFoundError when neither exists."""
    z = np.load(_asset_path(name))
    return z["V"].copy(), z["T"].copy(), z["SF"].copy()
