"""assets.load_obj (Wavefront reader for real duckietown-world meshes) against the REFERENCE's ObjMesh loader
(objmesh.py:65-293) on a synthetic OBJ/MTL pair.  tests/golden/objmesh.npz holds what ObjMesh produced for this pair
(`python oracle/make_golden.py interfaces`, which runs the reference through the stub-import harness)."""
import hashlib
import os

import numpy as np

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "objmesh.npz")

OBJ = """# synthetic prop
mtllib prop.mtl
o prop
v 0.0 0.1 0.0
v 1.0 0.1 0.0
v 1.0 0.9 0.5
v 0.0 0.9 0.5
v 0.5 1.4 2.0
vt 0.0 0.0
vt 1.0 0.0
vt 1.0 1.0
vn 0.0 0.0 1.0
vn 0.0 1.0 0.0
usemtl red
f 1/1/1 2/2/1 3/3/1
f 1/1/1 3/3/1 4/2/1
usemtl blue
f 3//2 4//2 5//2
usemtl unknown_material
f 1//2 2//2 5//2
"""
MTL = """newmtl red
Kd 0.8 0.1 0.1
newmtl blue
Kd 0.1 0.2 0.9
"""


def source_digest():
    return hashlib.sha256((OBJ + MTL).encode()).hexdigest()


def test_load_obj_matches_reference_objmesh(tmp_path):
    from gym_duckietown_b200 import assets
    (tmp_path / "prop.obj").write_text(OBJ)
    (tmp_path / "prop.mtl").write_text(MTL)
    ref = np.load(GOLD)
    assert str(ref["source_sha"]) == source_digest()      # the golden file was made from this very OBJ / MTL pair
    mine = assets.load_obj(str(tmp_path / "prop.obj"), "prop")
    assert np.array_equal(mine.min_coords, ref["min_coords"]) and np.array_equal(mine.max_coords, ref["max_coords"])
    assert np.array_equal(mine.tri_pos, ref["tri_pos"])      # incl. the max().min() re-centring quirk (objmesh.py:219)
    assert np.array_equal(mine.tri_nrm, ref["tri_nrm"]) and np.array_equal(mine.tri_uv, ref["tri_uv"])
    assert np.array_equal(mine.tri_col, ref["tri_col"])
