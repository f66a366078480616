"""The normalised scene fixtures (tests/levels/*.xml, written by tests/levels/make_levels.py) compile to exactly
the same model as the reference's own level files.  The reference side is tests/golden/reference_levels.npz,
which make_levels.py writes from the reference levels together with the fixtures."""
import hashlib
import json
import os

import numpy as np

from mujoco_rl_environment_wrapper_b200 import _lib as L

HERE = os.path.dirname(os.path.abspath(__file__))
GOLDEN = os.path.join(HERE, "golden", "reference_levels.npz")


def test_normalised_scenes_compile_identically():
    import importlib.util
    spec = importlib.util.spec_from_file_location("make_levels", os.path.join(HERE, "levels", "make_levels.py"))
    ml = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(ml)
    g = np.load(GOLDEN)
    for out in ml.SCENES:
        assert f"{out}/blob" in g.files, f"{out} has no reference in {GOLDEN}: rerun make_levels.py"
        a = L.parse_blob(g[f"{out}/blob"].tobytes())
        path = os.path.join(HERE, "levels", out)
        b = L.Model.from_xml_path(path)
        assert sorted(a) == sorted(b.fields), out
        keep_cams = out in ml.KEEP_CAMERAS
        for k in a:
            if k.startswith("cam_") or k == "ncam":   # the fixtures drop the cameras unless they are about cameras
                if not keep_cams:
                    assert b.ncam == 0
                    continue
            assert np.array_equal(a[k], b.fields[k]), (out, k)
        names = json.loads(str(g[f"{out}/names"]))
        for objtype, n in ((L.OBJ_BODY, b.nbody), (L.OBJ_JOINT, b.njnt), (L.OBJ_GEOM, b.ngeom), (L.OBJ_SITE, b.nsite), (L.OBJ_SENSOR, b.nsensor)):
            assert names[str(objtype)] == [b.id2name(objtype, i) for i in range(n)], (out, objtype)
        # and the fixture is the generator's normal form of the reference level
        assert hashlib.sha256(open(path).read().encode()).hexdigest() == str(g[f"{out}/sha256"]), out
