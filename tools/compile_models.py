"""Compile the composed MJCF scenes into flat tables (furniture_b200/compiled/*.npz).

Needs the reference's MJCF asset tree, named by FURNITURE_ASSETS.  Without it the package loads these tables
(mjcf.load_scene).  Only derived numeric tables are stored, no reference source."""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from furniture_b200 import mjcf  # noqa: E402

SCENES = [("Sawyer", "table_lack_0825"), ("None", "table_lack_0825"), ("Sawyer", "swivel_chair_0700"), ("Baxter", "chair_ingolf_0650"), ("Baxter", "table_lack_0825"), ("Cursor", "toy_table"), ("Cursor", "table_lack_0825"), ("SawyerTorque", "table_lack_0825")]
MIXED = True  # plus Sawyer + every furniture XML whose colliders the engine supports (BASELINE.json config 5, the mixed batch)


def write_feb(m, path):
    """the binary scene file of fe_create_from_file (fe_model + fe_scene), written through the library itself"""
    import ctypes as C

    from furniture_b200.engine import DEFAULT_LIB, build_scene
    from furniture_b200.engine_model import EngineModel

    if not os.path.exists(DEFAULT_LIB):
        return
    L = C.CDLL(DEFAULT_LIB)
    em = EngineModel(m)
    sc = build_scene(m, em)
    rc = L.fe_scene_file_write(path.encode(), C.byref(em.fm), C.c_size_t(C.sizeof(em.fm)), C.byref(sc), C.c_size_t(C.sizeof(sc)))
    assert rc == 0, path


def main():
    root = mjcf.default_assets_root()
    if root is None:
        print("asset tree not found; nothing compiled")
        return
    out = os.path.join(ROOT, "furniture_b200", "compiled")
    os.makedirs(out, exist_ok=True)
    scenes = list(SCENES)
    if MIXED:
        scenes += [("Sawyer", n) for n in mjcf.furniture_names(root) if ("Sawyer", n) not in scenes]
    skipped = []
    for agent, furn in scenes:
        xml, meta = mjcf.compose_agent(agent, furn, root)
        try:
            m = mjcf.compile_mjcf(xml, meta)
        except NotImplementedError as e:  # mesh colliders (7 of the 64 furniture models)
            skipped.append((furn, str(e)))
            continue
        path = os.path.join(out, "%s_%s.npz" % (agent, furn))
        m.save(path)
        write_feb(m, os.path.join(out, "%s_%s.feb" % (agent, furn)))
        print("wrote", path, "nq=%d nv=%d" % (m.nq, m.nv))
    for furn, why in skipped:
        print("skipped", furn, "--", why)


if __name__ == "__main__":
    main()
