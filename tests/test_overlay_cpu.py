"""The drop-in boundary: with icon_b200.overlay installed on an ICON checkout, the HGPIFuNet / Seg3dLossless /
query_func / get_visibility / clean_mesh names apps/ICON.py imports are the icon_b200 objects, and every other
`lib.*` name it uses is still the checkout's.

The checkout is a stand-in built from tests/golden/overlay_layout.json (recorded from YuliangXiu/ICON by
tests/golden/make_overlay_layout.py): the same modules, the same top-level names in the same order, the same
`from ... import` statements between them, with a placeholder behind every name.  A module the overlay replaces
raises when executed, so importing it proves it never runs.  Runs on the CPU."""
import json
import os
import subprocess
import sys
import textwrap

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

SCRIPT = r'''
import os, sys
CHECKOUT, ROOT = sys.argv[1], sys.argv[2]
sys.path.insert(0, ROOT)

import icon_b200.overlay as OV
OV.install(CHECKOUT)

import apps.ICON as A
import lib.common.train_util as TU, lib.dataset.mesh_util as MU, lib.net as LN
import icon_b200.net, icon_b200.engine, icon_b200.encoders, icon_b200.visibility, icon_b200.mesh
assert A.__file__.startswith(CHECKOUT) and TU.__file__.startswith(CHECKOUT) and MU.__file__.startswith(CHECKOUT)
for name in ("lib.net.HGPIFuNet", "lib.common.seg3d_lossless"):
    assert sys.modules[name].__icon_b200_overlay__ == "replace", name
assert A.HGPIFuNet is icon_b200.net.HGPIFuNet and LN.HGPIFuNet is icon_b200.net.HGPIFuNet
assert LN.NormalNet is icon_b200.encoders.NormalNet and LN.VolumeEncoder is icon_b200.encoders.VolumeEncoder
assert A.Seg3dLossless is icon_b200.engine.Seg3dLossless
assert A.query_func is icon_b200.net.query_func and TU.query_func is icon_b200.net.query_func
assert A.get_visibility is icon_b200.visibility.get_visibility
assert A.clean_mesh is icon_b200.mesh.clean_mesh and MU.clean_mesh is icon_b200.mesh.clean_mesh
# names of the patched modules that are NOT on the accelerated path are still the checkout's own objects
for name in ("SMPLX", "update_mesh_shape_prior_losses", "load_checkpoint", "cal_sdf_batch", "feat_select", "remesh"):
    assert getattr(MU, name).__module__ == "lib.dataset.mesh_util", name
for name in ("batch_mean", "accumulate", "calc_error", "tf_log_convert", "bar_log_convert", "export_cfg"):
    assert getattr(TU, name).__module__ == "lib.common.train_util", name
    assert getattr(A, name) is getattr(TU, name), name             # `from lib.common.train_util import *` still complete
assert TU.get_visibility is icon_b200.visibility.get_visibility    # train_util's own get_visibility as well
import lib.net.FBNet as FB, lib.net.net_util as NU
assert FB.LocalEnhancer.__module__ == "lib.net.FBNet" and NU.VGGLoss.__module__ == "lib.net.net_util"
assert isinstance(FB.define_G(6, 3, 64, "global", 4, 9, 1, 3, "instance"), icon_b200.encoders.GlobalGenerator)
assert FB.define_G(6, 3, 64, "local", 4, 9, 1, 3, "instance") == ("lib.net.FBNet", "define_G")
print("OVERLAY_OK")
'''


def write_checkout(root, layout, replaced):
    """One .py file per recorded module; `def` / `class` / value names become placeholders whose value (or
    __module__) names the module that defined them."""
    for name, mod in layout["modules"].items():
        parts = name.split(".")
        path = os.path.join(root, *parts) + ("/__init__.py" if mod["package"] else ".py")
        os.makedirs(os.path.dirname(path), exist_ok=True)
        for i in range(1, len(parts)):                 # parent packages that were not recorded
            init = os.path.join(root, *parts[:i], "__init__.py")
            if not os.path.exists(init):
                open(init, "w").close()
        if name in replaced:
            lines = [f"raise ImportError('{name} is replaced by icon_b200.overlay and must not run')"]
        else:
            lines = []
            for entry in mod["body"]:
                kind, n = entry[0], entry[1]
                if kind == "import":
                    lines.append(f"from {n} import {', '.join(entry[2])}")
                elif kind == "def":
                    lines.append(f"def {n}(*args, **kwargs):\n    return ({name!r}, {n!r})")
                elif kind == "class":
                    lines.append(f"class {n}:\n    pass")
                else:
                    lines.append(f"{n} = ({name!r}, {n!r})")
        with open(path, "w") as f:
            f.write("\n".join(lines) + "\n")


def test_overlay_on_recorded_icon_layout(tmp_path, golden_dir):
    from icon_b200 import overlay
    layout = json.load(open(os.path.join(golden_dir, "overlay_layout.json")))
    replaced, patched = set(overlay._replacements()), set(overlay._patches())
    assert (replaced | patched) <= set(layout["modules"])
    checkout = tmp_path / "ICON"
    write_checkout(str(checkout), layout, replaced)
    script = tmp_path / "overlay_check.py"
    script.write_text(textwrap.dedent(SCRIPT))
    env = dict(os.environ, PYTHONPATH="")
    r = subprocess.run([sys.executable, str(script), str(checkout), ROOT], capture_output=True, text=True, timeout=600,
                       env=env, cwd=str(tmp_path))
    assert r.returncode == 0, r.stdout[-3000:] + "\n" + r.stderr[-6000:]
    assert "OVERLAY_OK" in r.stdout
