"""Record tests/golden/overlay_layout.json from an ICON checkout:

    python tests/golden/make_overlay_layout.py /path/to/ICON

The layout is the part of the checkout icon_b200.overlay depends on: for each module below, in source order, the
names it defines at top level and the `from ... import` statements between these modules.  Imports of other modules
(third-party packages, other lib.* modules) are left out: the overlay does not touch them.  tests/test_overlay_cpu.py
builds a stand-in checkout from this file, with a placeholder behind every recorded name.
"""
import ast
import json
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))

# apps/ICON.py and what it reaches through the overlay: the REPLACE and PATCH modules of icon_b200.overlay, the lib.net
# package that re-exports them, and lib.net.net_util (not patched; its names must stay the checkout's)
MODULES = ["apps.ICON", "lib.net", "lib.net.BasePIFuNet", "lib.net.HGPIFuNet", "lib.net.voxelize",
           "lib.common.seg3d_lossless", "lib.common.train_util", "lib.dataset.mesh_util", "lib.net.NormalNet",
           "lib.net.MLP", "lib.net.HGFilters", "lib.net.FBNet", "lib.net.VE", "lib.net.net_util"]


def module_path(root, name):
    p = os.path.join(root, *name.split("."))
    return (os.path.join(p, "__init__.py"), True) if os.path.isdir(p) else (p + ".py", False)


def resolve(name, is_pkg, node):
    if node.level == 0:
        return node.module
    base = (name if is_pkg else name.rpartition(".")[0]).split(".")
    base = base[:len(base) - (node.level - 1)]
    return ".".join(base + ([node.module] if node.module else []))


def layout(root, name):
    path, is_pkg = module_path(root, name)
    out = []
    for node in ast.parse(open(path).read(), path).body:
        if isinstance(node, ast.ImportFrom):
            src = resolve(name, is_pkg, node)
            if src in MODULES:
                out.append(["import", src, [a.name for a in node.names]])
        elif isinstance(node, (ast.FunctionDef, ast.AsyncFunctionDef)):
            out.append(["def", node.name])
        elif isinstance(node, ast.ClassDef):
            out.append(["class", node.name])
        elif isinstance(node, (ast.Assign, ast.AnnAssign)):
            for t in (node.targets if isinstance(node, ast.Assign) else [node.target]):
                if isinstance(t, ast.Name):
                    out.append(["value", t.id])
    return {"package": is_pkg, "body": out}


def main(root):
    data = {"source": "ICON (YuliangXiu/ICON) checkout: module layout only, no code",
            "modules": {m: layout(root, m) for m in MODULES}}
    with open(os.path.join(HERE, "overlay_layout.json"), "w") as f:
        json.dump(data, f, indent=1)
        f.write("\n")


if __name__ == "__main__":
    main(sys.argv[1])
