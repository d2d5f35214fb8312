"""Generates tests/golden/reference_imports.json: every import statement of the reference's SLAM modules that names one of
the packages this repository replaces (pygicp, diff_gaussian_rasterization, simple_knn), with the names it binds and the
attributes the module reads from them, found by parsing the reference's sources (nothing is executed or copied):
    python tests/golden/make_reference_imports_golden.py REFERENCE_TREE"""
import ast
import json
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
OURS = ("pygicp", "diff_gaussian_rasterization", "simple_knn")
MODULES = ("gaussian_renderer/__init__.py", "scene/gaussian_model.py", "mp_Tracker.py", "mp_Tracker_unlimit.py", "mp_Mapper.py",
           "gs_icp_slam.py", "gs_icp_slam_unlimit.py")


def scan(path):
    tree = ast.parse(open(path).read())
    found, aliases = [], {}
    for node in ast.walk(tree):
        if isinstance(node, ast.ImportFrom) and node.module and node.module.split(".")[0] in OURS:
            found.append({"module": node.module, "names": sorted(a.name for a in node.names)})
        elif isinstance(node, ast.Import):
            for a in node.names:
                if a.name.split(".")[0] in OURS:
                    aliases[a.asname or a.name] = a.name
                    found.append({"module": a.name, "names": []})
    for node in ast.walk(tree):  # attributes read from an imported module object: pygicp.FastGICP
        if isinstance(node, ast.Attribute) and isinstance(node.value, ast.Name) and node.value.id in aliases:
            rec = next(r for r in found if r["module"] == aliases[node.value.id])
            rec.setdefault("attributes", [])
            if node.attr not in rec["attributes"]:
                rec["attributes"].append(node.attr)
    for r in found:
        r.setdefault("attributes", [])
        r["attributes"].sort()
    return found


def main():
    ref = sys.argv[1]
    out = {m: scan(os.path.join(ref, m)) for m in MODULES if os.path.isfile(os.path.join(ref, m))}
    json.dump(out, open(os.path.join(HERE, "reference_imports.json"), "w"), indent=1, sort_keys=True)
    print(json.dumps(out, indent=1))


if __name__ == "__main__":
    main()
