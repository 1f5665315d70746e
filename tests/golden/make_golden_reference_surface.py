"""Names the reference defines in the files of the hot path and its neighbouring stages, for
tests/test_reference_surface.py: every module-level function and every method of the classes the mirror package
stands in for.

    python tests/golden/make_golden_reference_surface.py <checkout of krg-nandu/monkey-pose>

writes reference_surface.json: {file: {class name, or "" for module level: {name: "line N"}}} and a "_provenance"
note.  The reference is Python 2 source; it is read as text, never imported.
"""
import json
import os
import re
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
PATH = os.path.join(HERE, "reference_surface.json")

# file -> the classes whose methods are listed ("" = the file's module-level functions)
SCOPES = {
    "hgru_module.py": ("", "ContextualCircuit"),
    "hgru_pose.py": ("model",),
    "train_cnn_networks_hgru.py": ("", "attn_model_struct"),
    "tf_monkeydetector.py": ("tfMonkeyDetector",),
    "pose_evaluation.py": ("",),
}

DEF = re.compile(r"^([ \t]*)def\s+(\w+)\s*\(", re.M)


def defs(src, cls=""):
    """{name: "line N"} of the functions defined at module level (cls "") or inside class `cls` of a source text."""
    def line(pos):
        return "line %d" % (src.count("\n", 0, pos) + 1)
    if not cls:
        return {m.group(2): line(m.start(2)) for m in DEF.finditer(src) if m.group(1) == ""}
    start = re.search(r"^class\s+%s\b.*$" % cls, src, re.M).end()
    nxt = re.search(r"^(class|def)\s+\w+", src[start:], re.M)
    end = start + nxt.start() if nxt else len(src)
    return {m.group(2): line(m.start(2)) for m in DEF.finditer(src, start, end) if m.group(1) != ""}


def extract(ref_dir):
    out = {"_provenance": "extracted from a checkout of the reference by make_golden_reference_surface.py"}
    for path, scopes in SCOPES.items():
        src = open(os.path.join(ref_dir, path)).read()
        out[path] = {cls: defs(src, cls) for cls in scopes}
    return out


if __name__ == "__main__":
    if len(sys.argv) != 2:
        sys.exit("usage: make_golden_reference_surface.py <checkout of krg-nandu/monkey-pose>")
    with open(PATH, "w") as f:
        json.dump(extract(sys.argv[1]), f, indent=1, sort_keys=True)
        f.write("\n")
    print("wrote", PATH)
