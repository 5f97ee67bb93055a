"""Builds the committed input fixtures from the reference's regression data.  The tests read only the .npz files;
this script is run by hand against a checkout of insight-platform/Similari:

  python tests/golden/make_fixtures.py <path to the Similari checkout>

  python/bugfixes/bug_vs_1/in/**/*.json  -> bug_vs_1.npz   (real 512-d re-id features, VisualSort; the reference
                                                             script asserts "a track id appears once per frame")
  python/bugfixes/github-84.py           -> github_84.npz  (two frames of thin oriented boxes, Sort IoU(0.3); the
                                                             reference script only has to survive them: issue #84)

Only DATA is extracted (numbers), no reference code.  Boxes are stored as float32 rows
(xc, yc, angle|NaN, aspect, height, confidence), the layout of sb200_predict_batch.
"""
import ast
import json
import pathlib
import sys

import numpy as np

REF = None   # <checkout>/python/bugfixes, set from the command line
OUT = pathlib.Path(__file__).parent


def bug_vs_1():
    # the script globs in/*.json (sorted): in-1.json, in-2.json; fixed-1/ holds the two frames of the follow-up report
    seqs = {"main": ["in-1.json", "in-2.json"], "fixed": ["fixed-1/bug_vs_1.json", "fixed-1/bug_vs_2.json"]}
    out = {}
    for name, files in seqs.items():
        for k, f in enumerate(files):
            objs = json.load(open(REF / "bug_vs_1" / "in" / f))
            boxes = np.array([[o["bbox"]["xc"], o["bbox"]["yc"],
                               np.nan if o["bbox"]["angle"] is None else o["bbox"]["angle"],
                               o["bbox"]["aspect"], o["bbox"]["height"], o["bbox"]["confidence"]] for o in objs], np.float32)
            feats = np.array([o["feature"] for o in objs], np.float32)
            qual = np.array([o["feature_quality"] for o in objs], np.float32)
            out[f"{name}_{k}_boxes"], out[f"{name}_{k}_features"], out[f"{name}_{k}_quality"] = boxes, feats, qual
    np.savez_compressed(OUT / "bug_vs_1.npz", **out)


def github_84():
    tree = ast.parse(open(REF / "github-84.py").read())
    frames = {}
    for node in tree.body:
        if isinstance(node, ast.Assign) and isinstance(node.targets[0], ast.Name) and node.targets[0].id.startswith("BOXES_"):
            rows = np.array(ast.literal_eval(node.value), np.float64)   # xc, yc, angle, aspect, height
            b = np.ones((len(rows), 6), np.float32)                     # Universal2DBox(...) default confidence 1.0
            b[:, :5] = rows.astype(np.float32)
            frames[node.targets[0].id.lower()] = b
    np.savez_compressed(OUT / "github_84.npz", **frames)


if __name__ == "__main__":
    if len(sys.argv) != 2:
        raise SystemExit(__doc__)
    REF = pathlib.Path(sys.argv[1]) / "python" / "bugfixes"
    bug_vs_1()
    github_84()
    for f in ("bug_vs_1.npz", "github_84.npz"):
        z = np.load(OUT / f)
        print(f, {k: z[k].shape for k in z.files})
