#!/usr/bin/env python3
"""Regenerate tests/golden/*.json from the reference's own test expectations.

Needs a checkout of the reference crate (arroy) and is not part of the test run:
`python tests/golden/make_golden.py <path of the arroy checkout>`. It parses the *expected values* held by
the reference's tests — the insta `.snap` files under src/tests/snapshots/ and the inline
snapshots in src/tests/writer.rs / src/tests/reader.rs / src/tests/upgrade.rs — into small
JSON fixtures. No reference source code is copied; only golden numbers (node ids, child
ids, 4-decimal header/normal values, descendant id lists, query results).
"""
import json
import os
import re
import sys

REF = None   # the reference checkout, from the command line
OUT = os.path.dirname(os.path.abspath(__file__))

TREE_SPLIT = re.compile(
    r"Tree (\d+): SplitPlaneNormal\(SplitPlaneNormal<([a-z\-]+)> \{ left: (\d+), right: (\d+), normal: (.*) \}\)$")
TREE_DESC = re.compile(r"Tree (\d+): Descendants\(Descendants \{ descendants: \[(.*)\] \}\)$")
ITEM = re.compile(r"Item (\d+): Leaf\(Leaf \{ header: (\w+) \{ (.*?) \}, vector: \[(.*)\] \}\)$")
ROOT = re.compile(r"Root: Metadata \{ dimensions: (\d+), items: RoaringBitmap<(.*?)>, roots: \[(.*?)\], distance: \"(.*?)\" \}")
LEAF = re.compile(r"Leaf \{ header: (\w+) \{ (.*?) \}, vector: \[(.*)\] \}")


def parse_header(fields):
    out = {}
    for m in re.finditer(r"(\w+): \"(-?[\d\.a-zA-Z]+)\"", fields):
        out[m.group(1)] = m.group(2)
    return out


def parse_vec(s):
    vals = []
    truncated = False
    for tok in s.split(","):
        tok = tok.strip()
        if not tok:
            continue
        if tok.startswith('"'):
            truncated = True
            continue
        vals.append(tok)
    return vals, truncated


def parse_dump(lines):
    """Parse one `DatabaseHandle` dump (src/tests/mod.rs:28-91) -> dict."""
    db = {"tree": {}, "items": {}}
    for line in lines:
        line = line.strip()
        m = ROOT.match(line)
        if m:
            db["dimensions"] = int(m.group(1))
            db["items_desc"] = m.group(2)
            db["roots"] = [int(x) for x in m.group(3).split(",") if x.strip()]
            db["distance"] = m.group(4)
            continue
        m = TREE_SPLIT.match(line)
        if m:
            node = {"kind": "split", "left": int(m.group(3)), "right": int(m.group(4))}
            nm = LEAF.match(m.group(5))
            if nm:
                node["header"] = parse_header(nm.group(2))
                node["normal"], node["truncated"] = parse_vec(nm.group(3))
            else:
                node["normal"] = None
            db["tree"][m.group(1)] = node
            continue
        m = TREE_DESC.match(line)
        if m:
            db["tree"][m.group(1)] = {"kind": "descendants",
                                      "descendants": [int(x) for x in m.group(2).split(",") if x.strip()]}
            continue
        m = ITEM.match(line)
        if m:
            vec, trunc = parse_vec(m.group(4))
            db["items"][m.group(1)] = {"header": parse_header(m.group(3)), "vector": vec, "truncated": trunc}
    return db


def snap_file(name):
    with open(os.path.join(REF, "src/tests/snapshots", name)) as f:
        txt = f.read().split("---", 2)[2]
    return parse_dump(txt.splitlines())


def inline_snapshots(path):
    """Yield (line_number, [lines]) for every inline `@r#"..."#` / `@r###"..."###` / `@r"..."` block."""
    with open(os.path.join(REF, path)) as f:
        src = f.read()
    for m in re.finditer(r'@r(#*)"(.*?)"\1', src, re.S):
        line_no = src.count("\n", 0, m.start()) + 1
        yield line_no, m.group(2).splitlines()


def main():
    global REF
    if len(sys.argv) != 2 or not os.path.isdir(os.path.join(sys.argv[1], "src", "tests")):
        sys.exit("usage: make_golden.py <path of the arroy checkout>")
    REF = sys.argv[1]
    g = {}
    g["lot_of_random_points"] = snap_file("arroy__tests__writer__write_and_update_lot_of_random_points.snap")
    # second snapshot of the same test: only its *items* are used (even ids redrawn after the
    # first build), which pins how many words Writer::build takes from the user rng
    second = snap_file("arroy__tests__writer__write_and_update_lot_of_random_points-2.snap")
    g["lot_of_random_points_2_items"] = second["items"]
    g["lot_of_random_points_2"] = {k: v for k, v in second.items() if k != "items"}   # forest after the incremental update (10 roots)
    g["little_memory"] = snap_file("arroy__tests__writer__write_and_update_lot_of_random_points_with_little_memory.snap")
    # inline snapshots of src/tests/writer.rs, keyed by the line they start on
    inl = {}
    for line_no, lines in inline_snapshots("src/tests/writer.rs"):
        if any(l.strip().startswith("Root: Metadata") for l in lines):
            inl[str(line_no)] = parse_dump(lines)
    g["writer_inline"] = inl
    # query results of src/tests/reader.rs
    q = {}
    for line_no, lines in inline_snapshots("src/tests/reader.rs"):
        res = []
        for l in lines:
            m = re.match(r"\s*id\((\d+)\): distance\(([-\d\.eE]+)\)", l)
            if m:
                res.append([int(m.group(1)), float(m.group(2))])
        if res:
            q[str(line_no)] = res
    g["reader_inline"] = q
    # raw item vector printed at full precision in src/tests/upgrade.rs:117 (item 25 of the
    # 100x30 uniform dataset == draws 750..779 of StdRng::from_seed([42;32]))
    with open(os.path.join(REF, "src/tests/upgrade.rs")) as f:
        up = f.read()
    for item in (25,):
        m = re.search(r"item_vector\(&rtxn, %d\)\.unwrap\(\)\), @\"Some\(\[(.*?)\]\)\"" % item, up, re.S)
        if m:  # kept as strings: Rust prints the shortest round-trip repr of each f32
            g["upgrade_item%d" % item] = [x.strip() for x in m.group(1).split(",") if x.strip()]
    # src/tests/upgrade.rs:119-128: by_vector([0;30]) on the updated 100x30 dataset, full precision
    m = re.search(r"by_vector\(&rtxn, &\[0\.0; 30\]\).*?@r\"(.*?)\"", up, re.S)
    if m:
        g["upgrade_nns_zero"] = [[int(a), b] for a, b in re.findall(r"id\((\d+)\): distance\(([-\d\.eE]+)\)", m.group(1))]
    # src/tests/upgrade.rs: the two LMDB files the reference ships (written by arroy v0.6 through heed / LMDB / roaring) are
    # copied as binary fixtures; the post-upgrade dumps and the pre-upgrade query results are the goldens they are checked against
    import shutil
    for name in ("smol", "large"):
        shutil.copyfile(os.path.join(REF, "src/tests/assets/v0_6", name + ".mdb"), os.path.join(OUT, "v0_6_%s.mdb" % name))
    g["upgrade_large_dump"] = snap_file("arroy__tests__upgrade__large_upgrade_v0_6_to_v0_7-10.snap")
    for line_no, lines in inline_snapshots("src/tests/upgrade.rs"):
        if any(l.strip().startswith("Root: Metadata") for l in lines) and any("Version:" in l for l in lines):
            g["upgrade_smol_dump"] = parse_dump(lines)
    m = re.search(r"by_vector\(&rtxn, &\[1\.0, 0\.0\]\).*?@r\"(.*?)\"", up, re.S)
    if m:
        g["upgrade_smol_nns"] = [[int(a), b] for a, b in re.findall(r"id\((\d+)\): distance\(([-\d\.eE]+)\)", m.group(1))]
    # target_n_trees table — src/tests/writer.rs:14-79
    with open(os.path.join(REF, "src/tests/writer.rs")) as f:
        w = f.read()
    g["target_n_trees_src_lines"] = "src/tests/writer.rs:14-79"
    tbl = []
    for m in re.finditer(r"quick_target\((\d+), &b([\d_]+)\), @\"(\d+)\"", w):
        tbl.append([int(m.group(2).replace("_", "")), int(m.group(1)), int(m.group(3))])  # [n_items, dims, trees]
    g["target_n_trees"] = tbl
    with open(os.path.join(OUT, "reference_golden.json"), "w") as f:
        json.dump(g, f, indent=0, sort_keys=True)
    print("wrote", os.path.join(OUT, "reference_golden.json"),
          {k: (len(v) if hasattr(v, "__len__") else v) for k, v in g.items()})


if __name__ == "__main__":
    main()
