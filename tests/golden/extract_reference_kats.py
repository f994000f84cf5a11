#!/usr/bin/env python3
"""Mechanical provenance of tests/golden/reference_kats.json.

The reference (pluto/ronkathon) is Rust, so its known-answer vectors were transcribed by hand.  This script ties
the transcription back to the Rust sources instead of trusting it:

  * the rstest `#[case(...)]` tables of src/algebra/field/prime/arithmetic.rs (add, sub, mul, field_pow,
    multiplicative_inverse, halve) are PARSED and must contain every entry of the JSON's field section
    (`--write` regenerates that section from the parse, adding nothing by hand);
  * every other integer vector of the JSON (polynomial, GF(101²), curve, kzg, Reed–Solomon sections) is located
    in the cited source file as a contiguous run of its numeric literals, after stripping the type parameters
    (`PlutoBaseField`, const-generic sizes, `usize` suffixes) — a vector that cannot be found is an error;
  * sections the JSON itself marks as derived (config1_extra: computed with the reference's schoolbook algorithm,
    reed_solomon_decode: round trips) are listed as derived, not searched.

A run against a reference checkout stores what it parsed and located in tests/golden/reference_kat_sources.json:
the case tables, and for every other vector the first run of literals in the cited files that equals it, with the
file:line of that run's first literal.  The search is by value only, so a short vector such as [1, 1, 0] may be
matched by unrelated literals that precede the test which states it.  Without a checkout the same checks run against
that record, so the suite keeps the comparison on any machine.

Run:  python tests/golden/extract_reference_kats.py                          (check against the stored record)
      python tests/golden/extract_reference_kats.py --reference DIR          (check against the sources in DIR
                                                                              and rewrite the record)
      python tests/golden/extract_reference_kats.py --reference DIR --write  (also rewrite the parsed sections)
Exit code 1 on any unlocated vector."""
from __future__ import annotations

import argparse
import json
import os
import re
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
JSON_PATH = os.path.join(HERE, "reference_kats.json")
RECORD_PATH = os.path.join(HERE, "reference_kat_sources.json")
REFERENCE = "pluto/ronkathon @ 86de329d7fe873d78374f266fde8c351c8cb72ae"
FIELD_FILE = "src/algebra/field/prime/arithmetic.rs"
FIELD_OF = {"PlutoScalarField": 17, "PlutoBaseField": 101}


def rstest_cases(src: str, fn_name: str):
    """The `#[case(...)]` lines directly above `fn <fn_name>`; each case → list of (modulus | None, int)."""
    m = re.search(r"((?:\s*(?://[^\n]*|#\[[^\n]*\])\n)+)\s*fn " + re.escape(fn_name) + r"\b", src)
    assert m, f"fn {fn_name} not found"
    cases = []
    for line in m.group(1).splitlines():
        line = line.strip()
        if not line.startswith("#[case("):
            continue
        toks = re.findall(r"(Pluto(?:Scalar|Base)Field)::new\((\d+)\)|(?<![\w:])(\d+)(?![\w:])", line)
        vals = []
        for fld, v, bare in toks:
            vals.append((FIELD_OF[fld], int(v)) if fld else (None, int(bare)))
        cases.append(vals)
    return cases


def field_section_from_source(src: str):
    out = {}
    for key, fn in (("add", "add"), ("sub", "sub"), ("mul", "mul")):
        out[key] = [[c[0][0], c[0][1], c[1][1], c[2][1]] for c in rstest_cases(src, fn)]
    out["pow"] = [[c[0][0], c[0][1], c[1][1], c[2][1]] for c in rstest_cases(src, "field_pow")]
    inv = rstest_cases(src, "multiplicative_inverse")
    out["inverse"] = [[c[0][0], c[0][1], c[1][1]] for c in inv if c[0][1] != 0]       # the 0 cases are #[should_panic]
    out["inverse_of_zero_panics"] = sorted({c[0][0] for c in inv if c[0][1] == 0})
    out["halve"] = [[c[0][0], c[0][1], c[1][1]] for c in rstest_cases(src, "halve")]
    return out


def number_stream(src: str):
    """(value, line) of the numeric literals of a Rust source in order, without const-generic sizes / type
    parameters / suffixes.  Every rewrite keeps the line count, so `line` is where the literal is written."""
    def blank(m):
        return "\n" * m.group(0).count("\n")

    def repeat(m):   # [x; n] → [x, x, …]
        return "[" + ", ".join([m.group(1).replace("\n", " ")] * int(m.group(2))) + "]" + blank(m)

    src = re.sub(r"//[^\n]*", "", src)
    src = re.sub(r"::<\{[^}]*\}>", blank, src)                # PrimeField::<{ PlutoPrime::Base as usize }>
    src = re.sub(r"::<[^>]*>", blank, src)                    # Polynomial::<Monomial, PlutoBaseField, 4>
    src = re.sub(r"\[([^\[\];]+);\s*(\d+)\]", repeat, src)
    src = re.sub(r"(?<=\w)\[\s*\d+\s*\]", blank, src)         # index expressions: arr[0], data[1]
    src = re.sub(r"<[A-Za-z_][\w, ]*\d+\s*>", blank, src)     # Polynomial<Monomial, PlutoBaseField, 4>
    src = src.replace("::ZERO", "::new(0)").replace("::ONE", "::new(1)")
    out, line, pos = [], 1, 0
    for m in re.finditer(r"(?<![\w.])(\d+)(?:usize|u32|u64|i32)?(?![\w.])", src):
        line += src.count("\n", pos, m.start())
        pos = m.start()
        out.append((int(m.group(1)), line))
    return out


def find_run(stream, vec):
    """Line of the first literal of a contiguous run equal to `vec`, or None."""
    n = len(vec)
    values = [v for v, _ in stream]
    for i, v in enumerate(values):
        if v == vec[0] and values[i:i + n] == vec:
            return stream[i][1]
    return None


class Sources:
    """A reference checkout: parses the case tables and searches the cited files."""

    def __init__(self, root: str):
        self.root, self.streams = root, {}

    def read(self, rel):
        with open(os.path.join(self.root, rel)) as f:
            return f.read()

    def field_cases(self):
        return field_section_from_source(self.read(FIELD_FILE))

    def locate(self, vec, files):
        for rel in files:
            if rel not in self.streams:
                self.streams[rel] = number_stream(self.read(rel))
            line = find_run(self.streams[rel], vec)
            if line is not None:
                return rel, line
        return None


class Record:
    """What an earlier run against a reference checkout parsed and located (reference_kat_sources.json)."""

    def __init__(self, path: str):
        with open(path) as f:
            self.data = json.load(f)

    def field_cases(self):
        return self.data["field_cases"]

    def locate(self, vec, files):
        for e in self.data["located"]:
            if e["file"] in files and e["values"] == vec:
                return e["file"], e["line"]
        return None


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--reference", metavar="DIR", help="a checkout of the reference; without it, the stored record")
    ap.add_argument("--write", action="store_true", help="rewrite the field section of reference_kats.json")
    args = ap.parse_args()
    if args.write and not args.reference:
        ap.error("--write needs --reference")
    src = Sources(args.reference) if args.reference else Record(RECORD_PATH)
    with open(JSON_PATH) as f:
        kats = json.load(f)
    problems, found, derived = [], [], []

    # ---- field section: parsed tables -------------------------------------------------------------------------
    parsed = src.field_cases()
    located = 0
    for key, rows in parsed.items():
        have = kats["field"].get(key)
        if have is None:
            continue
        for row in have:
            if row not in rows:
                problems.append(f"field.{key}: {row} is not a #[case] of the reference")
            else:
                located += 1
    if args.write:
        for key, rows in parsed.items():
            kats["field"][key] = rows

    # ---- every other vector: located in the cited file ----------------------------------------------------------
    def locate(label, forms, files):
        forms = [[int(v) for v in form] for form in forms]
        for form in forms:
            hit = src.locate(form, files)
            if hit is not None:
                found.append({"what": label, "file": hit[0], "line": hit[1], "values": form})
                return
        problems.append(f"{label}: none of {forms} found in {files}")

    poly_files = ["src/polynomial/tests.rs", "src/polynomial/arithmetic.rs"]
    for key, v in kats["polynomial"].items():
        if isinstance(v, list) and v and all(isinstance(x, int) for x in v):
            locate(f"polynomial.{key}", [v], poly_files)
    gf_file = ["src/algebra/field/extension/gf_101_2.rs"]
    for op, rows in kats["gf101_2"].items():
        if op == "src":
            continue
        for row in rows:
            for pair in row:
                locate(f"gf101_2.{op}", [pair], gf_file)
    curve_files = ["src/curve/pluto_curve.rs", "src/kzg/tests.rs", "src/kzg/setup.rs"]
    pts = [kats["curve"]["G1"], kats["curve"]["G2"], kats["curve"]["two_G2"], kats["curve"]["off_curve"]]
    pts += list(kats["curve"]["multiples_of_G1"].values()) + kats["kzg"]["g1srs"] + kats["kzg"]["g2srs"]
    for p in pts:
        # base-field points are written (x0, y0), extension points with all four coordinates in either order
        x0, x1, y0, y1 = p
        forms = [[x0, y0]] if x1 == 0 and y1 == 0 else [[x0, x1, y0, y1], [x0, y0, y1], [x0, y1], [x0, 0, 0, y1]]
        locate(f"point {p}", forms, curve_files)
    for c in kats["kzg"]["commit"]:
        locate("kzg.commit.coeffs", [c["coeffs"]], ["src/kzg/tests.rs"])
    rs = kats["reed_solomon"]
    for key in ("msg", "x", "y"):
        locate(f"reed_solomon.{key}", [rs[key]], ["src/codes/reed_solomon.rs"])
    for key in ("config1_extra", "reed_solomon_decode"):
        if key in kats:
            derived.append(key)
    located += len(found)

    if args.write:
        with open(JSON_PATH, "w") as f:
            json.dump(kats, f, indent=1)
            f.write("\n")
    if args.reference and not problems:
        record = {"_comment": f"Written by extract_reference_kats.py from {REFERENCE}: the parsed #[case] tables "
                              f"of {FIELD_FILE}, and for each other vector of reference_kats.json the first "
                              "matching literal run in the cited files (file:line of its first literal).",
                  "field_cases": parsed, "located": found}
        with open(RECORD_PATH, "w") as f:
            json.dump(record, f, indent=1)
            f.write("\n")
    print(json.dumps({"located": located, "derived_sections": derived, "problems": problems}, indent=1))
    return 1 if problems else 0


if __name__ == "__main__":
    sys.exit(main())
