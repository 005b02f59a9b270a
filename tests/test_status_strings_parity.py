"""Boundary parity of the error/status-string convention (SURVEY.md §8b) between the reference's `SimpleReverso` and
revers_o_b200/core_system.py, against tests/golden/reference_status_strings.json (tests/golden/make_reference_status_strings.py):
  * `status_lines`: every status line the UNMODIFIED reference printed in the recorded scenario (tests/golden/reference_trace.json)
    must be produced by a template of the same method here;
  * `templates` / `signatures` (stored when the file is generated from a revers-o checkout): every status-line template of the
    reference's mirrored methods exists here character for character (f-string holes aside), and the mirrored methods take the
    same arguments with the same defaults.
Checkpoint messages are excluded (dead code in the reference, SURVEY.md F6)."""
import ast
import json
import os
import re

import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
GOLDEN = os.path.join(HERE, "golden", "reference_status_strings.json")
OURS = os.path.join(os.path.dirname(HERE), "revers_o_b200", "core_system.py")
METHODS = ["load_database", "delete_database", "unlock_database", "create_database", "search_similar"]
SIGNATURE_METHODS = ["load_database", "delete_database", "unlock_database", "list_databases", "detect_regions", "extract_embeddings",
                     "process_image_direct_pe", "request_stop", "create_database", "search_similar", "visualize_detections"]
PREFIXES = ("❌", "✅", "⚠️", "ℹ️", "🎯", "📦", "💾", "🔄", "📊", "📁", "📂", "🔧", "🛑", "🔍", "\n📊", "\n\n⏸️")
SKIP = ("checkpoint", "Resuming", "already processed", "Error loading/processing image", "Image not found")


def _class(path):
    tree = ast.parse(open(path, encoding="utf-8").read())
    return [n for n in tree.body if isinstance(n, ast.ClassDef) and n.name == "SimpleReverso"][0]


def templates(path):
    """method -> status-line templates ("{}" for each f-string hole) of SimpleReverso in the source file `path`."""
    out = {}
    for fn in [n for n in _class(path).body if isinstance(n, ast.FunctionDef) and n.name in METHODS]:
        found = set()
        for node in ast.walk(fn):
            if isinstance(node, ast.JoinedStr):
                text = "".join(v.value if isinstance(v, ast.Constant) else "{}" for v in node.values)
            elif isinstance(node, ast.Constant) and isinstance(node.value, str):
                text = node.value
            else:
                continue
            if text.startswith(PREFIXES) and not any(w in text for w in SKIP):
                found.add(text)
        out[fn.name] = found
    return out


def signatures(path):
    """method -> [argument names, defaults] of SimpleReverso in the source file `path`."""
    out = {}
    for fn in [n for n in _class(path).body if isinstance(n, ast.FunctionDef)]:
        a = fn.args
        out[fn.name] = [[x.arg for x in a.args], [ast.unparse(d).replace("'", '"') for d in a.defaults]]
    return out


@pytest.fixture(scope="module")
def golden():
    with open(GOLDEN, encoding="utf-8") as f:
        return json.load(f)


def test_every_reference_status_line_exists_in_the_drop_in(golden):
    ours = templates(OURS)
    # a printed line is covered when one line of a template here matches it in full, each hole standing for any text
    patterns = {m: [re.compile(".+?".join(map(re.escape, piece.split("{}")))) for t in ours.get(m, ()) for piece in t.split("\n") if piece]
                for m in METHODS}
    assert set(golden["status_lines"]) == set(METHODS)
    unmatched = {m: [line for line in lines if not any(p.fullmatch(line) for p in patterns[m])]
                 for m, lines in golden["status_lines"].items()}
    assert not any(unmatched.values()), unmatched
    if "templates" in golden:
        missing = {m: sorted(set(golden["templates"][m]) - ours.get(m, set())) for m in METHODS
                   if set(golden["templates"].get(m, ())) - ours.get(m, set())}
        assert not missing, missing


def test_mirrored_method_signatures_match_the_reference(golden):
    if "signatures" not in golden:
        pytest.skip("reference_status_strings.json holds no signatures: generate it from a revers-o checkout "
                    "(tests/golden/make_reference_status_strings.py REVERSO_DIR)")
    ref, ours = golden["signatures"], signatures(OURS)
    for m in SIGNATURE_METHODS:
        assert m in ours, m
        assert ours[m] == ref[m], (m, ours[m], ref[m])
