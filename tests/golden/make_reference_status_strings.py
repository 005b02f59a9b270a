"""Generates tests/golden/reference_status_strings.json: what tests/test_status_strings_parity.py compares the drop-in with.

    python tests/golden/make_reference_status_strings.py [REVERSO_DIR]

  * `status_lines`, always: per mirrored method, the status lines the UNMODIFIED reference printed in the recorded scenario,
    read from tests/golden/reference_trace.json (make_reference_trace.py);
  * `templates` and `signatures`, when REVERSO_DIR (a checkout of kolenyo2099/revers-o) is given: the status-line templates and
    the argument lists of SimpleReverso, parsed from REVERSO_DIR/core_system.py.
The stored file was generated without a checkout at hand, so it holds `status_lines` only.
"""
import json
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
import test_status_strings_parity as P  # noqa: E402

# which UI output of the recorded scenario each mirrored method returned (tests/reference_harness.py: run_scenario)
TRACE_KEYS = {"create_database": ["build_regions", "build_direct"], "load_database": ["load", "load_missing", "load_direct"],
              "unlock_database": ["unlock"], "delete_database": ["delete"], "search_similar": ["searches"]}


def generate(reverso_dir=None):
    with open(os.path.join(HERE, "reference_trace.json"), encoding="utf-8") as f:
        ui = json.load(f)["ui"]
    lines = {}
    for m, keys in TRACE_KEYS.items():
        texts = [s["text"] for s in ui["searches"]] if keys == ["searches"] else [ui[k] for k in keys]
        lines[m] = sorted({ln for t in texts for ln in t.split("\n")
                           if ln.startswith(P.PREFIXES) and not any(w in ln for w in P.SKIP)})
    out = {"status_lines": lines}
    if reverso_dir:
        src = os.path.join(reverso_dir, "core_system.py")
        out["templates"] = {m: sorted(t) for m, t in P.templates(src).items()}
        out["signatures"] = {m: s for m, s in P.signatures(src).items() if m in P.SIGNATURE_METHODS}
    return out


if __name__ == "__main__":
    data = generate(sys.argv[1] if len(sys.argv) > 1 else None)
    with open(os.path.join(HERE, "reference_status_strings.json"), "w", encoding="utf-8") as f:
        json.dump(data, f, indent=1, ensure_ascii=False)
        f.write("\n")
    print({k: sum(map(len, v.values())) for k, v in data.items()})
