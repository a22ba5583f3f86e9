"""Extracts the reference's wire / status struct DECLARATIONS — field order, Go types, json tags, omitempty — from its Go
source and writes tests/golden/wire_structs.json.  Run from the repo root (needs /root/reference):

    python tests/golden/make_wire_structs.py            # (re)write the fixture
    python tests/golden/make_wire_structs.py --check    # exit 1 if the committed fixture differs from the reference

No reference test reads a request body (SURVEY.md §8c: "parity unpinned" for the emitted bytes), so what CAN be pinned
mechanically is pinned here: the names, the order and the omitempty flags encoding/json walks are the declarations'
— tests/test_wire_structs.py holds the product's emitters and the oracle's type descriptions against them."""
import hashlib
import json
import os
import re
import sys

REF = "/root/reference"
FILES = ["internal/cdi/fti/fm/api/common.go", "internal/cdi/fti/fm/api/scale_up.go", "internal/cdi/fti/fm/api/scale_down.go",
         "internal/cdi/fti/fm/api/get.go", "internal/cdi/fti/cm/api/machine.go", "internal/cdi/fti/cm/client.go",
         "internal/cdi/sunfish/client.go", "internal/cdi/client.go", "api/v1alpha1/composableresource_types.go",
         "api/v1alpha1/composabilityrequest_types.go"]
ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
OUT = os.path.join(ROOT, "tests", "golden", "wire_structs.json")

STRUCT = re.compile(r"^type\s+(\w+)\s+struct\s*\{(.*?)^\}", re.S | re.M)
FIELD = re.compile(r"^\s*(\w+)\s+([\w\.\[\]\*]+)\s*(?:`([^`]*)`)?\s*(?://.*)?$")


def extract():
    out = {}
    for rel in FILES:
        src = open(os.path.join(REF, rel)).read()
        structs = {}
        for m in STRUCT.finditer(src):
            name, body = m.group(1), m.group(2)
            line = src.count("\n", 0, m.start()) + 1
            fields = []
            for raw in body.split("\n"):
                raw = raw.rstrip()
                if not raw.strip() or raw.strip().startswith("//"):
                    continue
                f = FIELD.match(raw)
                if not f:
                    # embedded field (metav1.TypeMeta `json:",inline"`) or a multi-line comment: record it verbatim
                    fields.append({"raw": raw.strip()})
                    continue
                go_name, go_type, tag = f.group(1), f.group(2), f.group(3) or ""
                jm = re.search(r'json:"([^"]*)"', tag)
                if not jm:
                    continue
                parts = jm.group(1).split(",")
                if parts[0] == "-":
                    continue
                fields.append({"go": go_name, "type": go_type, "json": parts[0] or go_name, "omitempty": "omitempty" in parts[1:]})
            structs[name] = {"line": line, "fields": fields}
        out[rel] = structs
    return out


if __name__ == "__main__":
    got = extract()
    text = json.dumps(got, indent=1, sort_keys=True) + "\n"
    # the seal tests/test_wire_structs.py holds the fixture to where the reference tree is not at hand
    seal = hashlib.sha256(text.encode()).hexdigest() + "  wire_structs.json\n"
    if "--check" in sys.argv:
        same = all(os.path.exists(p) and open(p).read() == t for p, t in ((OUT, text), (OUT + ".sha256", seal)))
        print("wire_structs.json", "matches the reference" if same else "DIFFERS from the reference")
        sys.exit(0 if same else 1)
    open(OUT, "w").write(text)
    open(OUT + ".sha256", "w").write(seal)
    print("wrote", sum(len(v) for v in got.values()), "structs from", len(got), "files")
