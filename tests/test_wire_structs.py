"""The wire / status structs against the reference's own DECLARATIONS (tests/golden/wire_structs.json, extracted from the
Go source by tests/golden/make_wire_structs.py): field names, order, Go types and omitempty flags.

No reference test reads a request body, so the emitted bytes stay "parity unpinned" (SURVEY.md §8c) — but what
encoding/json does with a struct is determined by its declaration, and THAT is held here mechanically: the product's
emitters must produce exactly the declared keys in the declared order (omitempty fields only when non-empty), and the
reply-struct descriptions the decoders walk (csrc/gotypes.cpp, twin oracle/go_decode.py) must equal the declarations."""
import hashlib
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FIX = json.load(open(os.path.join(ROOT, "tests", "golden", "wire_structs.json")))
FM = ["internal/cdi/fti/fm/api/scale_up.go", "internal/cdi/fti/fm/api/scale_down.go", "internal/cdi/fti/fm/api/get.go", "internal/cdi/fti/fm/api/common.go"]
CM = ["internal/cdi/fti/cm/client.go", "internal/cdi/fti/cm/api/machine.go"]
SUNFISH = ["internal/cdi/sunfish/client.go"]
CRD = ["api/v1alpha1/composableresource_types.go", "api/v1alpha1/composabilityrequest_types.go"]
PRIM = {"string": "string", "int": "int", "int64": "int64", "bool": "bool"}


def find(files, name):
    for f in files:
        if name in FIX[f]:
            return FIX[f][name]["fields"]
    raise KeyError(name)


def test_fixture_is_what_the_reference_declares():
    """wire_structs.json is byte for byte what make_wire_structs.py extracted from the reference's Go source: the SHA-256
    the extraction recorded beside it (wire_structs.json.sha256; the script's --check re-extracts and compares both)."""
    with open(os.path.join(ROOT, "tests", "golden", "wire_structs.json"), "rb") as f:
        got = hashlib.sha256(f.read()).hexdigest()
    with open(os.path.join(ROOT, "tests", "golden", "wire_structs.json.sha256")) as f:
        assert f.read().split() == [got, "wire_structs.json"]


def walk_emitted(files, struct, pairs, path=""):
    """pairs: [(key, value)] of one emitted JSON object, in emitted order; value objects are lists of pairs too."""
    decl = [f for f in find(files, struct) if "json" in f]
    allowed = [f["json"] for f in decl]
    keys = [k for k, _ in pairs]
    assert [k for k in allowed if k in keys] == keys, (path + struct, "emitted", keys, "declared", allowed)    # declared order, nothing foreign
    for f in decl:
        if f["json"] not in keys:
            assert f["omitempty"], (path + struct, f["json"], "is not omitempty and must be present")
    for k, v in pairs:
        f = next(x for x in decl if x["json"] == k)
        t = f["type"]
        elem = t[2:] if t.startswith("[]") else t
        if t.startswith("[]"):
            assert isinstance(v, list) and not (v and isinstance(v[0], tuple)), (path, k, "must be an array")
            items = v
        else:
            items = [v]
        for it in items:
            if elem in PRIM or elem.startswith("map[") or elem.startswith("*"):
                assert not isinstance(it, list) or elem.startswith("map[") or elem.startswith("*") or it == [], (path, k, elem, it)
                if elem == "string":
                    assert isinstance(it, str), (path, k)
                elif elem in ("int", "int64"):
                    assert isinstance(it, int) and not isinstance(it, bool), (path, k)
                elif elem == "bool":
                    assert isinstance(it, bool), (path, k)
            else:
                walk_emitted(files, elem, it, path + struct + "." + k + "/")


def ordered(text):
    return json.loads(text, object_pairs_hook=lambda p: p)


def test_request_bodies_follow_the_declarations(cro):
    walk_emitted(FM, "ScaleUpBody", ordered(cro.emit_fm_scale_up("tenant", "mach", "gpu", "NVIDIA-B200")))
    walk_emitted(FM, "ScaleDownBody", ordered(cro.emit_fm_scale_down("tenant", "mach", "gpu", "res-uuid")))
    walk_emitted(CM, "scaleUpRequestBody", ordered(cro.emit_cm_scale_up("spec", 2)))
    walk_emitted(CM, "scaleDownRequestBody", ordered(cro.emit_cm_scale_down("spec", 1, "GPU-x")))
    walk_emitted(SUNFISH, "CompositionRequest", ordered(cro.emit_sunfish_request("worker-0", 1, "GPU", "NVIDIA-A100-PCIE-40GB")))


def test_status_structs_follow_the_declarations(cro):
    for args in (("Online", "", "GPU-x", "res"), ("Attaching", "boom", "", ""), ("", "", "", "")):
        walk_emitted(CRD, "ComposableResourceStatus", ordered(cro.emit_status_json(*args)))
    for args in (("Online", "GPU-x", "res", "worker-0", ""), ("Attaching", "", "", "", "boom"), ("", "", "", "", "")):
        walk_emitted(CRD, "ScalarResourceStatus", ordered(cro.emit_scalar_status_json(*args)))
    # omitempty as declared: `state` always, the rest only when non-empty
    assert cro.emit_status_json("", "", "", "") == '{"state":""}'
    assert [k for k, _ in ordered(cro.emit_status_json("Online", "e", "d", "c"))] == ["state", "error", "device_id", "cdi_device_id"]


def go_type_of(files, decl_type):
    if decl_type in PRIM:
        return decl_type
    if decl_type.startswith("[]"):
        return "[]" + go_type_of(files, decl_type[2:])
    return "api." + decl_type


def check_described(files, struct, desc, path=""):
    decl = [f for f in find(files, struct) if "json" in f]
    assert desc["struct"] == struct and desc["type"] == "api." + struct, (path, desc["type"])
    assert [f["json"] for f in desc["fields"]] == [f["json"] for f in decl], (path + struct, "field order")
    for got, want in zip(desc["fields"], decl):
        assert got["of"]["type"] == go_type_of(files, want["type"]), (path + struct, want["json"], got["of"]["type"], want["type"])
        inner = got["of"].get("elem", got["of"])
        if "struct" in inner:
            check_described(files, inner["struct"], inner, path + struct + ".")


def test_reply_struct_descriptions_equal_the_declarations(cro):
    """csrc/gotypes.cpp — what FMScaleUpResponseToIDs / FMCheckResource / CMCheckAddingResources decode INTO."""
    check_described(FM, "ScaleUpResponse", cro.describe_wire_type("FMScaleUpResponse"))
    check_described(FM, "GetMachineResponse", cro.describe_wire_type("FMGetMachineResponse"))
    check_described(["internal/cdi/fti/cm/api/machine.go"], "MachineData", cro.describe_wire_type("CMMachineData"))


def test_oracle_type_descriptions_equal_the_declarations():
    """oracle/go_decode.py:TYPES — the twin the typed-decode fuzz uses as its oracle."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import go_decode as gd

    def check(files, struct, t, path=""):
        assert t[0] == "struct" and t[1] == struct, (path, t[:2])
        decl = {f["json"]: f["type"] for f in find(files, struct) if "json" in f}
        assert set(t[2]) == set(decl), (path + struct, sorted(set(t[2]) ^ set(decl)))
        for tag, ft in t[2].items():
            want = decl[tag]
            if want in PRIM:
                assert ft == want, (path + struct, tag, ft, want)
            elif want.startswith("[]"):
                assert ft[0] == "slice", (path + struct, tag)
                if want[2:] in PRIM:
                    assert ft[1] == want[2:]
                else:
                    check(files, want[2:], ft[1], path + struct + ".")
            else:
                check(files, want, ft, path + struct + ".")
    check(FM, "ScaleUpResponse", gd.TYPES["api.ScaleUpResponse"])
    check(FM, "GetMachineResponse", gd.TYPES["api.GetMachineResponse"])
    check(["internal/cdi/fti/cm/api/machine.go"], "MachineData", gd.TYPES["api.MachineData"])
