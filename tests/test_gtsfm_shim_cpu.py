"""CPU: the B200 plugins against GTSfM's plugin API, recorded from the reference in tests/golden/gtsfm_bases.json
(oracle/make_golden.py golden_gtsfm_bases): module paths, abstract methods and their parameters, what each base's __init__
stores, and the verifier repr that keys GTSfM's two-view cache.

Two branches of gtsfm_b200/gtsfm_api.py are checked against that record:
  * without GTSfM (this environment): the mirrors have the reference's abstract methods, parameters and stored state;
  * with GTSfM importable (`HAVE_GTSFM`): a `gtsfm` package with the recorded layout, generated into a temporary directory,
    is picked up and the plugins subclass its bases.  Run in a subprocess so that package never leaks into the suite."""
import inspect
import json
import pickle
import subprocess
import sys
import textwrap
from pathlib import Path

import pytest

from gtsfm_b200 import gtsfm_api, synthetic as syn

ROOT = Path(__file__).resolve().parent.parent


@pytest.fixture(scope="module")
def api(golden_dir):
    return json.loads((golden_dir / "gtsfm_bases.json").read_text())


def params(f):
    return [[p.name, None if p.default is p.empty else repr(p.default)] for p in inspect.signature(f).parameters.values()]


def plugins():
    from gtsfm_b200.detector_descriptor import B200SuperPointDetectorDescriptor
    from gtsfm_b200.matcher import B200LightGlueMatcher, B200SuperGlueMatcher
    from gtsfm_b200.verifier import B200Ransac

    return {"B200SuperPointDetectorDescriptor": B200SuperPointDetectorDescriptor(max_keypoints=5000, weights_path=syn.superpoint_state_dict(0)),
            "B200LightGlueMatcher": B200LightGlueMatcher("superpoint", weights_path=syn.lightglue_state_dict(2)),
            "B200SuperGlueMatcher": B200SuperGlueMatcher(weights_path=syn.superglue_state_dict(1)),
            "B200Ransac": B200Ransac(use_intrinsics_in_verification=True, estimation_threshold_px=4)}


def test_mirrors_match_the_reference_api(api):
    assert not gtsfm_api.HAVE_GTSFM, "this check is of the mirrors; GTSfM is importable here"
    for name, base in api["bases"].items():
        mirror = getattr(gtsfm_api, name)
        assert sorted(mirror.__abstractmethods__) == sorted(base["abstract"]), name
        for meth, want in base["abstract"].items():
            assert params(getattr(mirror, meth)) == want, (name, meth)
        if base["init"] is not None:
            assert params(mirror.__init__) == base["init"], name
    for meth, want in api["keypoints"]["methods"].items():
        if meth in vars(gtsfm_api.Keypoints):  # the mirror carries a subset, each with the reference's parameters
            assert params(getattr(gtsfm_api.Keypoints, meth)) == want, meth
    for name, obj in plugins().items():
        rec = api["plugins"][name]
        base = api["bases"][rec["base"]]
        assert isinstance(obj, getattr(gtsfm_api, rec["base"]))
        for meth, want in base["abstract"].items():  # GTSfM calls these; extra parameters must be optional
            got = params(getattr(type(obj), meth))
            assert [p[0] for p in got[:len(want)]] == [p[0] for p in want] and all(p[1] is not None for p in got[len(want):]), (name, meth)
        assert {k: repr(getattr(obj, k)) for k in rec["state"]} == rec["state"], name
        if "repr" in rec:
            assert repr(obj) == rec["repr"], name
        pickle.loads(pickle.dumps(obj))


def write_stand_in(api, root: Path) -> None:
    """The recorded layout as a package: every class the plugin API imports, at its module path, with the recorded abstract
    methods and constructor parameters and no behaviour."""

    def sig(ps):
        return ", ".join(n if d is None else f"{n}={d}" for n, d in ps)

    def module(path, src):
        parts = path.split(".")
        for i in range(1, len(parts)):
            pkg = root.joinpath(*parts[:i])
            pkg.mkdir(parents=True, exist_ok=True)
            (pkg / "__init__.py").touch()
        root.joinpath(*parts[:-1], parts[-1] + ".py").write_text(src)

    proc = api["process"]
    module(proc["module"], f"import abc\n\n\nclass {proc['name']}(abc.ABC):\n"
           + "".join(f"    @staticmethod\n    @abc.abstractmethod\n    def {m}():\n        ...\n\n" for m in proc["abstract"]))
    for cls in ("keypoints", "image"):
        rec = api[cls]
        body = "".join(f"    def {m}({sig(ps)}):\n        raise NotImplementedError\n\n" for m, ps in rec["methods"].items() if m != "__init__")
        init = rec["methods"].get("__init__", [["self", None], ["*args", None], ["**kwargs", None]])
        store = "".join(f"        self.{n} = {n}\n" for n, _ in init[1:] if not n.startswith("*"))
        module(rec["module"], f"class {cls.capitalize()}:\n    def __init__({sig(init)}):\n{store or '        pass'}\n\n{body}")
    for name, base in api["bases"].items():
        body = "".join(f"    @abc.abstractmethod\n    def {m}({sig(ps)}):\n        ...\n\n" for m, ps in base["abstract"].items())
        init = f"    def __init__({sig(base['init'])}):\n        pass\n\n" if base["init"] else ""
        ui = "".join(f"    @staticmethod\n    def {m}():\n        return {name!r}\n\n" for m in proc["abstract"])
        module(base["module"], f"import abc\n\nfrom {proc['module']} import {proc['name']}\n\n\nclass {name}({proc['name']}):\n{ui}{init}{body}")


SCRIPT = textwrap.dedent(
    """
    import importlib, json, pickle, sys
    api = json.loads(open(sys.argv[1]).read())
    sys.path[:0] = [sys.argv[2], sys.argv[3]]
    from gtsfm_b200 import gtsfm_api, synthetic as syn
    assert gtsfm_api.HAVE_GTSFM, "the gtsfm bases imported but gtsfm_api fell back to its mirrors"
    load = lambda rec, name: getattr(importlib.import_module(rec["module"]), name)
    assert gtsfm_api.Keypoints is load(api["keypoints"], "Keypoints") and gtsfm_api.Image is load(api["image"], "Image")
    process = load(api["process"], api["process"]["name"])
    from gtsfm_b200.detector_descriptor import B200SuperPointDetectorDescriptor
    from gtsfm_b200.matcher import B200LightGlueMatcher, B200SuperGlueMatcher
    from gtsfm_b200.verifier import B200Ransac
    objs = {"B200SuperPointDetectorDescriptor": B200SuperPointDetectorDescriptor(max_keypoints=5000, weights_path=syn.superpoint_state_dict(0)),
            "B200LightGlueMatcher": B200LightGlueMatcher("superpoint", weights_path=syn.lightglue_state_dict(2)),
            "B200SuperGlueMatcher": B200SuperGlueMatcher(weights_path=syn.superglue_state_dict(1)),
            "B200Ransac": B200Ransac(use_intrinsics_in_verification=True, estimation_threshold_px=4)}
    for name, obj in objs.items():
        base = api["plugins"][name]["base"]
        assert isinstance(obj, load(api["bases"][base], base)) and isinstance(obj, process), name
        pickle.loads(pickle.dumps(obj))
        assert obj.get_ui_metadata() is not None
    print("HAVE_GTSFM ok")
    """
)


def test_plugins_subclass_the_reference_bases(api, golden_dir, tmp_path):
    write_stand_in(api, tmp_path)
    r = subprocess.run([sys.executable, "-c", SCRIPT, str(golden_dir / "gtsfm_bases.json"), str(tmp_path), str(ROOT)],
                       capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and "HAVE_GTSFM ok" in r.stdout, r.stdout + r.stderr
