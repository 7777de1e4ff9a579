#!/usr/bin/env python
"""Golden record for tests/test_overlay_cpu.py, taken from the REFERENCE checkout:

* `packages`: the imports of the reference's own package files models/__init__.py and utils/__init__.py (module, names),
  read from their source, so the test's stand-in tree has regular packages that the overlay must shadow;
* `resolved`: a snapshot of what the drop-in overlay (seg_b200.launch.setup_paths) made of the reference at recording time:
  for every module a reference script imports through it, which public class / function each name resolves to, the
  B200-native one ("engine") or the reference's, with the file (relative to the reference root) that defines it;
* `config`: the config.json fields the test's train.py walk-through reads.

Third-party packages the reference imports only at module level (sklearn, scipy, ...) are replaced by empty stand-ins when
they are not installed: no name the record keeps comes from them.  Writes tests/golden/overlay_registries.json.
Run:  python oracle/make_golden_overlay.py <reference root>   (or set SEG_REFERENCE_ROOT)"""
import ast
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = sys.argv[1] if len(sys.argv) > 1 else os.environ.get("SEG_REFERENCE_ROOT")  # a checkout of the reference
MODULES = ["models", "utils.losses", "utils.metrics", "utils.lr_scheduler", "utils.helpers", "utils.lovasz_losses",
           "utils.sync_batchnorm", "base"]
PACKAGES = ["models/__init__.py", "utils/__init__.py"]
THIRD_PARTY = ["sklearn", "scipy", "cv2", "PIL", "tqdm", "tensorboard", "matplotlib"]

# import-time stand-ins for the THIRD_PARTY packages that fail to import (every attribute is another empty module)
STUBS = r"""
import importlib, importlib.abc, importlib.util, sys, types
class _Stub(types.ModuleType):
    def __getattr__(self, k):
        if k.startswith("__"):
            raise AttributeError(k)
        m = _Stub(self.__name__ + "." + k)
        sys.modules[m.__name__] = m
        setattr(self, k, m)
        return m
_missing = set()
for _n in STUB_NAMES:
    try:
        importlib.import_module(_n)
    except Exception:
        _missing.add(_n)
class _Finder(importlib.abc.MetaPathFinder, importlib.abc.Loader):
    def find_spec(self, name, path, target=None):
        return importlib.util.spec_from_loader(name, self, is_package=True) if name.split(".")[0] in _missing else None
    def create_module(self, spec):
        return _Stub(spec.name)
    def exec_module(self, module):
        pass
sys.meta_path.insert(0, _Finder())
"""

# shared with the test: prints {module: {name: "engine" | "<path under the reference root>"}} for the tree at sys.argv[1]
RESOLVE = r"""
import importlib, inspect, json, os, sys
from seg_b200 import launch
root = os.path.abspath(sys.argv[1])
launch.setup_paths(root)
pkg = os.path.dirname(os.path.dirname(os.path.abspath(launch.__file__)))

def origin(obj):
    if inspect.isfunction(obj):
        return obj.__code__.co_filename
    for v in vars(obj).values():  # classes of exec'd modules are not in sys.modules: ask their own methods
        if inspect.isfunction(v):
            return v.__code__.co_filename
    return inspect.getsourcefile(obj)

out = {}
for name in sys.argv[2:]:
    mod, got = importlib.import_module(name), {}
    for k, v in vars(mod).items():
        if k.startswith("_") or not (inspect.isclass(v) or inspect.isfunction(v)):
            continue
        try:
            f = os.path.abspath(origin(v))
        except (TypeError, OSError):
            continue
        if f.startswith(pkg + os.sep):
            got[k] = "engine"
        elif f.startswith(root + os.sep):
            got[k] = os.path.relpath(f, root).replace(os.sep, "/")
    out[name] = dict(sorted(got.items()))
print("RESOLVED " + json.dumps(out))
"""


def resolve(ref_root, stub=()):
    """Runs RESOLVE on the tree at ref_root in a fresh interpreter; `stub`: THIRD_PARTY names to stand in for if missing."""
    env = dict(os.environ, PYTHONPATH=os.path.join(ROOT, "pytorch-segmentation_b200"))
    env.pop("SEG_REFERENCE_ROOT", None)
    code = (STUBS.replace("STUB_NAMES", repr(list(stub))) if stub else "") + RESOLVE
    r = subprocess.run([sys.executable, "-W", "ignore", "-c", code, ref_root] + MODULES, env=env, cwd=ref_root,
                       capture_output=True, text=True, timeout=600)
    line = [ln for ln in r.stdout.splitlines() if ln.startswith("RESOLVED ")]
    assert line, r.stdout[-2000:] + r.stderr[-4000:]
    return json.loads(line[0][len("RESOLVED "):])


def package_imports(path):
    """[(module, [names])] of the `from X import a, b` statements of a package file."""
    with open(path) as f:
        tree = ast.parse(f.read())
    return [["." * n.level + (n.module or ""), [a.name for a in n.names]] for n in tree.body if isinstance(n, ast.ImportFrom)]


def main():
    if not REF:
        sys.exit(__doc__)
    with open(os.path.join(REF, "config.json")) as f:
        cfg = json.load(f)
    golden = {"config": {k: cfg[k] for k in ("use_synch_bn", "arch", "loss", "ignore_index")},
              "packages": {p: package_imports(os.path.join(REF, p)) for p in PACKAGES},
              "resolved": resolve(REF, THIRD_PARTY)}
    dst = os.path.join(ROOT, "tests", "golden", "overlay_registries.json")
    with open(dst, "w") as f:
        json.dump(golden, f, indent=1, sort_keys=True)
        f.write("\n")
    print("wrote", dst)


if __name__ == "__main__":
    main()
