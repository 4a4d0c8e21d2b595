"""Loader for the UNMODIFIED reference (TimoStoff/event_utils) -- TEST / BASELINE INFRASTRUCTURE ONLY.

Where the reference lives: ``$EVK_REFERENCE_ROOT`` (a checkout of TimoStoff/event_utils).  It is used by
``tests/golden/make_golden.py`` and ``tests/golden/make_reference_checks.py`` to generate the committed golden
vectors and by the module-swap test, which runs the reference's own callers and skips where it is absent.

Two of the hot-path files do not parse as shipped (SURVEY.md section 8c):
  * lib/contrast_max/warps.py:7-10  class docstring at column 0, :81 stray text, :3 bogus import
  * lib/contrast_max/objectives.py:11-13 class docstring at column 0
so those two are read as text, minimally patched IN MEMORY (nothing is written anywhere) and
exec'd into module objects.  Missing third-party imports (matplotlib, h5py, skimage) are
stubbed with empty modules; none of them is touched by the functions we call.
"""
import importlib
import os
import sys
import types


REF_ROOT = os.environ.get("EVK_REFERENCE_ROOT", "")


def available():
    return bool(REF_ROOT) and os.path.isdir(os.path.join(REF_ROOT, "lib", "representations"))


def _stub(name, **attrs):
    if name in sys.modules:
        return sys.modules[name]
    m = types.ModuleType(name)
    m.__dict__.update(attrs)
    m.__path__ = []  # behave like a package so "import a.b" works
    sys.modules[name] = m
    return m


def _install_stubs():
    for name in ("matplotlib", "matplotlib.pyplot", "matplotlib.patches", "matplotlib.cm",
                 "matplotlib.colors", "h5py", "skimage", "skimage.measure", "mpl_toolkits",
                 "mpl_toolkits.mplot3d", "event_utils"):
        try:
            importlib.import_module(name)
        except Exception:
            _stub(name)
    sk = sys.modules.get("skimage.measure")
    if sk is not None and not hasattr(sk, "block_reduce"):
        sk.block_reduce = lambda *a, **k: None
    m3 = sys.modules.get("mpl_toolkits.mplot3d")
    if m3 is not None and not hasattr(m3, "Axes3D"):
        m3.Axes3D = object


def _indent_column0_docstring(src):
    """Indent a triple-quoted block that sits at column 0 right after a ``class`` line."""
    out, lines, i = [], src.split("\n"), 0
    while i < len(lines):
        out.append(lines[i])
        if lines[i].startswith("class ") and i + 1 < len(lines) and lines[i + 1].startswith('"""'):
            i += 1
            out.append("    " + lines[i])
            if lines[i].count('"""') < 2:
                i += 1
                while '"""' not in lines[i]:
                    out.append("    " + lines[i])
                    i += 1
                out.append("    " + lines[i])
        i += 1
    return "\n".join(out)


def _exec_patched(modname, relpath, drop_substrings=()):
    path = os.path.join(REF_ROOT, relpath)
    with open(path) as f:
        src = f.read()
    src = "\n".join(l for l in src.split("\n") if not any(s in l for s in drop_substrings))
    src = _indent_column0_docstring(src)
    mod = types.ModuleType(modname)
    mod.__file__ = path
    mod.__package__ = modname.rsplit(".", 1)[0]
    sys.modules[modname] = mod
    exec(compile(src, path, "exec"), mod.__dict__)
    return mod


_cache = {}


def load():
    """Return a namespace with the reference's hot-path modules:
    .image .voxel_grid .optic_flow .event_util .warps .objectives"""
    if "ns" in _cache:
        return _cache["ns"]
    if not available():
        raise RuntimeError("reference tree not present at %s" % REF_ROOT)
    _install_stubs()
    if REF_ROOT not in sys.path:
        sys.path.insert(0, REF_ROOT)
    ns = types.SimpleNamespace()
    ns.image = importlib.import_module("lib.representations.image")
    ns.optic_flow = importlib.import_module("lib.transforms.optic_flow")
    ns.event_util = importlib.import_module("lib.util.event_util")
    ns.voxel_grid = importlib.import_module("lib.representations.voxel_grid")
    # lib.contrast_max/__init__ imports events_cmax (needs visualisation); bypass the package
    pkg = types.ModuleType("lib.contrast_max")
    pkg.__path__ = [os.path.join(REF_ROOT, "lib", "contrast_max")]
    sys.modules["lib.contrast_max"] = pkg
    ns.warps = _exec_patched("lib.contrast_max.warps", "lib/contrast_max/warps.py",
                             drop_substrings=("{not:timeslice}", "from event_utils import"))
    ns.objectives = _exec_patched("lib.contrast_max.objectives", "lib/contrast_max/objectives.py")
    _cache["ns"] = ns
    return ns
