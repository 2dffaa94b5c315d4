"""Build the reference's own Cython helpers for the running Python into oracle/_ref/ (git-ignored).

TEST INFRASTRUCTURE ONLY.  The sources stay where they are under /root/reference (read-only); only the
generated C and the compiled extension modules land in oracle/_ref/.  Nothing is copied into the repo.

  /root/reference/dataloader/cython_cnt2event/cnt2event.pyx
      -> oracle/_ref/dataloader/cython_cnt2event/cnt2event.<abi>.so
  /root/reference/dataloader/cython_event_redistribute/event_redistribute.pyx
      -> oracle/_ref/dataloader/cython_event_redistribute/event_redistribute.<abi>.so

`dataloader` is a namespace package in the reference (no __init__.py), so with
sys.path = [oracle/_ref, /root/reference] the reference's dataloader/encodings.py imports these builds.
On the GPU box /root/reference is absent; the two .so files still import on their own (numpy only) and
serve as the "reference" CPU baseline for cnt2event / event_redistribute.
"""
import os
import subprocess
import sys
import sysconfig

REF = os.environ.get("ESR_REFERENCE", "/root/reference")
HERE = os.path.dirname(os.path.abspath(__file__))
OUT = os.path.join(HERE, "_ref")

MODULES = [
    ("dataloader/cython_cnt2event", "cnt2event"),
    ("dataloader/cython_event_redistribute", "event_redistribute"),
]


def built_paths():
    ext = sysconfig.get_config_var("EXT_SUFFIX")
    return [os.path.join(OUT, d, name + ext) for d, name in MODULES]


def build(force=False):
    """Returns True when both extension modules exist under oracle/_ref (building them if possible)."""
    paths = built_paths()
    if not force and all(os.path.exists(p) for p in paths):
        return True
    if not os.path.isdir(REF):
        return False
    import numpy as np
    from Cython.Compiler import Options
    from Cython.Compiler.Main import compile as cy_compile, CompilationOptions

    for (d, name), so in zip(MODULES, paths):
        pyx = os.path.join(REF, d, name + ".pyx")
        os.makedirs(os.path.dirname(so), exist_ok=True)
        c_file = os.path.join(os.path.dirname(so), name + ".c")
        opts = CompilationOptions(Options.default_options, output_file=c_file, language_level=3)
        res = cy_compile(pyx, opts)
        if res.num_errors:
            raise RuntimeError(f"cython failed on {pyx}")
        cmd = ["gcc", "-O2", "-shared", "-fPIC", "-w", "-DNPY_NO_DEPRECATED_API=NPY_1_7_API_VERSION",
               "-I" + sysconfig.get_paths()["include"], "-I" + np.get_include(), c_file, "-o", so]
        subprocess.check_call(cmd)
        os.remove(c_file)  # generated from reference source: do not keep it around
    return True


def import_ref_modules():
    """(cnt2event, event_redistribute) reference modules, or (None, None) if not built.  Builds nothing: its caller
    (bench.py) may run from a read-only tree."""
    if not all(os.path.exists(p) for p in built_paths()):
        return None, None
    import importlib.util
    mods = []
    for (d, name), so in zip(MODULES, built_paths()):
        spec = importlib.util.spec_from_file_location(name, so)
        m = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(m)
        mods.append(m)
    return tuple(mods)


if __name__ == "__main__":
    ok = build(force="--force" in sys.argv)
    print("oracle/_ref built" if ok else "reference not available; oracle/_ref not built")
