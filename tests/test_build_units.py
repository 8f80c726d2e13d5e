"""CPU: the incremental build knows every translation unit and every file each one includes, so that an edited header
recompiles exactly the units that include it and no stale object survives."""
import os
import re

from pfb_imaging_b200 import _lib


def quoted_includes(path):
    src = open(path).read()
    return [os.path.normpath(os.path.join(os.path.dirname(path), f))
            for f in re.findall(r'^\s*#\s*include\s+"([^"]+)"', src, flags=re.M)]


def include_closure(path):
    seen, todo = set(), [path]
    while todo:
        for dep in quoted_includes(todo.pop()):
            if dep not in seen:
                seen.add(dep)
                todo.append(dep)
    return seen


def test_every_unit_is_built():
    units = sorted(f for f in os.listdir(_lib.CSRC) if f.endswith(".cu"))
    assert units == sorted(_lib._UNITS)


def test_unit_dependencies_are_the_include_closure():
    for unit, deps in _lib._UNITS.items():
        listed = {os.path.normpath(os.path.join(_lib.CSRC, d)) for d in deps}
        assert len(listed) == len(deps), f"{unit}: a dependency is listed twice"
        want = include_closure(os.path.join(_lib.CSRC, unit))
        assert listed == want, (f"{unit}: missing {sorted(os.path.relpath(d, _lib.CSRC) for d in want - listed)}, "
                                f"extra {sorted(os.path.relpath(d, _lib.CSRC) for d in listed - want)}")
