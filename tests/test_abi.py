"""The C-ABI library loads and exports exactly what include/voxcarve.h declares (no compute calls)."""
import ctypes
import os
import re

import pytest

from conftest import ROOT, _has_gpu


def _declared():
    hdr = open(os.path.join(ROOT, "include", "voxcarve.h")).read()
    return sorted(set(re.findall(r"VC_EXPORT[^;]*?\b(vc_[a-z0-9_]+)\s*\(", hdr)))


def test_header_declares_the_boundary():
    names = _declared()
    for must in ("vc_create", "vc_destroy", "vc_set_views", "vc_set_masks", "vc_carve", "vc_fast_carve", "vc_color",
                 "vc_mc_classify", "vc_download_occupied", "vc_download_seen", "vc_download_colors", "vc_download_mc",
                 "vc_bind_volumes", "vc_last_error"):
        assert must in names


def test_library_exports_every_declared_symbol(lib_built):
    lib = ctypes.CDLL(lib_built)
    for name in _declared():
        assert hasattr(lib, name), f"libvoxcarve.so lacks {name}"


def test_binding_covers_header_exactly(lib_built):
    from ar_voxel_project_b200 import _lib
    assert sorted(_lib.SIGNATURES) == _declared()
    assert _lib.load().vc_api_version() == 3


def test_no_torch_types_in_abi():
    hdr = open(os.path.join(ROOT, "include", "voxcarve.h")).read()
    assert "torch" not in hdr and "at::" not in hdr and "std::" not in hdr


@pytest.mark.skipif(_has_gpu(), reason="checks the no-GPU failure mode")
def test_create_fails_loudly_without_gpu(lib_built):
    """no CPU fallback: the product path must refuse to run when CUDA is unavailable"""
    import ar_voxel_project_b200 as A
    with pytest.raises(A.VoxCarveError) as ei:
        A.VoxelEngine(8, 8, 8, 0.1)
    assert ei.value.code == 2 and "no CPU fallback" in str(ei.value)


def test_product_never_imports_oracle():
    """oracle/ is test infrastructure: nothing under the package or include/ may reference it"""
    pkg = os.path.join(ROOT, "ar_voxel_project_b200")
    for dp, _, fs in os.walk(pkg):
        for f in fs:
            if f.endswith((".py", ".cu", ".cuh", ".h", ".hpp", ".inc")):
                txt = open(os.path.join(dp, f)).read()
                assert "oracle" not in txt.lower() or f == "vc_kernels.cuh" and "oracle: vo_pixel" in txt, os.path.join(dp, f)


def test_binding_structs_match_the_header(tmp_path):
    """vc_grid_desc and vc_stats cross the ABI by pointer: the ctypes mirrors must have the header's fields, in its order, at its
    offsets (gcc compiles the header and prints offsetof / sizeof)."""
    import subprocess
    from ar_voxel_project_b200 import _lib
    hdr = open(os.path.join(ROOT, "include", "voxcarve.h")).read()
    prog = ['#include <stdio.h>', '#include <stddef.h>', '#include "voxcarve.h"', 'int main(void) {']
    mirrors = {"vc_grid_desc": _lib.GridDesc, "vc_stats": _lib.Stats}
    for cname, mirror in mirrors.items():
        body = re.search(r"typedef struct %s \{(.*?)\} %s;" % (cname, cname), hdr, re.S).group(1)
        body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
        fields = []
        for decl in body.split(";"):
            decl = decl.strip()
            if decl:
                fields += [n.strip() for n in decl.split(None, 1)[1].split(",")]
        assert fields == [n for n, _ in mirror._fields_], (cname, fields)
        for f in fields:
            prog.append(f'    printf("{cname}.{f} %zu\\n", offsetof({cname}, {f}));')
        prog.append(f'    printf("{cname} %zu\\n", sizeof({cname}));')
    prog += ['    return 0;', '}']
    src = tmp_path / "layout.c"
    src.write_text("\n".join(prog))
    exe = tmp_path / "layout"
    subprocess.run(["gcc", "-I", os.path.join(ROOT, "include"), "-o", str(exe), str(src)], check=True)
    out = dict(line.split() for line in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.splitlines())
    for cname, mirror in mirrors.items():
        assert int(out[cname]) == ctypes.sizeof(mirror)
        for n, _ in mirror._fields_:
            assert int(out[f"{cname}.{n}"]) == getattr(mirror, n).offset, (cname, n)


def test_environment_switches_are_documented():
    """The environment variables the library reads (getenv in csrc/) are exactly the ones include/voxcarve.h documents."""
    csrc = os.path.join(ROOT, "ar_voxel_project_b200", "csrc")
    read = set()
    for f in os.listdir(csrc):
        read |= set(re.findall(r'getenv\("([A-Za-z0-9_]+)"\)', open(os.path.join(csrc, f)).read()))
    hdr = open(os.path.join(ROOT, "include", "voxcarve.h")).read()
    documented = set(re.findall(r"\bVOXCARVE_[A-Z0-9_]+", hdr)) - {"VOXCARVE_H"}  # minus the include guard
    assert read and read == documented, (sorted(read), sorted(documented))
