"""The C-ABI library loads without a GPU and exports every symbol include/uqs_mapping.h declares."""
import ctypes
import os
import re
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def declared_symbols():
    txt = open(os.path.join(ROOT, "include", "uqs_mapping.h")).read()
    txt = re.sub(r"/\*.*?\*/", "", txt, flags=re.S)
    funcs = re.findall(r"^\s*(?:const\s+)?[A-Za-z_][\w\s\*]*?\b(\w+)\s*\([^;{]*\)\s*;", txt, flags=re.M)
    data = re.findall(r"^\s*extern\s+[\w\s\*]+?\b(\w+)\s*(?:\[[^\]]*\])*\s*;", txt, flags=re.M)
    return sorted(set(funcs) | set(data))


def test_header_declares_the_reference_signatures():
    syms = declared_symbols()
    for s in ["world_to_grid", "raycast_update", "map_update_from_beams", "occ_grid", "map_inited", "map_origin_x",
              "map_origin_y", "tof_beams_m", "pending_kf_flags", "uqs_replay", "uqs_replay_dev", "uqs_pose_integrate",
              "uqs_init", "uqs_last_error"]:
        assert s in syms, s


def test_library_exports_every_declared_symbol(pkg):
    L = pkg.lib()
    missing = [s for s in declared_symbols() if not hasattr(L, s)]
    assert not missing, missing


def test_python_binding_lists_only_exported_symbols(pkg):
    L = pkg.lib()
    assert not [s for s in pkg.exported_symbols() if not hasattr(L, s)]


def test_header_compiles_as_c99():
    src = '#include "uqs_mapping.h"\nint main(void){ uqs_params p; (void)p; return (int)sizeof(uqs_stats) == 0; }\n'
    r = subprocess.run(["gcc", "-std=c99", "-Wall", "-Wextra", "-Werror", "-fsyntax-only", "-I", os.path.join(ROOT, "include"),
                        "-x", "c", "-"], input=src, text=True, capture_output=True)
    assert r.returncode == 0, r.stderr


def test_params_struct_layout_matches_header(pkg, tmp_path):
    src = '#include <stdio.h>\n#include <stddef.h>\n#include "uqs_mapping.h"\nint main(void){printf("%zu %zu %zu %zu %zu", sizeof(uqs_params), offsetof(uqs_params,res_m), offsetof(uqs_params,lo_free), sizeof(uqs_stats), offsetof(uqs_stats,domain_errors));return 0;}\n'
    exe = str(tmp_path / "uqs_layout_probe")
    r = subprocess.run(["gcc", "-I", os.path.join(ROOT, "include"), "-x", "c", "-", "-o", exe], input=src, text=True, capture_output=True)
    assert r.returncode == 0, r.stderr
    out = subprocess.check_output([exe], text=True).split()
    P, S = pkg.Params, pkg.Stats
    assert [int(v) for v in out] == [ctypes.sizeof(P), P.res_m.offset, P.lo_free.offset, ctypes.sizeof(S), S.domain_errors.offset]


def test_fails_loudly_without_a_device(pkg):
    """No CPU fallback: on a machine without CUDA every entry point reports an error."""
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    with pytest.raises(pkg.UqsError) as e:
        pkg.init(0)
    assert e.value.code == pkg.ERR_NO_DEVICE
    import numpy as np
    p = pkg.make_params(400, 400, 0.05)
    z = np.zeros((1, 4), np.float32)
    with pytest.raises(pkg.UqsError) as e:
        pkg.replay(p, z, z, z, np.zeros((1, 4, 32), np.float32))
    assert e.value.code == pkg.ERR_NOT_INIT
    # the profiling exports report "not initialised" too, and the file readers (host-only C) still work
    assert pkg.lib().uqs_profile_timeline(None, 0) == -1
    assert pkg.profile_timeline() == []


def test_product_never_references_the_oracle():
    """Nothing under the package (sources or binding) may import, link or name the oracle."""
    pk = os.path.join(ROOT, "micro-quad-slam_b200")
    for dp, _, files in os.walk(pk):
        for f in files:
            if f.endswith((".so", ".pyc")):
                continue
            txt = open(os.path.join(dp, f), errors="replace").read()
            assert "liborc" not in txt and "oracle/" not in txt and "from oracle" not in txt and "import oracle" not in txt, os.path.join(dp, f)
    out = subprocess.check_output(["ldd", os.path.join(pk, "libuqs_mapping.so")], text=True)
    assert "liborc" not in out and "libref" not in out
