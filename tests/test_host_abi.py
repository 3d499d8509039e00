"""CPU-side checks of the drop-in boundary: the C-ABI library loads without a GPU and exports every symbol that
include/snp_b200.h declares; host-side tables agree with the reference's recorded values."""
import ctypes
import os
import re

import numpy as np
import pytest

from helpers import GOLDEN, traj_names, load_traj

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared_functions():
    text = open(os.path.join(ROOT, "include", "snp_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(snp_[a-z0-9_]+)\s*\(", text)))


def test_library_builds_loads_and_exports_every_declared_symbol():
    from social_navigation_pyenvs_b200 import build, _lib
    path = build.build()
    assert os.path.exists(path)
    handle = ctypes.CDLL(path)
    declared = _declared_functions()
    assert len(declared) >= 15
    for name in declared:
        assert hasattr(handle, name), f"{name} declared in include/snp_b200.h but not exported"
    assert sorted(_lib.EXPORTED_SYMBOLS) == declared, "ctypes signature table and header disagree"
    lib = _lib.lib()
    assert lib.snp_abi_version() == 4


def test_ctypes_struct_layouts_match_the_header(tmp_path):
    """Field offsets / sizes of the ctypes mirrors against the header itself, as gcc lays it out (a drift here would silently
    corrupt every call)."""
    import subprocess
    from social_navigation_pyenvs_b200 import _lib as L
    structs = {"snp_crowd": L.SnpCrowd, "snp_step_opts": L.SnpStepOpts, "snp_laser_args": L.SnpLaserArgs, "snp_lookahead_args": L.SnpLookaheadArgs,
               "snp_reset_args": L.SnpResetArgs}
    lines = []
    for cname, cls in structs.items():
        lines.append(f'printf("{cname} %zu\\n", sizeof({cname}));')
        for f, _ in cls._fields_:
            lines.append(f'printf("{cname}.{f} %zu\\n", offsetof({cname}, {f}));')
    src = tmp_path / "layout.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "snp_b200.h"\nint main(void) {\n' + "\n".join(lines) + "\nreturn 0; }\n")
    exe = tmp_path / "layout"
    subprocess.run(["gcc", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)], check=True)
    out = dict(l.split() for l in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.splitlines())
    for cname, cls in structs.items():
        assert int(out[cname]) == ctypes.sizeof(cls), cname
        for f, _ in cls._fields_:
            assert int(out[f"{cname}.{f}"]) == getattr(cls, f).offset, (cname, f)


def test_python_constants_match_the_header_enums(tmp_path):
    """The option bits, dtype codes, field counts and flag bits the Python side uses are the header's."""
    import subprocess
    from social_navigation_pyenvs_b200 import _lib as L
    names = ["SNP_F32", "SNP_F64", "SNP_OPT_FULL_PAIR_LOOP", "SNP_OPT_NO_CULLING", "SNP_OPT_MAP_WARP", "SNP_OPT_MAP_BLOCK", "SNP_OPT_STAGED_COPIES"]
    src = tmp_path / "enums.c"
    src.write_text('#include <stdio.h>\n#include "snp_b200.h"\nint main(void) {\n' + "\n".join(f'printf("{n} %d\\n", (int){n});' for n in names) +
                   '\nprintf("DYN_FIELDS %d\\nSTAT_FIELDS %d\\nROBOT_FIELDS %d\\n", (int)SNP_DYN_FIELDS, (int)SNP_STAT_FIELDS, (int)SNP_ROBOT_FIELDS);\nreturn 0; }\n')
    exe = tmp_path / "enums"
    subprocess.run(["gcc", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)], check=True)
    out = dict(l.split() for l in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.splitlines())
    for n in names:
        assert int(out[n]) == getattr(L, n), n
    assert (int(out["DYN_FIELDS"]), int(out["STAT_FIELDS"]), int(out["ROBOT_FIELDS"])) == (L.DYN_FIELDS, L.STAT_FIELDS, L.ROBOT_FIELDS)


def test_missing_library_fails_loudly(monkeypatch, tmp_path):
    from social_navigation_pyenvs_b200 import _lib
    monkeypatch.setattr(_lib, "_lib", None)
    monkeypatch.setattr(_lib, "LIB_PATH", str(tmp_path / "nope.so"))
    with pytest.raises(ImportError):
        _lib.lib()


def test_model_parameter_rows_match_the_reference():
    """model_parameters(title) == Agent.get_parameters(title) as recorded in every golden fixture (agent.py:268-388)."""
    from social_navigation_pyenvs_b200 import model_parameters, SFMS
    import oracle
    seen = set()
    for name in traj_names():
        d = load_traj(name)
        title = SFMS[int(d["type"])]
        seen.add(title)
        assert np.array_equal(model_parameters(title), d["params"][0]), title
        assert np.array_equal(oracle.default_params(title), d["params"][0]), title
    assert seen == set(SFMS)
    with pytest.raises(Exception):
        model_parameters("orca")


def test_pack_walls_matches_reference_segment_order():
    """Vertex lists -> sorted-endpoint NaN-padded segments == what the reference's Obstacle built (obstacle.py:26-32)."""
    from social_navigation_pyenvs_b200 import scenarios
    d = load_traj("walls7_sfm_helbing")
    assert np.array_equal(scenarios.pack_walls(scenarios.EXAMPLE_WALLS), d["walls"], equal_nan=True)


def test_operator_argument_validation_needs_no_gpu():
    from social_navigation_pyenvs_b200 import update_humans_parallel
    with pytest.raises(ValueError):
        update_humans_parallel(-1, np.zeros((2, 13)), np.zeros((2, 1, 2)), None, np.zeros((2, 20)), 0.01, np.zeros(2))
    with pytest.raises(ValueError):
        update_humans_parallel(0, np.zeros((2, 12)), np.zeros((2, 1, 2)), None, np.zeros((2, 20)), 0.01, np.zeros(2))
    with pytest.raises(ValueError):
        update_humans_parallel(0, np.zeros((3, 13)), np.zeros((2, 1, 2)), None, np.zeros((2, 20)), 0.01, np.zeros(2))


def test_large_crowd_scratch_size_covers_every_region():
    """snp_large_scratch_bytes is host arithmetic (no GPU): it must cover the per-chunk partial sums, the live map, the list of
    (agent block, chunk) units, the per-block ascending lists and the queue counters -- for whole and ragged sizes."""
    from social_navigation_pyenvs_b200 import _lib as L
    lib = L.lib()
    for n_local, M in ((8192, 65536), (65536, 65536), (5184, 5184), (1, 2), (130, 1000)):
        for dtype, w in ((L.SNP_F64, 8), (L.SNP_F32, 4)):
            J, blocks = -(-M // 128), -(-n_local // 128)
            Jp = (J + 15) // 16 * 16
            need = w * J * 2 * n_local + blocks * Jp + 4 * (260 + blocks * J + blocks + blocks * Jp)
            got = int(lib.snp_large_scratch_bytes(n_local, M, dtype))
            assert need <= got <= need + 4 * 16, (n_local, M, dtype, need, got)  # (at most 15 bytes of alignment per region)


def test_large_crowd_step_rejects_bad_slices_and_rank_counts_before_any_launch():
    """snp_large_run_p2p validates on the host: a slice reaching past the view (offset + N = M + 1) or a world outside 1..8 is
    SNP_ERR_INVALID before anything touches the device (the pointers are dummies)."""
    from social_navigation_pyenvs_b200 import _lib as L
    lib = L.lib()
    dummy = ctypes.c_void_p(4096)
    c = L.SnpCrowd(E=1, N=256, G=2, dtype=L.SNP_F64, dyn=dummy, stat=dummy, goals=dummy, goal_idx=dummy, goal_cnt=dummy)
    o = L.SnpStepOpts(type=3, dt=0.0125)
    for offset, M, world, rank in ((1, 256, 1, 0), (257, 512, 1, 0), (0, 256, 0, 0), (0, 2304, 9, 0), (0, 512, 2, 2)):
        views = (ctypes.c_void_p * 9)(*[4096] * 9)
        n_bytes = int(lib.snp_large_scratch_bytes(256, M, L.SNP_F64))
        rc = lib.snp_large_run_p2p(ctypes.byref(c), ctypes.byref(o), views, views, 0, M, offset, world, rank, views, 0, 1, dummy, dummy,
                                   n_bytes, None)
        assert rc == -1, (offset, M, world, rank)
        assert "snp_large_run_p2p" in lib.snp_last_error().decode()


def test_product_package_never_imports_the_oracle():
    """The oracle is test infrastructure: nothing under social_navigation_pyenvs_b200/ may reference it."""
    pkg = os.path.join(ROOT, "social_navigation_pyenvs_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                src = open(os.path.join(dirpath, f)).read()
                assert not re.search(r"^\s*(import|from)\s+oracle\b", src, flags=re.M), f
                assert "libsnp_oracle" not in src and "oracle/_build" not in src, f  # no dlopen / link of the checker
