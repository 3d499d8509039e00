"""CPU-side checks of the unit-sized scratch of the tiled path (SNP_OPT_UNIT_SCRATCH): snp_large_scratch_bytes_units and
snp_large_batch_scratch_bytes_units are host arithmetic that covers every region, equal the default sizes when every unit has a slot,
and refuse bad arguments; snp_large_run_p2p and snp_large_batch_step refuse, before anything touches the device (the pointers are
dummies), a scratch short of the size for no slot and everything that needs the static grid."""
import ctypes
import os

import pytest

DUMMY = ctypes.c_void_p(4096)
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
COUNTERS = 4 * 260  # the counter block in front of the partial sums


def _one(n_local, M, w, units):
    """The regions of one crowd's scratch with `units` slots, without alignment: counters, partial sums, live map, work list, live
    counts, live lists."""
    J, blocks = -(-M // 128), -(-n_local // 128)
    Jp = (J + 15) // 16 * 16
    return COUNTERS + units * 2 * 128 * w + blocks * Jp + 4 * (blocks * J + blocks + blocks * Jp)


@pytest.mark.parametrize("dtype", ["f64", "f32"])
def test_unit_scratch_size_covers_every_region(dtype):
    from social_navigation_pyenvs_b200 import _lib as L
    lib = L.lib()
    dt, w = (L.SNP_F64, 8) if dtype == "f64" else (L.SNP_F32, 4)
    for n_local, M in ((65536, 65536), (8192, 65536), (5120, 5120), (1517, 1517), (1, 2), (130, 1000), (1500625, 1500625)):
        for units in (0, 1, 7, 1000, 123457):
            need = _one(n_local, M, w, units)
            got = int(lib.snp_large_scratch_bytes_units(n_local, M, dt, units))
            assert need <= got <= need + 5 * 16, (n_local, M, units, need, got)  # at most 15 bytes of alignment per region
    for E, N in ((64, 1024), (5, 513), (3, 1000), (1, 1)):
        J = -(-N // 128)
        views = 2 * w * 5 * (E * N + E * J)
        for units in (0, 3, 999):
            Jp = (J + 15) // 16 * 16
            blocks = E * J
            need = COUNTERS + units * 2 * 128 * w + blocks * Jp + 4 * (blocks * J + blocks + blocks * Jp) + views
            got = int(lib.snp_large_batch_scratch_bytes_units(E, N, dt, units))
            assert need <= got <= need + 7 * 16, (E, N, units, need, got)


@pytest.mark.parametrize("dtype", ["f64", "f32"])
def test_every_unit_with_a_slot_is_the_default_size(dtype):
    """At units = ceil(n_local/128) * ceil(M/128) with n_local a multiple of 128 the size is the default one, byte for byte; it grows
    with the units."""
    from social_navigation_pyenvs_b200 import _lib as L
    lib = L.lib()
    dt = L.SNP_F64 if dtype == "f64" else L.SNP_F32
    for n_local, M in ((65536, 65536), (8192, 65536), (5120, 5120)):
        units = (n_local // 128) * -(-M // 128)
        assert int(lib.snp_large_scratch_bytes_units(n_local, M, dt, units)) == int(lib.snp_large_scratch_bytes(n_local, M, dt))
        sizes = [int(lib.snp_large_scratch_bytes_units(n_local, M, dt, u)) for u in (0, 1, 2, units // 3, units, units + 1)]
        assert sizes == sorted(sizes) and sizes[0] < sizes[-1]
    for E, N in ((64, 1024), (4, 16384), (1, 5120)):
        units = E * (N // 128) ** 2
        assert int(lib.snp_large_batch_scratch_bytes_units(E, N, dt, units)) == int(lib.snp_large_batch_scratch_bytes(E, N, dt))
        sizes = [int(lib.snp_large_batch_scratch_bytes_units(E, N, dt, u)) for u in (0, 1, units // 2, units)]
        assert sizes == sorted(sizes) and sizes[0] < sizes[-1]


def test_unit_scratch_sizes_refuse_bad_arguments():
    from social_navigation_pyenvs_b200 import _lib as L
    lib = L.lib()
    for bad in ((0, 10, L.SNP_F64, 1), (10, 5, L.SNP_F64, 1), (10, 10, 7, 1), (10, 10, L.SNP_F32, -1)):
        assert int(lib.snp_large_scratch_bytes_units(*bad)) == -1, bad
        assert "snp_large_scratch_bytes_units" in lib.snp_last_error().decode()
    for bad in ((0, 10, L.SNP_F64, 1), (2, 0, L.SNP_F64, 1), (2, 10, 7, 1), (2, 10, L.SNP_F32, -1)):
        assert int(lib.snp_large_batch_scratch_bytes_units(*bad)) == -1, bad
        assert "snp_large_batch_scratch_bytes_units" in lib.snp_last_error().decode()
    with pytest.raises(ValueError):
        L.check_size(lib.snp_large_scratch_bytes_units(10, 10, L.SNP_F64, -1))


def _params(L, model):
    from social_navigation_pyenvs_b200 import model_parameters
    return (ctypes.c_double * 20)(*model_parameters(model))


def _run_p2p(L, model, type_, reserved, n_bytes=None, offset=0, N=256, M=1024):
    lib = L.lib()
    c = L.SnpCrowd(E=1, N=N, G=2, dtype=L.SNP_F64, dyn=DUMMY, stat=DUMMY, goals=DUMMY, goal_idx=DUMMY, goal_cnt=DUMMY, params=_params(L, model))
    o = L.SnpStepOpts(type=type_, dt=0.0125, reserved=reserved)
    if n_bytes is None:
        n_bytes = int(lib.snp_large_scratch_bytes_units(N, M, L.SNP_F64, 10))
    views = (ctypes.c_void_p * 1)(4096)
    return lib.snp_large_run_p2p(ctypes.byref(c), ctypes.byref(o), views, views, 0, M, offset, 1, 0, views, 0, 1, DUMMY, DUMMY, n_bytes, None)


def _batch(L, model, type_, reserved, n_bytes=None, E=3, N=700):
    lib = L.lib()
    c = L.SnpCrowd(E=E, N=N, G=2, dtype=L.SNP_F64, dyn=DUMMY, stat=DUMMY, goals=DUMMY, goal_idx=DUMMY, goal_cnt=DUMMY, params=_params(L, model))
    o = L.SnpStepOpts(type=type_, dt=0.0125, n_substeps=1, reserved=reserved)
    if n_bytes is None:
        n_bytes = int(lib.snp_large_batch_scratch_bytes_units(E, N, L.SNP_F64, 10))
    return lib.snp_large_batch_step(ctypes.byref(c), ctypes.byref(o), DUMMY, n_bytes, None)


@pytest.mark.parametrize("entry,case", [(e, c) for e in ("snp_large_run_p2p", "snp_large_batch_step")
                                        for c in ("scratch_short", "moussaid2", "moussaid5", "moussaid8", "no_culling")] +
                         [("snp_large_run_p2p", "offset")])  # (a batch has no slice offset)
def test_unit_scratch_refusals_before_any_launch(entry, case):
    from social_navigation_pyenvs_b200 import _lib as L, SFMS
    lib = L.lib()
    run = _run_p2p if entry == "snp_large_run_p2p" else _batch
    U, NC = L.SNP_OPT_UNIT_SCRATCH, L.SNP_OPT_NO_CULLING
    if case == "scratch_short":
        none = (lib.snp_large_scratch_bytes_units(256, 1024, L.SNP_F64, 0) if entry == "snp_large_run_p2p"
                else lib.snp_large_batch_scratch_bytes_units(3, 700, L.SNP_F64, 0))
        rc, want = run(L, "hsfm_farina", 3, U, n_bytes=int(none) - 1), -1
    elif case.startswith("moussaid"):
        t = int(case[-1])
        rc, want = run(L, SFMS[t], t, U), -3
    elif case == "no_culling":
        rc, want = run(L, "hsfm_farina", 3, U | NC), -3
    else:
        rc, want = _run_p2p(L, "hsfm_farina", 3, U, offset=64), -3
    assert rc == want, (entry, case, rc)
    assert entry in lib.snp_last_error().decode()


def test_unit_scratch_bit_matches_the_header(tmp_path):
    import subprocess
    from social_navigation_pyenvs_b200 import _lib as L
    src = tmp_path / "bit.c"
    src.write_text('#include <stdio.h>\n#include "snp_b200.h"\nint main(void) { printf("%d\\n", (int)SNP_OPT_UNIT_SCRATCH); return 0; }\n')
    exe = tmp_path / "bit"
    subprocess.run(["gcc", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)], check=True)
    assert int(subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout) == L.SNP_OPT_UNIT_SCRATCH == 32


@pytest.mark.parametrize("bad", ["many", -1, 2.5, True])
def test_unit_capacity_argument_is_checked(bad):
    """A capacity that is not None, an int >= 0 or "auto" is a ValueError before any allocation."""
    from social_navigation_pyenvs_b200.large import _UnitSlots
    with pytest.raises(ValueError):
        _UnitSlots()._setup_units(bad, 4, 4, lambda u: 0, "cpu")
