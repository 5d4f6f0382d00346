"""Arena size queries (femo_problem_device_bytes, femo_amg_symbolic info[1]) on the host, without a device.  Each figure is
the count pass of the layout walk that upload places, so it is exact.  The figures before the walk existed were written
down by hand with slack on top; the exact ones may only be smaller than those, by the removed slack and over-counts."""
import ctypes as C

import numpy as np
import pytest

from femo_b200 import engine as E

KIB = 1024


def _motor():
    m = E.EngineMesh.annulus(4, 32)
    return E.EngineProblem(m, E.FAMILY_MOTOR_EM, params=[1.0] * 21, cell_tags=np.arange(m.ncells) % 4)


# name: (build, enable_multigrid, static and work bytes of the hand-written size query)
CASES = {
    'poisson_p1_n8': (lambda: E.EngineProblem(E.EngineMesh.unit_square(8), E.FAMILY_POISSON_P1), False, 38912, 237312),
    'nlpoisson_p1_n64_mg': (lambda: E.EngineProblem(E.EngineMesh.unit_square(64), E.FAMILY_NLPOISSON_P1), True,
                            2143744, 2777088),
    'nlpoisson_p1_n256_mg': (lambda: E.EngineProblem(E.EngineMesh.unit_square(256), E.FAMILY_NLPOISSON_P1), True,
                             33508864, 35782656),
    'nlpoisson_p2_n32_mg': (lambda: E.EngineProblem(E.EngineMesh.unit_square(32), E.FAMILY_NLPOISSON_P2), True,
                            1931008, 3057152),
    'simp_q1_32x16_mg': (lambda: E.EngineProblem(E.EngineMesh.rectangle_quad((0.0, 0.0), (2.0, 1.0), 32, 16),
                                                 E.FAMILY_SIMP_Q1, tagged=[0]), True, 716032, 1462784),
    'simp_hex8_16x8x8_mg': (lambda: E.EngineProblem(E.EngineMesh.box_hex((0.0, 0.0, 0.0), (2.0, 1.0, 1.0), 16, 8, 8),
                                                    E.FAMILY_SIMP_HEX8, tagged=[0]), True, 8961024, 16156160),
    'eb_beam_50': (lambda: E.EngineProblem(E.EngineMesh.interval(50, 0.0, 1.0), E.FAMILY_EB_BEAM, tagged=[1]), False,
                   34048, 300544),
    'rm_plate_n8': (lambda: E.EngineProblem(E.EngineMesh.unit_square(8), E.FAMILY_RM_PLATE), False, 390656, 3823616),
    'mass_p1_n8': (lambda: E.EngineProblem(E.EngineMesh.unit_square(8), E.FAMILY_MASS_P1, params=(0, 1, 1)), False,
                   38912, 237312),
    'motor_em_4x32': (_motor, False, 118272, 3021056),
}


def _device_bytes(p):
    sb, wb = C.c_size_t(), C.c_size_t()
    E.check(E.lib.femo_problem_device_bytes(p._h, C.byref(sb), C.byref(wb)))
    return sb.value, wb.value


def _host_layout(p):
    out = []
    for w in range(1 + p.nin):
        ptr, src = p.gather_map(w)
        out.append((p.pattern_info(w), ptr, src))
    return out


def _check_smaller(name, hand_written, exact, levels):
    # slack: 4096 + 1024 per level per arena; over-counts: the u_ex table, the transposed row blocks of square
    # patterns, the rounding of the GMRES vectors
    assert 0 <= hand_written - exact <= 32 * KIB + 4 * KIB * levels, (name, hand_written, exact)


@pytest.mark.parametrize('name', sorted(CASES))
def test_problem_size_query_is_exact_and_host_only(name):
    build, mg, static_before, work_before = CASES[name]
    p = build()
    levels = p.enable_multigrid() if mg else 0
    before = _host_layout(p)
    sb, wb = _device_bytes(p)
    assert _device_bytes(p) == (sb, wb)                  # the count pass leaves the problem as it found it
    after = _host_layout(p)
    for (i0, p0, s0), (i1, p1, s1) in zip(before, after):
        assert i0 == i1 and np.array_equal(p0, p1) and np.array_equal(s0, s1)
    assert sb % 256 == 0 and wb % 256 == 0
    _check_smaller(name + ' static', static_before, sb, levels)
    _check_smaller(name + ' work', work_before, wb, levels)


def test_amg_size_query_is_exact_and_host_only():
    p = _motor()
    a = p.amg_symbolic(None, coarse_size=40)
    assert a['levels'] == 2
    assert p.amg_symbolic(None, coarse_size=40)['bytes'] == a['bytes']
    assert a['bytes'] % 256 == 0
    _check_smaller('motor_em_4x32 amg', 81664, a['bytes'], a['levels'])
