"""The oracle's graph-coloured update (oracle_update_coloured, the specification of CLOTHB200_MODE_COLOURED).

It is not the reference's update, so there is no reference to pin it to; these tests check its structure (the colour
classes), that it reduces to the reference-order update where the two orders cannot differ, and how far it moves from
reference order on a crumpled state.  tests/test_gpu_coloured_oracle.py pins the f64 coloured kernels to it."""
import numpy as np
import pytest

from conftest import load_golden
from oracle.oracle import OracleCloth, params_from_cfg

KIND_OFF = lambda W: (W, 1, W + 1, W - 1, 2 * W, 2)


def _params(W):
    P = params_from_cfg(None)
    P.num_width_points = W; P.num_height_points = W
    return P


@pytest.mark.parametrize("W", [5, 6, 7, 25, 64])
def test_colour_classes_partition_springs_into_matchings(W):
    o = OracleCloth(_params(W), mode="coloured")
    a, b, _, _ = o.springs()
    cls = o.colours()
    assert cls.shape == (o.S,) and cls.min() >= 0 and cls.max() <= 11
    # the class's kind is the spring's creation kind: ptA = ptB - off[kind]
    kind = cls // 2
    assert np.array_equal(b - a, np.array(KIND_OFF(W))[kind])
    for k in range(6):
        assert (kind == k).any()
    for j in range(12):
        m = cls == j
        ends = np.concatenate([a[m], b[m]])
        assert len(np.unique(ends)) == len(ends), (W, j)         # no point in two springs of one class
    # the parity rule of DESIGN.md §4
    r, c = b // W, b % W
    key = np.select([kind == 1, kind == 4, kind == 5], [c, r >> 1, c >> 1], r)
    assert np.array_equal(cls % 2, key & 1)


def _quiet_pair(relax):
    ref, col = OracleCloth(), OracleCloth(mode="coloured", relax_iters=relax)
    for o in (ref, col):
        assert o.grab_top(0.5, 0.5) > 0
    return ref, col


@pytest.mark.parametrize("relax", [1, 3])
def test_equals_reference_order_while_nothing_collides_or_stretches(relax):
    """The first lift substeps of the flat cloth: no pair within 2*thickness, no spring past 1.1*rest.  Then the
    Jacobi collision and the limit pass are both no-ops and one coloured update equals one reference-order update."""
    ref, col = _quiet_pair(relax)
    quiet = 0
    for i in range(50):
        for o in (ref, col):
            o.adjust(0.0, 0.0, 0.0025)
            o.update(1)
        cr = ref.counters()
        if cr["collide_hits"] or cr["stretched"]:
            break
        quiet += 1
        pr, qr, nr = ref.get_state(); pc, qc, nc = col.get_state()
        assert np.array_equal(pr, pc) and np.array_equal(qr, qc) and np.array_equal(nr, nc), i
        assert col.counters()["collide_hits"] == 0 and col.counters()["stretched"] == 0
    assert quiet >= 3, quiet
    assert quiet < 50                                             # the lift does stretch springs eventually


def _one_update_from_phases(relax):
    g = load_golden("phases.npz")
    o = OracleCloth(mode="coloured", relax_iters=relax)
    o.set_state(g["pos_0"], g["prev_0"], g["pin_0"], grabbed=g["grabbed"])
    o.adjust(0.0016, -0.0012, 0.0)
    o.update(1)
    return o, g


def test_relax_iters_zero_is_one_pass_and_two_differ():
    o0, _ = _one_update_from_phases(0)
    o1, _ = _one_update_from_phases(1)
    o2, _ = _one_update_from_phases(2)
    assert np.array_equal(o0.pos, o1.pos)
    assert not np.array_equal(o1.pos, o2.pos)
    assert o1.counters()["stretched"] > 0 and o1.counters()["collide_hits"] > 0


def test_one_update_near_reference_order():
    """A sanity bound only (measured 7.6e-4); the pin is the GPU comparison."""
    o, g = _one_update_from_phases(1)
    pos, prev, pin = o.get_state()
    assert np.abs(pos - g["pos_limit"]).max() <= 1e-3
    assert np.array_equal(prev, g["prev_limit"]) and np.array_equal(pin, g["pin_0"])
    assert not o.tear


def test_phases_compose_to_the_update():
    """update() in coloured mode is gravity, Hooke, Verlet, map, Jacobi collision, plane, coloured limit."""
    g = load_golden("phases.npz")
    o, _ = _one_update_from_phases(2)
    p = OracleCloth(mode="coloured", relax_iters=2)
    p.set_state(g["pos_0"], g["prev_0"], g["pin_0"], grabbed=g["grabbed"])
    p.adjust(0.0016, -0.0012, 0.0)
    for name in ("gravity", "hookes", "verlet", "build_map", "self_collide_jacobi", "plane"):
        p.phase(name)
    p.phase("limit_coloured", 2)
    assert np.array_equal(p.pos, o.pos)


def test_jacobi_reads_the_snapshot():
    """Two free points in one bucket, closer than 2*thickness: both move by the same amount in opposite directions
    (in place, the second would see the first one already moved)."""
    P = _params(5)
    o = OracleCloth(P, mode="coloured")
    pos, prev, pin = o.get_state()
    pos[12] = (0.51, 0.5, 0.3); pos[18] = (0.5, 0.5, 0.3)          # two points far from the rest, 0.01 apart
    prev[:] = pos
    o.set_state(pos, prev, pin)
    o.phase("build_map")
    o.phase("self_collide_jacobi")
    q = o.pos
    assert np.array_equal(q[12] - pos[12], -(q[18] - pos[18]))
    assert q[12, 0] > pos[12, 0]
    r = OracleCloth(P)
    r.set_state(pos, prev, pin)
    r.phase("build_map")
    r.phase("self_collide")
    assert not np.array_equal(r.pos[18], q[18])                     # reference order: Gauss-Seidel


def test_coincident_points_raise_zero_division():
    g = load_golden("phases.npz")
    o = OracleCloth(mode="coloured")
    pos = g["pos_0"].copy()
    pos[300] = pos[20]                                            # not connected, one bucket
    o.set_state(pos, g["prev_0"], np.zeros(625, np.uint8))
    o.phase("build_map")
    with pytest.raises(ZeroDivisionError):
        o.phase("self_collide_jacobi")


def test_whole_action_runs_in_coloured_mode():
    ref, col = OracleCloth(), OracleCloth(mode="coloured", relax_iters=2)
    a = np.array([0.1, -0.2, 0.3, 0.2])
    n_r, g_r, ip_r = ref.step_action(a)
    n_c, g_c, ip_c = col.step_action(a)
    assert (n_c, g_c, ip_c) == (n_r, g_r, ip_r) and n_c > 1400
    assert not np.array_equal(ref.pos, col.pos)
    assert abs(ref.coverage() - col.coverage()) < 5e-2
