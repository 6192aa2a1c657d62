"""CPU tests of oracle.desc_ref, the extended-precision descriptor evaluator behind tests/test_gpu_assembly.py: on every
block of every class table, the descriptors of operators.make_desc evaluated by desc_ref (value and d/dtheta) match the
oracle's closed-form blocks (oracle.closed_form in longdouble for the squared exponential, oracle.matern_ref for the
Matern kernels), coincident points included."""
import numpy as np
import pytest

from oracle import blocks_ref, closed_form, desc_ref, matern_ref
from stopro_b200 import operators

LD = np.longdouble


def _blocks_by_dim():
    """{dim: sorted block names used by any class table of that dimension}."""
    out = {}
    for table in blocks_ref.TABLES.values():
        dim = table["dim"]
        if dim is None:
            continue
        names = out.setdefault(dim, set())
        for key in ("training", "mixed", "test"):
            for row in table.get(key, []):
                names.update(row)
    return {d: sorted(n) for d, n in out.items()}


def _points(dim, rng):
    """Random points plus coincident ones: r shares its first points with r', and r' repeats one of its own."""
    r = rng.random((6, dim))
    rp = np.concatenate([r[:3], rng.random((3, dim))])
    rp[4] = rp[3]
    r[5, 0] = rp[5, 0]  # one shared coordinate: s_0 = 0 with s_1 != 0
    return r, rp


def _reference(name, table, kind, form, dim, r, rp, theta, lbox):
    """(value, d/dtheta) of a named block from the closed-form oracle, per hyper-parameter group."""
    terms, shift = blocks_ref.parse_spec(table["blocks"][name], table["blocks"])
    val = np.zeros((len(r), len(rp)), dtype=LD)
    grad = np.zeros((len(theta), len(r), len(rp)), dtype=LD)
    groups = list(table["groups"].values())
    for sign, op, group in terms:
        sl = table["groups"][group]
        idx = np.arange(len(theta))[sl]

        def base(a, b):
            if kind == "se":
                return closed_form.eval_operator(op, a, b, theta[sl].astype(LD), form, dim, with_grad=True, dtype=LD)
            v, g = matern_ref.eval_operator(kind, op, a, b, theta[sl], form, dim, with_grad=True)
            return v.astype(LD), g.astype(LD)

        combos = {None: [(1, 0, 0)], "Xp": [(1, 0, 1), (-1, 0, 0)], "X": [(1, 1, 0), (-1, 0, 0)],
                  "XX": [(1, 1, 1), (-1, 1, 0), (-1, 0, 1), (1, 0, 0)]}[shift]
        for sg, sa, sb in combos:
            # the oracle differences its arguments itself: hand it the float64 differences the kernels form (r + lbox
            # first, then the difference) against a zero second point
            s = ((r + sa * lbox)[:, None, :] - (rp + sb * lbox)[None, :, :]).reshape(-1, dim)
            v, g = base(s, np.zeros((1, dim)))
            val += sign * sg * v.reshape(val.shape)
            grad[idx] += sign * sg * g.reshape((len(idx),) + val.shape)
        assert len(groups) * len(idx) == len(theta)
    return val, grad


@pytest.mark.parametrize("kind", ["se", "mt52", "mt72", "mt92"])
@pytest.mark.parametrize("form", ["product", "additive"])
def test_desc_ref_matches_closed_form_blocks(kind, form):
    rng = np.random.default_rng(7)
    tables = {2: blocks_ref.TABLES["poiseuille"], 3: blocks_ref.TABLES["stokes3d"], 1: blocks_ref.TABLES["laplacian1d"]}
    checked = 0
    for dim, names in _blocks_by_dim().items():
        table = tables[dim]
        obs, fields = operators.stokes_observables(dim) if dim > 1 else operators.scalar_observables(1)
        theta = 0.4 * rng.standard_normal(len(fields) * (1 + dim))
        lbox = np.array([1.75, 0.5, 0.0])[:dim]
        r, rp = _points(dim, rng)
        for name in names:
            if name not in table["blocks"]:
                continue
            oa, ob = operators.parse_block_name(name, obs)
            desc = operators.make_desc(oa, ob, fields, dim, form == "product")
            want, want_g = _reference(name, table, kind, form, dim, r, rp, theta, lbox)
            first = np.repeat(r, len(rp), axis=0)
            second = np.tile(rp, (len(r), 1))
            got, got_g, A, U, dabs = desc_ref.eval_desc_all(desc, dim, first, second, theta, lbox, form == "product", kind)
            got, got_g = got.reshape(want.shape), got_g.reshape(want_g.shape)
            A, dabs = A.reshape(want.shape), dabs.reshape(want_g.shape)
            # longdouble against longdouble for the squared exponential; the Matern oracle is float64
            tol = 1e-17 if kind == "se" else 1e-13
            assert np.all(np.abs(got - want) <= tol * (A + 1e-300)), name
            assert np.all(np.abs(got_g - want_g) <= tol * (dabs + 1e-300)), name
            assert np.all(np.abs(got) <= A * (1 + 1e-15)) and np.all(U >= 0)
            checked += 1
    assert checked >= 100


def test_float64_block_matches_longdouble():
    """eval_desc in float64 (the CPU check of the descriptor compiler in tests/test_host.py) agrees with longdouble."""
    rng = np.random.default_rng(3)
    obs, fields = operators.stokes_observables(2)
    desc = operators.make_desc(obs["fx"], obs["difux"], fields, 2, True)
    r, rp, theta = rng.random((5, 2)), rng.random((4, 2)), 0.3 * rng.standard_normal(9)
    a = desc_ref.eval_desc(desc, 2, r, rp, theta, lbox=[2.5, 0.0])
    b = desc_ref.eval_desc(desc, 2, r, rp, theta, lbox=[2.5, 0.0], dtype=LD)
    assert a.dtype == np.float64 and b.dtype == LD
    assert np.max(np.abs(a - b)) <= 1e-13 * np.max(np.abs(b))
