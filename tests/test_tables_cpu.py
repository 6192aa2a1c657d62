"""CPU test: every block of every class table (training / mixed / test) that stopro_b200 derives from its observables
equals the block the reference's class puts in that slot (oracle.blocks_ref.TABLES restates the reference tables name
by name), evaluated on random points.  Covers the BASELINE classes and the other live classes of SURVEY.md 8(f) n2."""
import numpy as np
import pytest

from oracle import blocks_ref, closed_form
from oracle.desc_ref import eval_desc
from stopro_b200 import synthetic
from stopro_b200 import operators

MODELS = {
    "naive": lambda: synthetic.sin_1d_naive(),
    "laplacian1d": lambda: synthetic.sin_1d_laplacian(),
    "poiseuille": lambda: synthetic.poiseuille(kernel_form="product"),
    "poiseuille_additive": lambda: synthetic.poiseuille(kernel_form="additive"),
    "sinusoidal": lambda: synthetic.sinusoidal(u_num=6, f_nx=5, f_ny=3, dif_num=4, n_test=4),
    "sinusoidal_infer_gov": lambda: dict(synthetic.sinusoidal(u_num=6, f_nx=5, f_ny=3, dif_num=4, n_test=4),
                                         model="sinusoidal_infer_gov",
                                         model_kwargs=dict(lbox=np.array([2.5, 0.0]), use_difp=True, use_difu=True,
                                                           infer_governing_eqs=True)),
    "sinusoidal_infer_difp": lambda: synthetic.sinusoidal_without_difp("infer_difp", u_num=6, f_nx=5, f_ny=3, dif_num=4, n_test=4),
    "sinusoidal_infer_u_without_difp": lambda: synthetic.sinusoidal_without_difp("infer_u_without_difp", u_num=6, f_nx=5, f_ny=3, dif_num=4, n_test=4),
    "sinusoidal_infer_gov_without_difp": lambda: synthetic.sinusoidal_without_difp("infer_gov_without_difp", u_num=6, f_nx=5, f_ny=3, dif_num=4, n_test=4),
    "stokes3d": lambda: synthetic.drag3d(n_u=3, n_f=3, n_test=4),
    "stokes3d_infer_difp": lambda: synthetic.drag3d_variant("stokes3d_infer_difp", n_u=3, n_f=3, n_test=4),
    "stokes3d_naive": lambda: synthetic.drag3d_variant("stokes3d_naive", n_u=3, n_f=3, n_test=4),
    "stokes2d2c": lambda: synthetic.drag3d_variant("stokes2d2c", n_u=3, n_f=3, n_test=4),
    "stokes2d2c_surface": lambda: synthetic.drag3d_variant("stokes2d2c_surface", n_u=3, n_f=3, n_test=4),
}


@pytest.mark.parametrize("name", list(MODELS))
def test_class_tables_match_the_reference_tables(name):
    cfg = MODELS[name]()
    gp = synthetic.make_model(cfg)  # no device work: plans are compiled in set_constants
    table = blocks_ref.TABLES[cfg["model"]]
    dim, form = gp.dim, ("product" if gp.product_form else "additive")
    rng = np.random.default_rng(5)
    n_theta = len(gp._fields) * (1 + dim)
    theta = 0.3 * rng.standard_normal(n_theta)
    lbox = None if gp.lbox is None else np.asarray(gp.lbox, dtype=float)
    shape = (lambda n: (n,)) if dim == 1 else (lambda n: (n, dim))
    r, rp = rng.random(shape(4)), rng.random(shape(3))

    def op_eval(op, a, b, th):
        return closed_form.eval_operator(op, a, b, th, form, dim)

    def check(obs_a, obs_b, block_name, zero=False):
        want = blocks_ref.eval_block(block_name, table, op_eval, r, rp, theta, lbox, lambda n, m: np.zeros((n, m)))
        desc = operators.make_desc(obs_a, obs_b, gp._fields, dim, gp.product_form)
        got = np.zeros_like(want) if zero else eval_desc(desc, dim, r, rp, theta, lbox, product=gp.product_form)
        assert np.max(np.abs(got - want)) <= 1e-12 * max(np.max(np.abs(want)), 1.0), (name, block_name)

    tr = gp._observables(gp.train_observables)
    te = gp._observables(gp.test_observables)
    assert len(tr) == len(table["training"]) and len(te) == len(table["test"]) == len(table["mixed"])
    for i in range(len(tr)):
        for j in range(i, len(tr)):
            check(tr[i], tr[j], table["training"][i][j - i])
    for i in range(len(te)):
        assert len(table["mixed"][i]) == len(tr)
        for j in range(len(tr)):
            check(te[i], tr[j], table["mixed"][i][j])
        for j in range(i, len(te)):
            check(te[i], te[j], table["test"][i][j - i], zero=(i, j) in gp.test_zero_blocks)
