"""CPU: the numpy oracle against the reference's golden vectors / recorded outputs.

The fixtures under tests/golden were produced by running the unmodified reference
(tests/golden/make_golden.py); this file is what "pins" the oracle (SURVEY 8c).
"""
import json

import numpy as np
import pytest

import oracle
from conftest import pairs_to_set, rel_fro


def test_pair_sd_and_constraint_sets(small_cln):
    coords = small_cln["coords"]
    sds = oracle.pair_distance_sd(coords)
    assert np.allclose(sds, small_cln["sds"], rtol=1e-9, atol=1e-12)
    assert oracle.guess_pairwise_constraints(coords[:10]) == pairs_to_set(small_cln["cons10"])
    assert oracle.guess_pairwise_constraints(coords) == pairs_to_set(small_cln["cons_all"])
    # float32 evaluation of the reference agrees on this (well separated) data: Q10
    assert pairs_to_set(small_cln["cons10_f32"]) == pairs_to_set(small_cln["cons10"])
    cross = oracle.guess_pairwise_constraints(coords[:, :60], cross_xyz=coords[:, 40:90])
    assert cross == {(int(i), int(j)) for i, j in small_cln["cross_pairs"]}
    assert len(cross) > 0


@pytest.mark.parametrize("cross", [False, True])
def test_pair_distance_moments_give_pair_distance_sd(small_cln, cross):
    """The per-pair moments (the quantity kernel (c) accumulates) reproduce pair_distance_sd on a pair
    list, for any shift: a shift only moves the moments, not the variance they imply."""
    coords = small_cln["coords"][:, :60]
    other = small_cln["coords"][:, 40:90] if cross else None
    sds = oracle.pair_distance_sd(coords, other)
    rng = np.random.default_rng(0)
    ii, jj = np.nonzero(np.ones_like(sds))
    pick = rng.choice(ii.size, 300, replace=False)
    pairs = np.stack([ii[pick], jj[pick]], axis=1)
    o = coords if other is None else other
    frame0 = np.linalg.norm(coords[0, pairs[:, 1]].astype(np.float64) - o[0, pairs[:, 0]], axis=-1)
    T = coords.shape[0]
    for shift in (frame0, np.zeros(len(pairs)), frame0 + rng.normal(0, 0.1, len(pairs))):
        s1, s2 = oracle.pair_distance_moments(coords, other, pairs, shift)
        assert s1.shape == s2.shape == (len(pairs),)
        # M2 = s2 - s1^2 / T loses what the shift leaves of the mean: compare on the scale of s2
        m2_ref = T * sds[pairs[:, 0], pairs[:, 1]] ** 2
        assert np.all(np.abs((s2 - s1 * s1 / T) - m2_ref) <= 1e-12 * s2 + 1e-300)
    # by definition: sum of e and of e^2 over frames
    d = np.linalg.norm(coords[:, pairs[:3, 1]].astype(np.float64) - o[:, pairs[:3, 0]], axis=-1)
    s1, s2 = oracle.pair_distance_moments(coords, other, pairs[:3], frame0[:3])
    assert np.allclose(s1, (d - frame0[:3]).sum(0), rtol=1e-13, atol=1e-13)
    assert np.allclose(s2, ((d - frame0[:3]) ** 2).sum(0), rtol=1e-13, atol=1e-16)


def test_constraints_are_the_xh_bonds(small_cln):
    from aggforce_b200.synth import chignolin_topology

    topo = chignolin_topology()
    assert pairs_to_set(small_cln["cons10"]) == topo.xh_constraints
    assert len(topo.xh_constraints) == 78


def test_gram_linear_matches_reference(small_cln):
    forces = small_cln["forces"]
    cons = pairs_to_set(small_cln["cons10"])
    assert rel_fro(oracle.gram_linear(forces, cons), small_cln["gram_raw"]) < 1e-13
    assert rel_fro(oracle.gram_linear(forces, ()), small_cln["gram_nocons"]) < 1e-13
    p = oracle.gram_linear(forces, cons) + 1e3 * oracle.l2_linear_term(forces.shape[1], cons)
    assert rel_fro(p, small_cln["gram_l2_1e3"]) < 1e-13
    assert p.shape == (97, 97)


def test_linear_weights_match_reference(small_cln):
    from aggforce_b200.synth import chignolin_topology

    topo = chignolin_topology()
    cm = np.zeros((10, 175))
    cm[np.arange(10), topo.bead_atoms] = 1
    cons = pairs_to_set(small_cln["cons10"])
    w = oracle.qp_linear_weights(small_cln["forces"], cm, cons, 1e3)
    assert rel_fro(w, small_cln["W_l2_1e3"]) < 1e-8
    assert np.allclose(cm @ w.T, np.eye(10), atol=1e-10)
    mapped = oracle.apply_map(small_cln["forces"], w)
    assert rel_fro(mapped, small_cln["mapped_forces"]) < 1e-8
    assert abs(oracle.force_smoothness(mapped) / small_cln["residual"] - 1) < 1e-8
    assert rel_fro(oracle.apply_map(small_cln["coords"], cm), small_cln["mapped_coords"]) < 1e-12


def test_uni_map_matches_reference_goldens(small_cln, golden):
    from aggforce_b200.synth import chignolin_topology

    topo = chignolin_topology()
    cm = np.zeros((10, 175))
    cm[np.arange(10), topo.bead_atoms] = 1
    uni = oracle.uni_map_matrix(cm, topo.xh_constraints)
    assert np.array_equal(uni, small_cln["uni_matrix"])
    # the reference's own golden file (tests/test_forces.py:154-157): exact
    assert ((uni - np.loadtxt(golden / "cln_basic_force_mat.txt")) ** 2).sum() < 1e-5
    assert uni.sum() == 21


def test_opt_golden_structure(golden):
    """cln_opt_force_mat.txt came from the real trajectory (not available): check the
    invariants any correct solution has -- it lies in range(C) for the X-H groups and
    satisfies the equality constraints."""
    from aggforce_b200.synth import chignolin_topology

    topo = chignolin_topology()
    w = np.loadtxt(golden / "cln_opt_force_mat.txt")
    cols = oracle.group_columns(175, topo.xh_constraints)
    assert cols.max() + 1 == 97
    for g in range(97):
        members = np.nonzero(cols == g)[0]
        assert np.abs(w[:, members] - w[:, members[:1]]).max() < 1e-12
    cm = np.zeros((10, 175))
    cm[np.arange(10), topo.bead_atoms] = 1
    a = cm @ oracle.bond_constraint_matrix(175, topo.xh_constraints)
    x = np.stack([w[:, np.nonzero(cols == g)[0][0]] for g in range(97)], axis=1)
    assert np.abs(a @ x.T - np.eye(10)).max() < 1e-12


def test_waterdimer_known_answer(golden):
    """tests/test_agg.py:17-44 of the reference with the exact solve."""
    forces = np.load(golden / "waterdimer.npz")["Fs"]
    cm = np.zeros((2, 6))
    cm[0, 0] = cm[1, 3] = 1
    w = oracle.qp_linear_weights(forces, cm, (), 0.0)
    expected = np.array([[1, 1, 1, 0, 0, 0], [0, 0, 0, 1, 1, 1]], dtype=float)
    assert np.allclose(w, expected, atol=5e-3)


def test_id_feature_gram_matches_reference(small_cln, golden):
    ref = np.load(golden / "ref_idfeat.npz")
    feats, divs = oracle.id_features(small_cln["forces"].shape[0], ref["ids"])
    p = oracle.feat_gram(small_cln["forces"], feats, divs, float(ref["kbt"]), 1e1)
    # the reference builds this Gram in float32 (SURVEY Q4): agreement to f32 accuracy
    for bead in range(ref["P"].shape[0]):
        assert rel_fro(ref["P"][bead], p) < 5e-6
    from aggforce_b200.synth import chignolin_topology

    cm = np.zeros((10, 175))
    cm[np.arange(10), chignolin_topology().bead_atoms] = 1
    a, b = oracle.feat_constraint_rows(feats, cm, 3, ref["frame_choice"])
    assert np.array_equal(a, ref["A"][3]) and np.array_equal(b, ref["b"][3])
    coefs = [oracle.solve_equality_qp(p, *oracle.feat_constraint_rows(feats, cm, c, ref["frame_choice"]))
             for c in range(10)]
    assert rel_fro(np.stack(coefs), ref["coefs"]) < 1e-4
    mapped = oracle.feat_map_apply(small_cln["forces"], [feats] * 10, [divs] * 10, coefs)
    assert rel_fro(mapped, ref["mapped_forces"]) < 1e-4


def test_id_gram_equals_linear_gram(small_cln, golden):
    """One-hot id features collapse the atom contraction to the group sum (SURVEY 8a)."""
    ref = np.load(golden / "ref_idfeat.npz")
    feats, divs = oracle.id_features(small_cln["forces"].shape[0], ref["ids"])
    p = oracle.feat_gram(small_cln["forces"], feats, divs, 0.7, 0.0)
    g = oracle.gram_linear(small_cln["forces"], pairs_to_set(small_cln["cons10"]))
    cols = oracle.group_columns(175, pairs_to_set(small_cln["cons10"]))
    perm = np.array([ref["ids"][np.nonzero(cols == c)[0][0]] for c in range(97)])
    assert rel_fro(p[np.ix_(perm, perm)], g) < 1e-13


def test_gb_divergence_against_finite_differences():
    rng = np.random.default_rng(3)
    n, T = 9, 4
    x = rng.uniform(0, 6, size=(T, n, 3))
    cons = {frozenset((0, 1)), frozenset((1, 2)), frozenset((5, 6))}
    labels = oracle.canonical_labels(n, cons)
    cm = np.zeros((2, n))
    cm[0, 3] = 1.0
    cm[1, [0, 7]] = 0.5
    kw = dict(outer=8.0, inner=0.0, n_basis=7, width=1.0)
    for bead in (0, 1):
        for drop in (True, False):
            feats, divs = oracle.gb_features(x, cm, cons, labels, bead, drop_last_channel=drop, **kw)
            fd = oracle.gb_divergence_fd(x, cm, cons, labels, bead, drop_last_channel=drop, **kw)
            ok = np.isfinite(divs)
            assert np.abs(divs[ok] - fd[ok]).max() < 1e-6
            # an unconstrained bead atom sits on the bead: NaN there (SURVEY Q6), finite elsewhere
            if bead == 1:
                assert ok.all()
            n_ch = labels.max() + (0 if drop else 1)
            assert feats.shape == (T, n, n_ch * 7) and divs.shape == (T, n_ch * 7, 3)
    mu = oracle.gb_centers(0.0, 8.0, 7)
    assert np.allclose(mu, 8 * np.arange(7) ** 2 / 36.0)


def test_condnormal_closed_form(golden):
    ref = np.load(golden / "ref_condnormal.npz")
    var = float(ref["var"])
    src, gen = ref["source"].astype(np.float64), ref["generated"].astype(np.float64)
    noise = (gen - src) / np.sqrt(var)
    eye = np.eye(src.shape[1])
    coords, forces = oracle.gauss_augment(src, np.zeros_like(src), eye, var, 1.0, noise)
    n = src.shape[1]
    assert np.allclose(coords[:, n:], gen, atol=1e-5)
    assert np.allclose(forces[:, :n], ref["lg_source"], rtol=2e-5, atol=2e-5)
    assert np.allclose(forces[:, n:], ref["lg_generated"], rtol=2e-5, atol=2e-5)


def test_merge_groups_matches_reference(golden):
    cases = json.loads((golden / "ref_sets.json").read_text())["cases"]
    for case in cases:
        merged = oracle.merge_constraint_groups(case["constraints"])
        assert sorted(list(g) for g in merged) == case["reduced"]


def test_apply_nan_protocol(golden):
    ref = np.load(golden / "ref_linearmap.npz")
    out = oracle.apply_map_nan_protocol(ref["pos_nan"], ref["slice_matrix"])
    assert np.allclose(out, ref["nan_out"], rtol=0, atol=1e-12)
    dense = ref["mat"]
    with pytest.raises(ValueError):
        oracle.apply_map_nan_protocol(ref["pos_nan"], dense)
    assert np.allclose(oracle.apply_map(ref["pos"], dense), ref["mapped"], rtol=1e-13)


# --------------------------------------------------------------------------------------
# the JAX half: fixtures from the reference's own jaxfeat / jaxgausstraj / jgauss / jaxmapval run
# behind tests/golden/jax_shim (tests/golden/make_golden_jax.py).  float32 reference -> float32 bars.
# --------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def gbfix(golden):
    return dict(np.load(golden / "ref_gbfeat.npz"))


@pytest.fixture(scope="module")
def jcn(golden):
    return dict(np.load(golden / "ref_jcondnormal.npz"))


F32_ABS = 5e-6  # float32 features are O(1); divergences O(1)


@pytest.mark.parametrize("nb", [4, 7])
@pytest.mark.parametrize("dm", ["reorder", "basic"])
def test_gb_features_match_reference_small(gbfix, nb, dm):
    """Slice map on the 12-site system: bead 1 sits on site 4, the only site of the LARGEST label
    (its feature block is dropped, Q5) and coincides with its own smeared position (Q6)."""
    x, ids = gbfix["small_x"], gbfix["small_ids"]
    cons = [tuple(p) for p in gbfix["small_cons"]]
    cm = gbfix["small_cmap_slice"]
    assert ids[4] == ids.max() and (ids == ids.max()).sum() == 1
    feats, divs = gbfix[f"small_slice_nb{nb}_{dm}_feats"], gbfix[f"small_slice_nb{nb}_{dm}_divs"]
    assert feats.shape == (3, 6, 12, nb * ids.max()) and divs.shape == (3, 6, nb * ids.max(), 3)
    for bead in range(3):
        of, od = oracle.gb_features(x, cm, cons, ids, bead, outer=8, inner=0, n_basis=nb, width=1.0, div_method=dm)
        assert np.abs(feats[bead] - of).max() < F32_ABS
        assert np.abs(feats[bead][:, 4]).max() == 0.0  # top-label site: all-zero feature row in the reference
        assert np.array_equal(np.isnan(divs[bead]), np.isnan(od))
        ok = ~np.isnan(od)
        assert not ok.any() or np.abs(divs[bead][ok] - od[ok]).max() < F32_ABS
    # the two readings of Q6 for the coincident bead: reverse mode poisons the frame, forward mode does not
    assert np.isnan(gbfix[f"small_slice_nb{nb}_reorder_divs"][1]).all()
    assert not np.isnan(gbfix[f"small_slice_nb{nb}_basic_divs"][1]).any()
    # keeping the last channel (our switch) only APPENDS a block: the reference part is unchanged
    of_keep, _ = oracle.gb_features(x, cm, cons, ids, 0, outer=8, inner=0, n_basis=nb, width=1.0,
                                    drop_last_channel=False)
    of_drop, _ = oracle.gb_features(x, cm, cons, ids, 0, outer=8, inner=0, n_basis=nb, width=1.0)
    assert np.array_equal(of_keep[..., : of_drop.shape[-1]], of_drop) and np.abs(of_keep[:, 4, -nb:]).max() > 0


def test_gb_features_match_reference_com_and_alt_parameters(gbfix):
    x, ids = gbfix["small_x"], gbfix["small_ids"]
    cons = [tuple(p) for p in gbfix["small_cons"]]
    cm = gbfix["small_cmap_com"]
    feats, divs = gbfix["small_com_nb7_basic_feats"], gbfix["small_com_nb7_basic_divs"]
    for bead in range(3):
        of, od = oracle.gb_features(x, cm, cons, ids, bead, outer=8, inner=0, n_basis=7, width=1.0)
        assert np.abs(feats[bead] - of).max() < F32_ABS
        # a centre-of-group bead coincides with its group's smeared position up to float32 rounding: the
        # direction of that channel's divergence is rounding noise in the reference -- compare the others
        ch = int(ids[np.argmax(cm[bead] > 0)])
        keep = np.ones(od.shape[1], dtype=bool)
        if ch < ids.max():
            keep[ch * 7 : (ch + 1) * 7] = False
        assert np.abs(divs[bead][:, keep] - od[:, keep]).max() < F32_ABS
    cm = gbfix["small_cmap_slice"]
    for bead in (0, 2):
        of, od = oracle.gb_features(x, cm, cons, ids, bead, outer=6.5, inner=0.5, n_basis=5, width=0.7, dist_power=1.0)
        assert np.abs(gbfix["small_alt_feats"][bead] - of).max() < F32_ABS
        assert np.abs(gbfix["small_alt_divs"][bead] - od).max() < 2e-5


def test_gb_features_match_reference_cln025(gbfix, small_cln):
    from aggforce_b200.synth import chignolin_topology

    topo = chignolin_topology()
    coords = small_cln["coords"][:4]
    cons = pairs_to_set(small_cln["cons10"])
    cm = np.zeros((10, 175))
    cm[np.arange(10), topo.bead_atoms] = 1
    ids = gbfix["cln_ids"]
    assert ids.max() == 96
    for bead in (0, 7):
        of, od = oracle.gb_features(coords, cm, cons, ids, bead, outer=8, inner=0, n_basis=7, width=1.0,
                                    div_method="reorder")
        assert gbfix[f"cln_feats_b{bead}"].shape == (4, 175, 672)
        assert np.abs(gbfix[f"cln_feats_b{bead}"] - of).max() < F32_ABS
        assert np.abs(gbfix[f"cln_divs_b{bead}"] - od).max() < 2e-5


def test_featurised_fit_matches_reference(gbfix):
    """qp_feat_linear_map(Multifeaturize([id_feat, Curry(gb_feat, n_basis=4)])) of the reference on a
    40-site sub-system: Gram (float32 in the reference), equality rows, coefficients, mapped forces."""
    c, f, ids = gbfix["fit_coords"], gbfix["fit_forces"], gbfix["fit_ids"]
    cons = pairs_to_set(gbfix["fit_cons"])
    beads = gbfix["fit_beads"]
    cm = np.zeros((len(beads), c.shape[1]))
    cm[np.arange(len(beads)), beads] = 1
    kbt, l2 = float(gbfix["fit_kbt"]), float(gbfix["fit_l2"])
    idf, idd = oracle.id_features(len(c), ids)
    feats, divs, coefs = [], [], []
    for bead in range(len(beads)):
        gf, gd = oracle.gb_features(c, cm, cons, ids, bead, outer=8.0, inner=0.0, n_basis=4, width=1.0)
        ph, dv = np.concatenate([idf, gf], axis=2), np.concatenate([idd, gd], axis=1)
        p = oracle.feat_gram(f, ph, dv, kbt, l2)
        assert p.shape == gbfix["fit_P"][bead].shape
        assert rel_fro(p, gbfix["fit_P"][bead]) < 2e-6  # the reference accumulates this Gram in float32
        a, b = oracle.feat_constraint_rows(ph, cm, bead, gbfix["fit_frame_choice"])
        assert np.abs(a - gbfix["fit_A"][bead]).max() < F32_ABS and np.array_equal(b, gbfix["fit_b"][bead])
        # the fitted coefficients amplify the Gram's float32 error: check through the solver on the
        # reference's own (P, A, b), and the mapped forces with the reference's coefficients
        sol = oracle.solve_equality_qp(gbfix["fit_P"][bead], gbfix["fit_A"][bead], gbfix["fit_b"][bead])
        assert rel_fro(sol, gbfix["fit_coefs"][bead]) < 1e-6
        feats.append(ph), divs.append(dv), coefs.append(gbfix["fit_coefs"][bead])
    mapped = oracle.feat_map_apply(f, feats, divs, coefs)
    assert rel_fro(mapped, gbfix["fit_mapped_forces"]) < 5e-6


@pytest.mark.parametrize("name", ["slice", "avg"])
def test_jcondnormal_matches_reference(jcn, name):
    src, var, a = jcn["source"], float(jcn["var"]), jcn[f"{name}_matrix"]
    gen, z = jcn[f"{name}_generated"], jcn[f"{name}_z"]
    # sample: y = A x + sqrt(var) z with the recorded standard-normal draw
    y = np.einsum("cf,tfd->tcd", a, src.astype(np.float64)) + np.sqrt(var) * z
    assert np.abs(gen - y).max() < 1e-5
    gx, gy = oracle.gauss_log_gradient(src, gen, a, var)
    assert np.abs(jcn[f"{name}_lg_source"] - gx).max() < 2e-5 * max(1.0, np.abs(gx).max())
    assert np.abs(jcn[f"{name}_lg_generated"] - gy).max() < 2e-5 * max(1.0, np.abs(gy).max())


def test_jcondnormal_identity_premap(jcn):
    gx, gy = oracle.gauss_log_gradient(jcn["source"][:, :6], jcn["ident_generated"], None, float(jcn["var"]))
    assert np.abs(jcn["ident_lg_source"] - gx).max() < 2e-5 and np.abs(jcn["ident_lg_generated"] - gy).max() < 2e-5


def test_joptgauss_matches_reference(jcn, gbfix):
    """joptgauss_map of the reference end to end (jgauss.py:114-138), with the noise it drew."""
    c, f = gbfix["fit_coords"], gbfix["fit_forces"]
    cons = pairs_to_set(jcn["jopt_cons"])
    beads = jcn["jopt_beads"]
    n_fg, n_cg = c.shape[1], len(beads)
    cm = np.zeros((n_cg, n_fg))
    cm[np.arange(n_cg), beads] = 1
    var, kbt, l2 = float(jcn["jopt_var"]), float(jcn["jopt_kbt"]), float(jcn["jopt_l2"])
    xa, fa = oracle.gauss_augment(c, f, cm, var, kbt, jcn["jopt_z_fit"])
    p = oracle.gram_linear(fa, cons) + l2 * oracle.l2_linear_term(n_fg + n_cg, cons)
    assert rel_fro(p, jcn["jopt_P"]) < 5e-6  # float32 augmented forces in the reference
    aug_cm = np.zeros((n_cg, n_fg + n_cg))
    aug_cm[np.arange(n_cg), n_fg + np.arange(n_cg)] = 1
    assert np.array_equal(aug_cm, jcn["jopt_coord_matrix"])
    w = oracle.qp_linear_weights(fa, aug_cm, cons, l2)
    assert rel_fro(w, jcn["jopt_W"]) < 1e-4
    xa2, fa2 = oracle.gauss_augment(c, f, cm, var, kbt, jcn["jopt_z_apply"])
    assert rel_fro(oracle.apply_map(xa2, aug_cm), jcn["jopt_mapped_coords"]) < 1e-6
    assert rel_fro(oracle.apply_map(fa2, jcn["jopt_W"]), jcn["jopt_mapped_forces"]) < 1e-5


def test_validation_projections_match_reference(golden):
    mvf = dict(np.load(golden / "ref_mapval.npz"))
    c, f = mvf["cg_coords"], mvf["cg_forces"]
    for s in range(3):
        off, w = oracle.rsqpg_offset(6.0, 12.0, 0.5, np.random.default_rng(s))
        assert abs(off - mvf["rsqpg_offsets"][s]) < 1e-12
        ref = mvf["rsqpg_forces"][s]
        assert np.abs(oracle.sq_gaussian_forces(c, off, w) - ref).max() < 1e-4 * max(1.0, np.abs(ref).max())
    off, w = oracle.rsqpg_offset(30.0, 80.0, 9.0, np.random.default_rng(1), sq_args=False)
    ref = mvf["rsqpg_forces_nosq"]
    assert np.abs(oracle.sq_gaussian_forces(c, off, w) - ref).max() < 1e-4 * max(1.0, np.abs(ref).max())
    kw = dict(inner=6.0, outer=12.0, width=0.5)
    proj = oracle.random_force_proj(c, f, 16, np.random.default_rng(42100), **kw)
    scale = np.abs(mvf["proj"]).max()
    assert np.abs(np.asarray(proj) - mvf["proj"]).max() < 1e-4 * scale
    assert abs(np.mean(proj) - mvf["proj_avg"]) < 1e-4 * scale
    shift = oracle.random_residual_shift(c, f, 16, np.random.default_rng(42100), **kw)
    # the reference subtracts two O(mean F^2) float numbers: absolute bar at that scale
    bar = 1e-5 * float(np.mean(f.astype(np.float64) ** 2)) + 1e-4 * np.abs(mvf["shift"]).max()
    assert np.abs(np.asarray(shift) - mvf["shift"]).max() < bar
    assert abs(np.mean(shift) - mvf["shift_avg"]) < bar
