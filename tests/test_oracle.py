"""CPU: pins the oracle against everything the reference offers for this path (SURVEY 4, 8c):
LQR gains, parameter trees of the pretrained pickles, closed-form geometry, the
dense (reference layout) == sparse equivalence, label semantics, optimizer restatement."""
import hashlib
import json
import os

import numpy as np
import pytest
import torch

from helpers import GOLDEN, ENVS, oracle_env, oracle_obstacles, oracle_params, random_scene
from oracle.algo import (AdamW, act, compute_norm_and_clip, gcbf_plus_loss, get_cbf, polyak, rates, rollout,
                         safe_mask_horizon, train_step)
from oracle.envs import OracleEnv
from oracle.geometry import Rectangle, Sphere, get_lidar, ray_table_2d, ray_table_3d


def test_lqr_gains_known_answers():
    """SURVEY 8a6 (recomputed there with scipy 1.18 from the reference's A, B, Q, R)."""
    K = OracleEnv("DoubleIntegrator", 2, 4.0).K
    np.testing.assert_allclose(K, [[1.5850302, 0, 1.70600375, 0], [0, 1.5850302, 0, 1.70600375]], atol=1e-7)
    K = OracleEnv("SingleIntegrator", 2, 4.0).K
    np.testing.assert_allclose(K, 1.38453172 * np.eye(2), atol=1e-7)
    K = OracleEnv("LinearDrone", 2, 2.0).K
    np.testing.assert_allclose(np.diag(K[:, :3]), [0.63123451, 0.63123451, 0.6365321], atol=1e-7)
    np.testing.assert_allclose(np.diag(K[:, 3:]), [0.11461079, 0.11461079, 0.10032613], atol=1e-7)


@pytest.mark.parametrize("env_id,n_actor,n_cbf", [("SingleIntegrator", 365955, 365698), ("DoubleIntegrator", 366467, 366210),
                                                 ("DubinsCar", 366467, 366210), ("LinearDrone", 367236, 366722)])
def test_pretrained_fixture_counts(env_id, n_actor, n_cbf):
    z = np.load(os.path.join(GOLDEN, f"params_{env_id}.npz"))
    assert sum(z[k].size for k in z.files if k.startswith("actor:")) == n_actor
    assert sum(z[k].size for k in z.files if k.startswith("cbf:")) == n_cbf
    ed = {"SingleIntegrator": 2, "DoubleIntegrator": 4, "DubinsCar": 4, "LinearDrone": 6}[env_id]
    assert z["cbf:params/GNN_0/GNNLayer_0/msg/Dense_0/kernel"].shape == (ed + 6, 256)
    assert z["cbf:params/GNN_0/GNNLayer_0/update/Dense_0/kernel"].shape == (131, 256)


def test_fixture_equals_reference_pickle():
    """params_<Env>.npz of every environment holds exactly the leaves of the reference's pretrained {actor,cbf}.pkl:
    shapes, SHA-256 of the float32 bytes and a seeded sample of values, as recorded from the pickles by
    tests/golden/make_pickle_digests.py."""
    g = np.load(os.path.join(GOLDEN, "ref_pickle_digests.npz"))
    meta = json.loads(str(g["meta"]))
    assert sorted(meta) == sorted(ENVS)
    for env_id in ENVS:
        want = meta[env_id]
        z = np.load(os.path.join(GOLDEN, f"params_{env_id}.npz"))
        assert sorted(z.files) == sorted(want), env_id
        for k, m in want.items():
            v = z[k]
            assert v.dtype == np.float32 and list(v.shape) == m["shape"], (env_id, k, v.dtype, v.shape)
            lo, hi = m["sample"]
            np.testing.assert_array_equal(v.ravel()[g["index"][lo:hi]], g["value"][lo:hi], err_msg=f"{env_id} {k}")
            assert hashlib.sha256(np.ascontiguousarray(v).tobytes()).hexdigest() == m["sha256"], (env_id, k)


def test_rectangle_raycast_closed_form():
    """Axis-aligned unit square at (2,0): ray from origin along +x hits at x = 1.5."""
    rect = Rectangle.create([[2.0, 0.0]], [1.0], [1.0], [0.0])
    tab = ray_table_2d(32, 2.0)                       # ray 16 is theta = 0, rays 15/17 are -/+ 11.25 deg
    hits = get_lidar(torch.tensor([0.0, 0.0]), rect, tab, 32)
    t = 1.5 * np.tan(np.pi / 16)
    got = sorted(hits[:2].tolist(), key=lambda p: p[1])
    np.testing.assert_allclose(got, [[1.5, -t], [1.5, t]], atol=1e-6)
    # reference quirk kept: the exactly horizontal ray is parallel to two edges of an axis-aligned
    # rectangle -> det == 0 -> sign(0) * clip = 0 -> alpha = x/0 -> NaN through jnp.min; NaNs sort last
    assert torch.isnan(hits[-1]).any()
    # rays that miss land 1e6 ranges away (obstacle.py:94)
    assert hits[-2].abs().max() > 1e5
    # inside the obstacle: every alpha is 0 -> all hit points equal the start (env/utils.py:124)
    hits_in = get_lidar(torch.tensor([2.0, 0.1]), rect, tab, 32)
    assert torch.equal(hits_in[:31], torch.tensor([2.0, 0.1]).expand(31, 2))      # (NaN * 0 = NaN: the quirk ray)
    assert rect.inside(torch.tensor([[2.0, 0.0], [2.55, 0.0], [2.6, 0.6]]), 0.1).squeeze(-1).tolist() == [True, True, False]


def test_sphere_raycast_closed_form_and_topk():
    sph = Sphere.create([[0.0, 0.0, 1.0]], [0.25])
    tab = ray_table_3d(32, 2.0)
    assert tab.shape == (514, 3)
    hits = get_lidar(torch.tensor([0.0, 0.0, 0.0]), sph, tab, 16)
    assert hits.shape == (16, 3)
    # closest return is the +z pole ray: hit at z = 0.75
    np.testing.assert_allclose(hits[0].numpy(), [0, 0, 0.75], atol=1e-6)
    assert (hits.norm(dim=-1)[1:] >= hits.norm(dim=-1)[:-1] - 1e-6).all()     # sorted by alpha


def test_zero_obstacles_all_rays_miss():
    hits = get_lidar(torch.tensor([1.0, 1.0]), None, ray_table_2d(32, 0.5), 32)
    assert (hits.abs().max(dim=-1).values > 1e4).all()


@pytest.mark.parametrize("env_id", ENVS)
def test_dense_reference_layout_equals_sparse(env_id):
    N, area, n_obs = 8, 1.6, 4
    agent, goal, obs = random_scene(env_id, N, 1, area, n_obs, seed=4)
    oenv = oracle_env(env_id, N, area, n_obs)
    from helpers import product_obstacles
    pobs = product_obstacles(env_id, obs, device="cpu")
    oobs = oracle_obstacles(pobs.packed.numpy()[0])
    dense = oenv.get_graph(torch.from_numpy(agent[0]), torch.from_numpy(goal[0]), oobs)
    sparse = oenv.sparsify(dense)
    R = oenv.n_hits
    assert dense.edges.shape[0] == (2 * N * N + N * R if env_id != "DubinsCar" else N * N + N + N * R)
    assert dense.nodes.shape[0] == 2 * N + N * R + 1
    ap, cp = oracle_params(env_id)
    with torch.no_grad():
        np.testing.assert_allclose(get_cbf(cp, dense).numpy(), get_cbf(cp, sparse).numpy(), atol=2e-6)
        a_d, a_s = act(oenv, ap, dense), act(oenv, ap, sparse)
        np.testing.assert_allclose(a_d.numpy(), a_s.numpy(), atol=2e-6)
        fd, fs = oenv.forward_graph(dense, a_d), oenv.forward_graph(sparse, a_d)
        np.testing.assert_allclose(get_cbf(cp, fd).numpy(), get_cbf(cp, fs).numpy(), atol=2e-6)


def test_cbf_sign_flips_at_collision_distance():
    """SURVEY 4 smoke check: two agents head-on, h < 0 inside 2r = 0.1, h > 0 well outside."""
    _, cp = oracle_params("DoubleIntegrator")
    env = OracleEnv("DoubleIntegrator", 2, 4.0, params={"n_obs": 0})
    hs = {}
    for d in (0.05, 0.10, 0.20, 0.60):
        agent = torch.tensor([[1.0, 1.0, 0.3, 0.0], [1.0 + d, 1.0, -0.3, 0.0]])
        goal = torch.tensor([[3.0, 1.0, 0, 0], [0.0, 1.0, 0, 0]])
        with torch.no_grad():
            hs[d] = get_cbf(cp, env.sparsify(env.get_graph(agent, goal, None))).squeeze(-1)
    assert (hs[0.05] < 0).all() and (hs[0.10] < 0).all() and (hs[0.20] > 0).all() and (hs[0.60] > 0).all()


def test_safe_mask_horizon_semantics():
    u = np.zeros((10, 2), dtype=bool)
    u[6, 0] = True
    s = safe_mask_horizon(u, 3)
    assert s[:, 1].all()
    assert s[:, 0].tolist() == [True, True, True, False, False, False, False, True, True, True]
    u[0, 1] = True
    assert safe_mask_horizon(u, 3)[0, 1]            # initial state always safe (gcbf_plus.py:170)


def test_adamw_clip_polyak_restatement():
    torch.manual_seed(0)
    p = {"w": torch.randn(5, 3), "b": torch.randn(3)}
    g = {"w": torch.randn(5, 3) * 10, "b": torch.randn(3) * 10}
    gc, n = compute_norm_and_clip(g, 2.0)
    assert abs(torch.sqrt(sum((v * v).sum() for v in gc.values())).item() - 2.0) < 1e-5
    small = {k: v * 1e-3 for k, v in g.items()}
    gs, _ = compute_norm_and_clip(small, 2.0)
    torch.testing.assert_close(gs["w"], small["w"])                        # below max_norm: unchanged
    opt, ref = AdamW(p, lr=1e-2), torch.optim.AdamW([torch.nn.Parameter(v.clone()) for v in p.values()], lr=1e-2,
                                                   weight_decay=1e-3, eps=1e-8)
    q = dict(p)
    for _ in range(3):
        q = opt.step(q, gc)
        for prm, k in zip(ref.param_groups[0]["params"], p):
            prm.grad = gc[k].clone()
        ref.step()
    # optax adamw decays with lr*wd*p inside the same update (equivalent to torch's decoupled form to O(lr^2 wd))
    for prm, k in zip(ref.param_groups[0]["params"], p):
        torch.testing.assert_close(q[k], prm.data, atol=1e-5, rtol=1e-4)
    bad = {"w": gc["w"].clone(), "b": gc["b"].clone()}
    bad["b"][0] = float("nan")
    t_before = opt.t
    assert opt.step(q, bad) is q and opt.t == t_before                     # apply_if_finite skips
    pk = polyak({"w": torch.ones(2)}, {"w": torch.zeros(2)}, 0.5)
    assert pk["w"].tolist() == [0.5, 0.5]


def test_loss_gradient_routing_float64():
    """update_inner semantics (gcbf_plus.py:399-407): for unlabelled agents the CBF parameters get
    no gradient through h(g') / h_dot, but the actor still does."""
    env_id, N, area = "DoubleIntegrator", 4, 1.2
    agent, goal, obs = random_scene(env_id, N, 2, area, 2, seed=8)
    from helpers import product_obstacles
    pobs = product_obstacles(env_id, obs, device="cpu")
    oenv = oracle_env(env_id, N, area, 2, dtype=torch.float64)
    ap, cp = oracle_params(env_id, dtype=torch.float64)
    cp = {k: v.clone().requires_grad_(True) for k, v in cp.items()}
    ap = {k: v.clone().requires_grad_(True) for k, v in ap.items()}
    graphs = [oenv.sparsify(oenv.get_graph(torch.from_numpy(agent[g]).double(), torch.from_numpy(goal[g]).double(),
                                           oracle_obstacles(pobs.packed.numpy()[g], torch.float64))) for g in range(2)]
    none = torch.zeros(2, N, dtype=torch.bool)
    u_qp = torch.zeros(2, N, 2, dtype=torch.float64)
    kw = dict(coef_action=0.0, coef_unsafe=0.0, coef_safe=0.0, coef_h_dot=1.0, eps=10.0)  # eps large: relu active
    total, _ = gcbf_plus_loss(oenv, cp, ap, graphs, none, none, u_qp, **kw)
    gc = torch.autograd.grad(total, list(cp.values()), retain_graph=True, allow_unused=True)
    ga = torch.autograd.grad(total, list(ap.values()), allow_unused=True)
    assert any(g is not None and g.abs().max() > 0 for g in ga)
    # unlabelled: d/dcbf of relu(-h_dot_ng - alpha h + eps) = -alpha dh/dcbf only
    h_only = sum(-1.0 * get_cbf(cp, g).sum() for g in graphs) / (2 * N)
    gh = torch.autograd.grad(h_only, list(cp.values()), allow_unused=True)
    for a, b in zip(gc, gh):
        if a is not None:
            torch.testing.assert_close(a, b, atol=1e-10, rtol=1e-8)


def test_rollout_and_rates_smoke():
    env_id, N, area = "DoubleIntegrator", 4, 2.0
    agent, goal, obs = random_scene(env_id, N, 1, area, 2, seed=3, vel_scale=0.0)
    from helpers import product_obstacles
    pobs = product_obstacles(env_id, obs, device="cpu")
    oenv = oracle_env(env_id, N, area, 2)
    ap, _ = oracle_params(env_id)
    out = rollout(oenv, ap, torch.from_numpy(agent[0]), torch.from_numpy(goal[0]),
                  oracle_obstacles(pobs.packed.numpy()[0]), T=8)
    assert out["states"].shape == (9, N, 4) and out["actions"].shape == (8, N, 2)
    s, f, ok = rates(out["collision"].numpy(), out["finish"].numpy())
    assert 0.0 <= s <= 1.0 and 0.0 <= f <= 1.0 and ok <= min(s, f) + 1e-9


# ------------------------------------------------------------------------------------ QP action labels
def _qp_case(env_id, N, area, seed, dtype=torch.float64):
    from oracle import qp
    agent, goal, obs = random_scene(env_id, N, 1, area, 4, seed)
    oenv = oracle_env(env_id, N, area, 4, dtype=dtype)
    from helpers import product_obstacles
    pobs = product_obstacles(env_id, obs, device="cpu")
    oobs = oracle_obstacles(pobs.packed.numpy()[0], dtype=dtype)
    _, cp = oracle_params(env_id, dtype)
    g = oenv.sparsify(oenv.get_graph(torch.tensor(agent[0], dtype=dtype), torch.tensor(goal[0], dtype=dtype), oobs))
    return oenv, cp, g, qp.qp_data(oenv, cp, g, 1.0)


@pytest.mark.parametrize("env_id,N,area", [("SingleIntegrator", 8, 0.8), ("DoubleIntegrator", 12, 1.2),
                                           ("DubinsCar", 8, 1.0), ("LinearDrone", 8, 0.9)])
def test_qp_dual_solver_matches_active_set_and_kkt(env_id, N, area):
    """The dual solver (the algorithm the CUDA kernel runs) against SciPy's SLSQP on the primal, and against
    the KKT conditions: the QP is strictly convex, so both pin the unique minimiser (oracle/qp.py header)."""
    from oracle import qp
    oenv, cp, g, d = _qp_case(env_id, N, area, seed=11)
    u, r, lam, it = qp.solve_qp_dual(d["Lg_h"], d["b"], d["u_ref"], d["u_lim"])
    assert it < 100000
    kkt = qp.kkt_residual(d["Lg_h"], d["b"], d["u_ref"], d["u_lim"], u, r, lam)
    assert max(kkt.values()) < 1e-6, kkt      # complementarity is lam * slack with lam up to ~1e3
    us, rs, res = qp.solve_qp_slsqp(d["Lg_h"], d["b"], d["u_ref"], d["u_lim"])
    np.testing.assert_allclose(u, us, atol=1e-6)
    np.testing.assert_allclose(r, rs, atol=1e-6)
    assert (lam > 0).sum() >= 1, "scene too easy: no CBF constraint active"
    # the label differs from u_ref exactly where a constraint is active
    assert np.abs(u - np.clip(d["u_ref"], -d["u_lim"], d["u_lim"])).max() > 1e-3


def test_qp_jacobian_is_graph_sparse_and_matches_finite_differences():
    """h is a one-layer GNN: d h_i / d x_j is non-zero only for j = i or an agent neighbour j -> i (the
    structure the CUDA path stores on the edge list); central differences confirm the autograd Jacobian."""
    from oracle import qp
    from oracle.algo import get_cbf
    oenv, cp, g, d = _qp_case("DoubleIntegrator", 10, 1.5, seed=5)
    N = 10
    hx = d["h_x"]
    nbr = np.eye(N, dtype=bool)
    for r_, s_ in zip(g.receivers.numpy(), g.senders.numpy()):
        if s_ < N:
            nbr[r_, s_] = True
    assert np.abs(hx[~nbr]).max() == 0.0
    assert np.abs(hx[nbr]).max() > 1e-3
    rest = g.states[N:]
    x0 = g.states[:N].clone()

    def h_of(x):
        with torch.no_grad():
            return get_cbf(cp, oenv.add_edge_feats(g, torch.cat([x, rest], 0))).squeeze(-1).numpy()
    eps = 1e-6
    for (j, c) in [(0, 0), (3, 2), (7, 1), (9, 3)]:
        xp, xm = x0.clone(), x0.clone()
        xp[j, c] += eps
        xm[j, c] -= eps
        np.testing.assert_allclose((h_of(xp) - h_of(xm)) / (2 * eps), hx[:, j, c], atol=1e-6)


def test_qp_relaxation_engages_when_infeasible():
    """A constraint no admissible u can satisfy is relaxed: lam sits above the 1e3 penalty and r > 0 makes the
    row feasible with equality (gcbf_plus.py:329-339)."""
    from oracle import qp
    Lg = np.array([[1.0, 0.0], [0.0, 0.5]])
    b = np.array([-5.0, 0.3])            # row 0 needs u0 >= 5 with |u| <= 1
    u_ref = np.array([0.2, -0.1])
    u, r, lam, _ = qp.solve_qp_dual(Lg, b, u_ref, 1.0)
    assert u[0] == 1.0 and abs(r[0] - 4.0) < 1e-9 and abs(lam[0] - (1000 + 10 * 4.0)) < 1e-6
    assert r[1] == 0.0 and lam[1] == 0.0 and abs(u[1] + 0.1) < 1e-12
    assert max(qp.kkt_residual(Lg, b, u_ref, 1.0, u, r, lam).values()) < 1e-8


# ------------------------------------------------------------------------------------ reset / jax.random restatement
def test_threefry_known_answers():
    """Random123 Threefry-2x32-20 vectors + the values jax prints for split / uniform of PRNGKey(0) and
    split(PRNGKey(42)) -- checked for both the product's host RNG and the oracle's scalar restatement."""
    from gcbfplus_b200.utils import jrandom as jr
    from oracle import reset as orr
    kat = [((0, 0), (0, 0), (0x6B200159, 0x99BA4EFE)),
           ((0xFFFFFFFF, 0xFFFFFFFF), (0xFFFFFFFF, 0xFFFFFFFF), (0x1CB996FC, 0xBB002BE7)),
           ((0x13198A2E, 0x03707344), (0x243F6A88, 0x85A308D3), (0xC4923A9C, 0x483DF7A0))]
    for key, ctr, exp in kat:
        assert orr.threefry2x32(key[0], key[1], ctr[0], ctr[1]) == exp
        y0, y1 = jr.threefry2x32(key[0], key[1], np.array([ctr[0]], np.uint32), np.array([ctr[1]], np.uint32))
        assert (int(y0[0]), int(y1[0])) == exp
    assert jr.split(jr.PRNGKey(0)).tolist() == [[4146024105, 967050713], [2718843009, 1272950319]]
    assert jr.split(jr.PRNGKey(42)).tolist() == [[2465931498, 3679230171], [255383827, 267815257]]
    assert orr.split(orr.prng_key(0)) == [(4146024105, 967050713), (2718843009, 1272950319)]
    assert abs(float(jr.uniform(jr.PRNGKey(0))) - 0.41845703) < 1e-8
    assert abs(float(orr.uniform(orr.prng_key(0), (), 0.0, 1.0)) - 0.41845703) < 1e-8
    # batched keys == a loop over keys (the reference vmaps reset over keys)
    ks = jr.split(jr.PRNGKey(7), 5)
    assert (jr.split(ks, 3) == np.stack([jr.split(k, 3) for k in ks])).all()
    assert (jr.uniform(ks, (3,), -1, 2) == np.stack([jr.uniform(k, (3,), -1, 2) for k in ks])).all()
    for k in ks:
        kk = (int(k[0]), int(k[1]))
        assert [tuple(map(int, r)) for r in jr.split(k, 3)] == orr.split(kk, 3)
        assert (jr.uniform(k, (5,), 0, 3) == orr.uniform(kk, (5,), 0, 3)).all()


def _jax_normal(jr_uniform, key):
    """jax.random.normal(key): sqrt(2) * erf_inv(uniform(key, minval=nextafter(-1, 0), maxval=1)) (jax/_src/random.py)."""
    from scipy.special import erfinv
    lo = np.nextafter(np.float32(-1), np.float32(0), dtype=np.float32)
    u = jr_uniform(key, lo, 1.0)
    return float(np.float32(np.sqrt(2)) * np.float32(erfinv(np.float64(u))))


@pytest.mark.parametrize("partitionable", [False, True])
def test_threefry_stream_layouts_against_values_jax_publishes(partitionable):
    """Both threefry stream layouts (`jax_threefry_partitionable` off = default of JAX 0.4.x, on = default from
    JAX 0.5.0) against numbers JAX's own documentation prints -- the `Pseudorandom numbers` tutorial's
    `key = random.key(42)`, `random.normal(key)` and its three split-and-draw iterations, and `random.uniform(key(0))`
    of the jax.random docs -- for the product's host RNG and the oracle's scalar restatement.  (Values quoted from the
    public docs of the respective JAX generations; there is no network here to re-fetch them, and an independent
    implementation reproducing them to 7 digits is what makes them known answers.)"""
    from gcbfplus_b200.utils import jrandom as jr
    from oracle import reset as orr
    want = {False: dict(normal42=-0.18471177, uniform0=0.41845703,
                        draws=(1.369469404220581, -0.19947023689746857, -2.298278331756592)),
            True: dict(normal42=-0.028304616, uniform0=0.947667,
                       draws=(0.6057640314102173, -0.21089035272598267, -0.3948981463909149))}[partitionable]
    old_h, old_o = jr.set_partitionable(partitionable), orr.PARTITIONABLE
    orr.PARTITIONABLE = partitionable
    try:
        impls = {
            "host": (lambda seed: jr.PRNGKey(seed), lambda k: [r for r in jr.split(k)],
                     lambda k, lo, hi: jr.uniform(k, (), lo, hi)),
            "oracle": (lambda seed: orr.prng_key(seed), lambda k: orr.split(k),
                       lambda k, lo, hi: orr.uniform(k, (), lo, hi)),
        }
        for name, (mk, split, uni) in impls.items():
            assert abs(float(uni(mk(0), 0.0, 1.0)) - want["uniform0"]) < 6e-7, name
            assert abs(_jax_normal(uni, mk(42)) - want["normal42"]) < 2e-7, name
            key = mk(42)
            for i in range(3):
                key, sub = split(key)
                assert abs(_jax_normal(uni, sub) - want["draws"][i]) < 1e-6 * max(1.0, abs(want["draws"][i])), (name, i)
        # host (vectorised over keys) == oracle (scalar) in this layout, shaped draws included
        ks = jr.split(jr.PRNGKey(7), 5)
        assert (jr.split(ks, 3) == np.stack([jr.split(k, 3) for k in ks])).all()
        for k in ks:
            kk = (int(k[0]), int(k[1]))
            assert [tuple(map(int, r)) for r in jr.split(k, 3)] == orr.split(kk, 3)
            assert (jr.uniform(k, (5,), 0, 3) == orr.uniform(kk, (5,), 0, 3)).all()
            assert (jr.uniform(k, (4, 2), 0, 3).ravel() == orr.uniform(kk, (8,), 0, 3)).all()
    finally:
        jr.set_partitionable(old_h)
        orr.PARTITIONABLE = old_o


@pytest.mark.parametrize("env_id,N,area,n_obs,max_travel", [
    ("SingleIntegrator", 6, 1.5, 3, None), ("DoubleIntegrator", 8, 2.0, 8, None), ("DoubleIntegrator", 5, 3.0, 4, 1.0),
    ("DubinsCar", 6, 2.0, 4, None), ("LinearDrone", 6, 1.0, 4, None)])
@pytest.mark.parametrize("partitionable", [False, True])
def test_reset_matches_oracle_bit_exact(env_id, N, area, n_obs, max_travel, partitionable, monkeypatch):
    """The product's vectorised host reset against the oracle's scalar, per-environment restatement of
    get_node_goal_rng (crowded scenes: rejection loops and per-env divergence are exercised), in both threefry
    stream layouts."""
    from gcbfplus_b200.env import make_env
    from gcbfplus_b200.utils import jrandom as jr
    from oracle import reset as orr
    monkeypatch.setattr(jr, "PARTITIONABLE", partitionable)
    monkeypatch.setattr(orr, "PARTITIONABLE", partitionable)
    env = make_env(env_id, N, area_size=area, num_obs=n_obs, max_travel=max_travel, device="cpu")
    keys = jr.split(jr.PRNGKey(3), 4)
    obstacles, k2 = env._sample_obstacles(keys)
    packed = obstacles.packed.numpy()
    sd, pd = env.state_dim, env.pos_dim
    agent = np.zeros((4, N, sd), np.float32)
    goal = np.zeros((4, N, sd), np.float32)
    agent[:, :, :pd], goal[:, :, :pd] = env._sample_agents_goals(k2, packed)
    env._reset_extra(k2, agent, goal)
    retried = 0
    for e in range(4):
        o = orr.reset(env_id, (int(keys[e, 0]), int(keys[e, 1])), N, area, n_obs, env._params["obs_len_range"],
                      env.radius, max_travel)
        assert np.array_equal(agent[e], o["agent"]) and np.array_equal(goal[e], o["goal"])
        assert np.array_equal(packed[e][:, :pd], o["obs"]["center"])
        if pd == 3:
            assert np.array_equal(packed[e][:, 3], o["obs"]["radius"])
        else:
            assert np.array_equal(packed[e][:, 2], o["obs"]["width"] / np.float32(2))
            assert np.array_equal(packed[e][:, 4], o["obs"]["cos"])
        # validity: pairwise distances and obstacle clearance of the accepted samples
        d = np.linalg.norm(agent[e][:, None, :pd] - agent[e][None, :, :pd], axis=-1) + np.eye(N) * 10
        assert d.min() > 4 * env.radius
        assert not any(orr.inside_obstacles(agent[e][i, :pd], o["obs"], 4 * env.radius) for i in range(N))
        first = orr.uniform(orr.split(orr.split((int(k2[e, 0]), int(k2[e, 1])), 3)[0], 2)[0], (pd,), 0, area)
        retried += int(not np.array_equal(first, agent[e][0, :pd]))
    assert agent.dtype == np.float32
    assert retried >= 0


def test_reset_key_plumbing_matches_reference_call_sites():
    """trainer.py:99-100,134-136 and test.py:117-119,158: which key reaches env.reset for environment i."""
    from gcbfplus_b200.utils import jrandom as jr
    seed, n_env = 5, 3
    key = jr.PRNGKey(seed)
    key_x0, key = jr.split(key)
    rollout_keys = jr.split(key_x0, n_env)                 # vmapped rollout(key): key_x0, _ = split(key); reset(key_x0)
    reset_keys = jr.split(rollout_keys, 2)[:, 0]
    for i in range(n_env):
        assert (reset_keys[i] == jr.split(rollout_keys[i])[0]).all()
    test_keys = jr.split(jr.PRNGKey(seed), 1_000)[:n_env]
    assert test_keys.shape == (n_env, 2) and len({tuple(k) for k in test_keys.tolist()}) == n_env
