""" The kernels for five / six derivative directions (step_kernel<5,5>, step_kernel<6,6>: full Hessians in three
dimensions, Laplacians / heat equations in four to six) and for derivatives of order 3 / 4 (hi_step_kernel<NF, K>: KdV,
beam, Kuramoto-Sivashinsky) on the GPU, to the bar of test_gpu_parity.py: goldens written by the unmodified reference,
the reference's own fit trajectories, the fp64 oracle on random problems through the bare C ABI, ragged batches,
in-kernel sampling, additivity at size.  (Sorted last on purpose: these kernels joined the library after its other
kernels had been measured.) """
import numpy as np
import pytest
import torch

import problems as P
from helpers import load_golden, oracle_problem, rel_l2
from test_emul_fuzz import _random_many_direction_problem, _random_high_order_problem, _layer_plan

# a hang in a kernel that has not met a GPU yet must end as a failure of that test, not stall the whole tier
pytestmark = [pytest.mark.gpu, pytest.mark.timeout(600)]

if torch.cuda.is_available():
    from gpu_helpers import make_solver, Replay, abi_step
    from oracle import autograd_port as ap
    from pydens_b200 import _native as N, tracer as T


@pytest.mark.parametrize('name', list(P.HI_DIRECTION))
def test_step_matches_reference_golden(name):
    g = load_golden(name)
    solver = make_solver(name, g['params'])
    eng = solver._get_engine()
    assert eng.n_params == g['params'].size
    assert eng.info.nf in (5, 6) and eng.info.ns == eng.info.nf and not eng.info.tensor_core
    loss, grads, residual = solver.loss_and_grads(g['points'])
    grads = grads.cpu().numpy()
    assert abs(loss - float(g['loss'])) <= 1e-5 * abs(float(g['loss']))
    assert rel_l2(residual.cpu().numpy(), g['residual']) <= 1e-5
    assert rel_l2(grads, g['grads']) <= 1e-4
    spec = eng.spec
    for l in range(spec.n_layers):
        w = slice(spec.w_off[l], spec.w_off[l] + spec.widths[l] * spec.widths[l + 1])
        b = slice(spec.b_off[l], spec.b_off[l] + spec.widths[l + 1])
        assert rel_l2(grads[w], g['grads'][w]) <= 1e-4, 'W%d' % l
        assert rel_l2(grads[b], g['grads'][b]) <= 1e-4, 'b%d' % l
    u = solver.predict(*[g['points'][:, i] for i in range(g['points'].shape[1])]).reshape(-1)
    assert rel_l2(u, g['u']) <= 1e-5


@pytest.mark.parametrize('adam', ['kernel', 'torch'])
@pytest.mark.parametrize('name', [n for n in P.GOLDEN_TRAJ if n in P.HI_DIRECTION])
def test_fit_trajectory_matches_reference_fit(name, adam, monkeypatch):
    monkeypatch.setenv('PYDENS_B200_FUSED_ADAM', '1' if adam == 'kernel' else '0')
    g = load_golden(name)
    niters, batch, lr = int(g['traj_meta'][0]), int(g['traj_meta'][1]), float(g['traj_meta'][2])
    solver = make_solver(name, g['params'])
    batches = [P.make_points(name, batch, seed=1000 + i) for i in range(niters)]
    solver.fit(niters=niters, batch_size=batch, sampler=Replay(batches), lr=lr)
    losses = np.asarray(solver.losses, dtype=np.float64)
    ref = g['traj_losses'].astype(np.float64)
    assert losses.shape == ref.shape
    assert np.max(np.abs(losses - ref) / np.maximum(np.abs(ref), 1e-6)) <= 2e-3
    assert abs(losses[-1] - ref[-1]) <= 1e-5 * max(1.0, abs(ref[-1]))
    final = solver.flat_params().cpu().numpy()
    assert np.linalg.norm(final - g['traj_params']) / np.linalg.norm(g['traj_params']) <= 1e-3


@pytest.mark.parametrize('n', [1, 31, 33, 1000, 4097])
def test_ragged_batches_against_oracle(n):
    g = load_golden('hess3d')
    solver = make_solver('hess3d', g['params'])
    prob = oracle_problem('hess3d', torch.float32, g['params'])
    pts = P.make_points('hess3d', n, seed=77)
    loss, grads, residual = solver.loss_and_grads(pts)
    l, _, gr = prob.loss_and_grads(pts)
    assert abs(loss - l) <= 1e-5 * abs(l)
    # the residual against fp64: the fp32 oracle's nested autograd is itself 3.6e-5 (rel-L2) off fp64 at n=4097,
    # one point carrying an error of 2.3e-4
    _, r64, _ = oracle_problem('hess3d', torch.float64, g['params'].astype(np.float64)).loss_and_grads(pts.astype(np.float64))
    assert rel_l2(residual.cpu().numpy(), r64) <= 1e-5
    assert rel_l2(grads.cpu().numpy(), gr.numpy()) <= 1e-4


def test_in_kernel_sampling_equals_explicit_points_and_runs_are_deterministic():
    """ Six point columns: the second Philox block serves columns 4 and 5. """
    g = load_golden('lap6d')
    solver = make_solver('lap6d', g['params'])
    eng = solver._get_engine()
    n = 20000
    eng._step(None, None, n, 1.0 / n, 0, use_counter=False, step_value=9)
    torch.cuda.synchronize()
    sampled = eng.out.clone()
    pts = eng.sample(n, None, step=9)
    assert pts.shape == (n, 6) and float(pts.min()) >= 0.0 and float(pts.max()) < 1.0
    for _ in range(2):
        eng._step(pts, None, n, 1.0 / n, 0, use_counter=False, step_value=9)
        torch.cuda.synchronize()
        assert torch.equal(sampled, eng.out)
    prob = oracle_problem('lap6d', torch.float32, g['params'])
    l, _, gr = prob.loss_and_grads(pts.cpu().numpy())
    assert abs(float(sampled[eng.n_params]) - l) <= 1e-5 * abs(l)
    assert rel_l2(sampled[:eng.n_params].cpu().numpy(), gr.numpy()) <= 1e-4


@pytest.mark.parametrize('name,n', [('heat4d', 200000), ('hess3d', 200000)])
def test_additivity_at_size(name, n):
    g = load_golden(name)
    solver = make_solver(name, g['params'])
    eng = solver._get_engine()
    pts = torch.from_numpy(P.make_points(name, n, seed=11)).cuda()
    h = n // 2 + 13
    eng._step(pts, None, n, 1.0 / n, 0, use_counter=False)
    whole = eng.out.clone()
    eng._step(pts[:h].contiguous(), None, h, 1.0 / n, 0, use_counter=False)
    a = eng.out.clone()
    eng._step(pts[h:].contiguous(), None, n - h, 1.0 / n, 0, use_counter=False)
    b = eng.out.clone()
    torch.cuda.synchronize()
    assert torch.isfinite(whole).all()
    np_ = eng.n_params
    assert abs(float(whole[np_] - (a + b)[np_])) <= 1e-5 * abs(float(whole[np_]))
    assert rel_l2((a + b)[:np_].cpu().numpy(), whole[:np_].cpu().numpy()) <= 1e-4


@pytest.mark.parametrize('seed', list(range(24)))
def test_random_many_direction_problem_on_gpu_matches_fp64_oracle(seed):
    cfg = _random_many_direction_problem(seed)
    sym_V = lambda n, init: T.Sym(T.var(n))
    nsp = cfg['ndims'] - 1 if cfg['ic'] is not None else cfg['ndims']
    traced = T.trace(lambda u, *xs: cfg['eq'](u, *xs, D=T.sym_D, V=sym_V), cfg['total'], None,
                     initial_condition=cfg['ic'], ndims_spatial=nsp)
    acts, skips = _layer_plan(cfg)
    spec = N.build_spec([cfg['total']] + cfg['features'], acts, cfg['ndims'], 0, cfg['bc'] is not None,
                        cfg['bc'] if cfg['bc'] is not None else 0.0, cfg['ic'] is not None, cfg['domain'], traced,
                        skips=skips)
    prob = ap.Problem(cfg['eq'], ndims=cfg['ndims'], nparams=0, initial_condition=cfg['ic'],
                      boundary_condition=cfg['bc'], domain=cfg['domain'], features=cfg['features'],
                      activation=cfg['acts'], dtype=torch.float64, variables=cfg['variables'], seed=seed,
                      layout=cfg['layout'])
    with torch.no_grad():
        prob.log_scale.fill_(cfg['log_scale'])
    params = prob.flat_params().numpy().astype(np.float32)
    rng = np.random.RandomState(3000 + seed)
    n = int(rng.choice([1, 31, 257, 3000]))
    pts = np.concatenate([rng.uniform(lo, hi, size=(n, 1)) for lo, hi in cfg['ranges']], axis=1).astype(np.float32)
    loss, residual, grads, u = abi_step(spec, params, pts)
    prob.load_flat(torch.from_numpy(params.astype(np.float64)))
    ref_loss, ref_res, ref_grads = prob.loss_and_grads(pts.astype(np.float64))
    tag = '%s %s %s acts=%s n=%d' % (cfg['eq_name'], cfg['layout'], cfg['features'], acts, n)
    cond = max(1.0, 0.05 / max(float(np.sqrt(np.mean(np.square(ref_res)))), 1e-30))
    assert abs(loss - ref_loss) <= 2e-5 * cond * max(abs(ref_loss), 1e-6), tag
    assert rel_l2(residual, ref_res) <= 2e-5 * cond, tag
    assert rel_l2(grads, ref_grads.numpy()) <= 1e-4 * cond, tag
    ref_u = prob.predict(pts.astype(np.float64))
    assert np.abs(u - ref_u).max() <= 1e-5 * max(1.0, np.abs(ref_u).max()), tag


def test_seven_directions_fall_back_loudly():
    """ More directions than the kernels carry: backend='auto' trains on autograd with a warning, 'fused' raises. """
    from pydens_b200 import Solver, D

    def eq(f, x, y, z, t):
        return D(D(f, x), y) + D(D(f, y), z) + D(D(f, x), z) - D(f, t)
    solver = Solver(eq, ndims=4, layout='fafaf', features=[6, 5, 1], activation='Tanh')
    with pytest.warns(UserWarning):
        solver.fit(niters=2, batch_size=32)
    assert len(solver.losses) == 2 and solver._engine is None
    with pytest.raises(RuntimeError):
        Solver(eq, ndims=4, layout='fafaf', features=[6, 5, 1], activation='Tanh', backend='fused')


# ---------------------------------------------------------------------------------------------------------------
# derivatives of order 3 / 4: hi_step_kernel<NF, K> (pinn_hi_kernel.cuh)
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('name', list(P.HI_ORDER))
def test_high_order_step_matches_reference_golden_and_fp64(name):
    """ Against the golden written by the unmodified reference — with the reference's own fp32 error as slack: nested
    autograd of order 3 / 4 in fp32 loses digits (beam: residual 1.1e-4 off fp64) — and, as the arbiter, against the
    fp64 oracle at the stated fp32 tolerances. """
    g = load_golden(name)
    solver = make_solver(name, g['params'])
    eng = solver._get_engine()
    assert eng.n_params == g['params'].size and eng.spec.order in (3, 4)
    assert eng.info.channels == 1 + eng.info.nf * eng.spec.order and not eng.info.tensor_core
    loss, grads, residual = solver.loss_and_grads(g['points'])
    grads, residual = grads.cpu().numpy(), residual.cpu().numpy()
    prob = oracle_problem(name, torch.float64, g['params'].astype(np.float64))
    l64, r64, g64 = prob.loss_and_grads(g['points'].astype(np.float64))
    g64 = g64.numpy()
    assert abs(loss - l64) <= 1e-5 * abs(l64)
    assert rel_l2(residual, r64) <= 1e-5 and rel_l2(grads, g64) <= 1e-4
    slack_r, slack_g = rel_l2(g['residual'], r64), rel_l2(g['grads'], g64)
    assert abs(loss - float(g['loss'])) <= (1e-5 + 2.0 * slack_r) * abs(float(g['loss']))
    assert rel_l2(residual, g['residual']) <= 1e-5 + 1.5 * slack_r
    assert rel_l2(grads, g['grads']) <= 1e-4 + 1.5 * slack_g
    spec = eng.spec
    for l in range(spec.n_layers):
        w = slice(spec.w_off[l], spec.w_off[l] + spec.widths[l] * spec.widths[l + 1])
        b = slice(spec.b_off[l], spec.b_off[l] + spec.widths[l + 1])
        assert rel_l2(grads[w], g64[w]) <= 1e-4, 'W%d' % l
        assert rel_l2(grads[b], g64[b]) <= 1e-4, 'b%d' % l
    u = solver.predict(*[g['points'][:, i] for i in range(g['points'].shape[1])]).reshape(-1)
    assert rel_l2(u, g['u']) <= 1e-5


@pytest.mark.parametrize('adam', ['kernel', 'torch'])
@pytest.mark.parametrize('name', [n for n in P.GOLDEN_TRAJ if n in P.HI_ORDER])
def test_high_order_fit_trajectory_matches_reference_fit(name, adam, monkeypatch):
    monkeypatch.setenv('PYDENS_B200_FUSED_ADAM', '1' if adam == 'kernel' else '0')
    g = load_golden(name)
    niters, batch, lr = int(g['traj_meta'][0]), int(g['traj_meta'][1]), float(g['traj_meta'][2])
    solver = make_solver(name, g['params'])
    batches = [P.make_points(name, batch, seed=1000 + i) for i in range(niters)]
    solver.fit(niters=niters, batch_size=batch, sampler=Replay(batches), lr=lr)
    losses = np.asarray(solver.losses, dtype=np.float64)
    ref = g['traj_losses'].astype(np.float64)
    assert losses.shape == ref.shape
    assert np.max(np.abs(losses - ref) / np.maximum(np.abs(ref), 1e-6)) <= 2e-3
    assert abs(losses[-1] - ref[-1]) <= 1e-5 * max(1.0, abs(ref[-1]))
    final = solver.flat_params().cpu().numpy()
    assert np.linalg.norm(final - g['traj_params']) / np.linalg.norm(g['traj_params']) <= 1e-3


@pytest.mark.parametrize('n', [1, 31, 33, 1000, 4097])
def test_high_order_ragged_batches_against_oracle(n):
    g = load_golden('kdv')
    solver = make_solver('kdv', g['params'])
    prob = oracle_problem('kdv', torch.float64, g['params'].astype(np.float64))
    pts = P.make_points('kdv', n, seed=77)
    loss, grads, residual = solver.loss_and_grads(pts)
    l, r, gr = prob.loss_and_grads(pts.astype(np.float64))
    assert abs(loss - l) <= 1e-5 * abs(l)
    assert rel_l2(residual.cpu().numpy(), r) <= 1e-5
    assert rel_l2(grads.cpu().numpy(), gr.numpy()) <= 1e-4


def test_high_order_sampling_determinism_and_additivity():
    g = load_golden('plate')
    solver = make_solver('plate', g['params'])
    eng = solver._get_engine()
    n = 100000
    eng._step(None, None, n, 1.0 / n, 0, use_counter=False, step_value=5)
    torch.cuda.synchronize()
    sampled = eng.out.clone()
    pts = eng.sample(n, None, step=5)
    for _ in range(2):
        eng._step(pts, None, n, 1.0 / n, 0, use_counter=False, step_value=5)
        torch.cuda.synchronize()
        assert torch.equal(sampled, eng.out)
    h = n // 2 + 13
    eng._step(pts[:h].contiguous(), None, h, 1.0 / n, 0, use_counter=False)
    a = eng.out.clone()
    eng._step(pts[h:].contiguous(), None, n - h, 1.0 / n, 0, use_counter=False)
    b = eng.out.clone()
    torch.cuda.synchronize()
    np_ = eng.n_params
    assert torch.isfinite(sampled).all()
    assert abs(float(sampled[np_] - (a + b)[np_])) <= 1e-5 * abs(float(sampled[np_]))
    assert rel_l2((a + b)[:np_].cpu().numpy(), sampled[:np_].cpu().numpy()) <= 1e-4


@pytest.mark.parametrize('seed', list(range(30)))
def test_random_high_order_problem_on_gpu_matches_fp64_oracle(seed):
    cfg = _random_high_order_problem(seed)
    sym_V = lambda n, init: T.Sym(T.var(n))
    nsp = cfg['ndims'] - 1 if cfg['ic'] is not None else cfg['ndims']
    traced = T.trace(lambda u, *xs: cfg['eq'](u, *xs, D=T.sym_D, V=sym_V), cfg['total'], None,
                     initial_condition=cfg['ic'], ndims_spatial=nsp)
    acts, skips = _layer_plan(cfg)
    spec = N.build_spec([cfg['total']] + cfg['features'], acts, cfg['ndims'], cfg['nparams'], cfg['bc'] is not None,
                        cfg['bc'] if cfg['bc'] is not None else 0.0, cfg['ic'] is not None, cfg['domain'], traced,
                        skips=skips)
    prob = ap.Problem(cfg['eq'], ndims=cfg['ndims'], nparams=cfg['nparams'], initial_condition=cfg['ic'],
                      boundary_condition=cfg['bc'], domain=cfg['domain'], features=cfg['features'],
                      activation=cfg['acts'] or 'Tanh', dtype=torch.float64, variables=cfg['variables'], seed=seed,
                      layout=cfg['layout'])
    with torch.no_grad():
        prob.log_scale.fill_(cfg['log_scale'])
    params = prob.flat_params().numpy().astype(np.float32)
    rng = np.random.RandomState(5000 + seed)
    n = int(rng.choice([1, 31, 257, 3000]))
    pts = np.concatenate([rng.uniform(lo, hi, size=(n, 1)) for lo, hi in cfg['ranges']], axis=1).astype(np.float32)
    loss, residual, grads, u = abi_step(spec, params, pts)
    prob.load_flat(torch.from_numpy(params.astype(np.float64)))
    ref_loss, ref_res, ref_grads = prob.loss_and_grads(pts.astype(np.float64))
    tag = '%s %s %s acts=%s n=%d' % (cfg['eq_name'], cfg['layout'], cfg['features'], acts, n)
    cond = max(1.0, 0.05 / max(float(np.sqrt(np.mean(np.square(ref_res)))), 1e-30))
    if cfg['eq_name'] in ('biharmonic', 'mixed3'):
        cond *= 5.0          # mixed derivatives by polarisation: (P_4 + M_4 - 2 u_xxxx - 2 u_yyyy) / 12 cancels leading digits
    assert abs(loss - ref_loss) <= 2e-5 * cond * max(abs(ref_loss), 1e-6), tag
    assert rel_l2(residual, ref_res) <= 2e-5 * cond, tag
    assert rel_l2(grads, ref_grads.numpy()) <= 1e-4 * cond, tag
    ref_u = prob.predict(pts.astype(np.float64))
    assert np.abs(u - ref_u).max() <= 1e-5 * max(1.0, np.abs(ref_u).max()), tag


def test_kdv_through_the_public_api_follows_the_fp64_oracle():
    """ The user-level call with D nested three times: the fused fit (host batches; then in-kernel sampling with graph
    replay and Adam in the kernel's tail) against the oracle port of the reference loop in fp64 on identical initial
    weights and batches.  (fp64 because fp32 nested autograd of order 3 is a noisy yardstick: on the CPU its loss is off by
    1 % at single steps of this very fit, while this path's host build follows fp64 to 1.5e-6.) """
    from pydens_b200 import Solver, D

    def kdv(f, x, t):
        return D(f, t) + 6.0 * f * D(f, x) + D(D(D(f, x), x), x)
    torch.manual_seed(0)
    fused = Solver(kdv, ndims=2, initial_condition=lambda x: torch.sin(np.pi * x), boundary_condition=0.0,
                   layout='fafaf', features=[16, 16, 1], activation='Tanh', backend='fused')
    start = fused.flat_params().cpu().numpy()
    rng = np.random.RandomState(3)
    batches = [rng.uniform(size=(256, 2)).astype(np.float32) for _ in range(25)]
    prob = ap.Problem(lambda u, x, t, D, V: D(u, t) + 6.0 * u * D(u, x) + D(D(D(u, x), x), x), ndims=2,
                      initial_condition=lambda x: torch.sin(np.pi * x), boundary_condition=0.0, domain=(0, 1),
                      features=[16, 16, 1], activation='Tanh', dtype=torch.float64)
    prob.load_flat(torch.from_numpy(start.astype(np.float64)))
    ref = ap.fit(prob, 25, 256, lr=0.005, point_stream=lambda i: torch.from_numpy(batches[i].astype(np.float64)))
    fused.fit(niters=25, batch_size=256, sampler=Replay(batches), lr=0.005)
    assert fused._engine is not None and fused._engine.spec.order == 3
    a = np.asarray(fused.losses, dtype=np.float64)
    assert a.shape == ref.shape == (25,)
    assert np.max(np.abs(a - ref) / np.maximum(np.abs(ref), 1e-6)) <= 2e-3
    final, want = fused.flat_params().cpu().numpy(), prob.flat_params().numpy()
    assert np.linalg.norm(final - want) / np.linalg.norm(want) <= 1e-3
    xs = np.linspace(0, 1, 7)
    pts = np.stack([xs, np.full(7, 0.3)], axis=1)
    assert np.abs(fused.predict(xs, 0.3).reshape(-1) - prob.predict(pts)).max() <= 1e-4
    fused.fit(niters=64, batch_size=4000, lr=0.005)                  # in-kernel sampling, graph replay
    assert len(fused.losses) == 89 and np.isfinite(np.asarray(fused.losses, dtype=np.float64)).all()
