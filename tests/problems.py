""" Problem registry shared by oracle/make_golden.py, the oracle tests and the GPU parity tests.

Equations are written once, token-agnostic: `eq(u, *xs, D=..., V=...)`; the harness binds D/V of
whichever implementation is under test (reference, oracle port, pydens_b200).  `V(name, init)`.

BASELINE.json configs: cfg1/cfg2 = poisson2d, cfg3 = ode_param, cfg4 = heat2d, cfg5 = wave3d.
The others cover the tutorial's remaining problems and the corner cases of the ansatz / programs.
"""
import math

import numpy as np
import torch

PI = math.pi


class Sin(torch.nn.Module):                          # the reference takes activation callables (model_torch.py:150-151)
    def forward(self, x):
        return torch.sin(x)


def _poisson2d(f, x, y, D, V):                       # README.md:36-37
    return D(D(f, x), x) + D(D(f, y), y) - 5 * torch.sin(np.pi * (x + y))


def _ode_param(f, x, e, D, V):                       # README.md:78-79
    return D(f, x) - e * np.pi * torch.cos(e * np.pi * x)


def _heat2d(f, x, y, t, D, V):                       # tutorial heat eq. without the parameter
    return D(D(f, x), x) + D(D(f, y), y) - D(f, t)


# --- more than four derivative directions (kernels with NF = NS = 5 / 6; the tracer promotes every direction) ---
def _hess3d(f, x, y, z, D, V):                       # anisotropic diffusion with cross terms: 3 axes + 3 diagonals
    return (D(D(f, x), x) + 2.0 * D(D(f, y), y) + 3.0 * D(D(f, z), z) + 0.5 * D(D(f, x), y) - 0.3 * D(D(f, y), z)
            + 0.7 * D(D(f, x), z) - torch.sin(x + y + z) * f)


def _heat4d(f, x, y, z, w, t, D, V):                 # heat equation in four space dimensions: 4 second-order + t
    return D(f, t) - 0.1 * (D(D(f, x), x) + D(D(f, y), y) + D(D(f, z), z) + D(D(f, w), w)) + 0.2 * f


def _lap6d(f, a, b, c, d, e, g, D, V):               # Poisson in six dimensions (the DGM paper's regime)
    return (D(D(f, a), a) + D(D(f, b), b) + D(D(f, c), c) + D(D(f, d), d) + D(D(f, e), e) + D(D(f, g), g)
            - torch.cos(a + b - c) * (d + e * g))


def _hess3d_var(f, x, y, z, D, V):                   # 3 axes + 2 diagonals, a first-order term and a variable
    return (D(D(f, x), x) + D(D(f, y), y) * V('kappa', 0.6) + D(D(f, z), z) + D(D(f, x), y) - 0.4 * D(D(f, y), z)
            + f * D(f, z) - V('kappa', 0.6) ** 2)


# --- derivatives of order 3 / 4 (D nested three / four times; kernels hi_step_kernel<NF, K>) ---
def _kdv(f, x, t, D, V):                             # Korteweg-de Vries
    return D(f, t) + 6.0 * f * D(f, x) + D(D(D(f, x), x), x)


def _beam(f, x, t, D, V):                            # Euler-Bernoulli beam with a trainable load
    return D(D(f, t), t) + 0.5 * D(D(D(D(f, x), x), x), x) - torch.sin(PI * x) * V('load', 0.7)


def _ks(f, x, t, D, V):                              # Kuramoto-Sivashinsky
    return D(f, t) + f * D(f, x) + D(D(f, x), x) + D(D(D(D(f, x), x), x), x)


def _ode3(f, x, D, V):                               # third-order ODE
    return D(D(D(f, x), x), x) + D(f, x) * f - torch.cos(x)


def _plate(f, x, y, t, D, V):                        # three directions at order 4 (no mixed term)
    return D(D(f, t), t) + 0.1 * (D(D(D(D(f, x), x), x), x) + D(D(D(D(f, y), y), y), y)) + D(D(D(f, x), x), x) * f


def _biharmonic(f, x, y, D, V):                      # clamped plate: the biharmonic operator in two dimensions
    def lap(g):
        return D(D(g, x), x) + D(D(g, y), y)
    return lap(lap(f)) - 8.0 * torch.sin(PI * x) * torch.sin(PI * y)


def _kdv_icvar(f, x, t, D, V):                       # order 3 with variables in the equation AND in the initial condition
    return D(f, t) + V('speed', 1.5) * f * D(f, x) + 0.2 * D(D(D(f, x), x), x)


def _icf_kdv(V):
    return lambda x: V('amp', 0.7) * torch.sin(2.0 * x) + V('shift', 0.2) ** 2 * x


def _ic_kdv(x):
    return torch.sin(2.0 * x) + 0.3


def _ic_beam(x):
    return x * (1.0 - x)


def _ic_plate(x, y):
    return torch.sin(PI * x) * torch.sin(PI * y)


def _ic_heat4d(x, y, z, w):
    return torch.sin(PI * x) * y * (1.0 - y) + 0.5 * z * w


def _heat_param(f, x, y, t, a, D, V):                # tutorial: `- a * D(f, t)`
    return D(D(f, x), x) + D(D(f, y), y) - a * D(f, t)


def _wave3d(f, x, y, z, t, D, V):                    # BASELINE.json cfg5
    return D(D(f, t), t) - (D(D(f, x), x) + D(D(f, y), y) + D(D(f, z), z))


def _ode_var(f, x, D, V):                            # tutorial `odevar`
    return D(f, x) - 2 * np.pi * torch.cos(2 * np.pi * x) + V('new_var', 1.0)


def _ode_tanh(f, x, D, V):                           # tutorial first example
    return D(f, x) - 2 * np.pi * torch.cos(2 * np.pi * x)


def _burgers(f, x, t, D, V):
    return D(f, t) + f * D(f, x) - 0.01 * D(D(f, x), x)


def _nonlinear(f, x, y, D, V):
    fx = D(f, x)
    return (fx * torch.exp(-x) + f ** 2 - torch.sqrt(x + 1.0) + torch.log(x + 2.0) / (y + 1.0)
            + torch.tanh(D(D(f, y), y)) * 0.5 - (2.0 - y) ** 3 + torch.cos(f) / 3.0 + abs(fx) * 0.1)


def _heat1d_icvar(f, x, t, D, V):                    # variables in the equation AND in the initial condition
    return 0.3 * D(D(f, x), x) - D(f, t) + V('src', 0.1) * torch.sin(x)


def _icf_heat1d(V):                                  # README.md:112-118 style: V inside initial_condition
    return lambda x: V('amp', 0.7) * torch.sin(PI * x) + V('shift', 0.2) ** 2


def _mixed2d(f, x, y, D, V):                         # mixed second derivatives (both argument orders)
    return (0.7 * D(D(f, x), y) + D(D(f, x), x) + 2 * D(D(f, y), y) - torch.sin(x * y)
            + 0.1 * f * D(D(f, y), x))


def _mixed_ic(f, x, y, t, D, V):
    return D(f, t) - D(D(f, x), y) + 0.5 * D(f, x)


def _ic_sincos(x, y):
    return torch.sin(x) * torch.cos(2.0 * y)


def _heat1d(f, x, t, D, V):
    return D(D(f, x), x) - D(f, t)


def _wave1d(f, x, t, D, V):
    return D(D(f, t), t) - 0.25 * D(D(f, x), x)


def _ic_sin(x):
    return torch.sin(PI * x)


def _ic_heat(x, y):
    return 10 * x * y * (1 - x) * (1 - y)


def _ic_wave(x, y, z):
    return torch.sin(PI * x) * torch.sin(PI * y) * torch.sin(PI * z)


def _ic_burgers(x):
    return 0.3 * torch.sin(x) + 0.1


PROBLEMS = {
    # name: dict(equation, ndims, nparams, ic, bc, domain, features, activation, variables, ranges, log_scale)
    'poisson2d': dict(equation=_poisson2d, ndims=2, nparams=0, ic=None, bc=1, domain=(0, 1),
                      features=[10, 12, 15, 1], activation='Tanh', layout='fa fa fa f',
                      ranges=[(0, 1), (0, 1)]),
    'ode_param': dict(equation=_ode_param, ndims=1, nparams=1, ic=1.0, bc=None, domain=(0, 1),
                      features=[20, 30, 1], activation='Sigmoid', layout='fafaf',
                      ranges=[(0, 1), (1, 5)]),
    'heat2d': dict(equation=_heat2d, ndims=3, nparams=0, ic=_ic_heat, bc=0, domain=(0, 1),
                   features=[30, 40, 1], activation='Sigmoid', layout='fafaf',
                   ranges=[(0, 1), (0, 1), (0, .5)]),
    'heat_param': dict(equation=_heat_param, ndims=3, nparams=1, ic=_ic_heat, bc=0, domain=(0, 1),
                       features=[30, 40, 1], activation='Sigmoid', layout='fafaf',
                       ranges=[(0, 1), (0, 1), (0, .5), (.1, 4)]),
    'wave3d': dict(equation=_wave3d, ndims=4, nparams=0, ic=_ic_wave, bc=0, domain=(0, 1),
                   features=[64, 64, 64, 64, 1], activation='Tanh', layout='fafafafaf',
                   ranges=[(0, 1)] * 4),
    'ode_var': dict(equation=_ode_var, ndims=1, nparams=0, ic=1, bc=None, domain=(0, 1),
                    features=[20, 30, 1], activation='Sigmoid', layout='fafaf',
                    variables={'new_var': 1.0}, ranges=[(0, 1)]),
    'ode_tanh': dict(equation=_ode_tanh, ndims=1, nparams=0, ic=.5, bc=None, domain=(0, 1),
                     features=[12, 10, 1], activation='Tanh', layout='fafaf', ranges=[(0, 1)]),
    'burgers': dict(equation=_burgers, ndims=2, nparams=0, ic=_ic_burgers, bc=0.5,
                    domain=[(-1, 2), (0, 3)], features=[8, 9, 1], activation='Tanh', layout='fafaf',
                    ranges=[(-1, 2), (0, 3)], log_scale=0.3),
    'heat1d_icvar': dict(equation=_heat1d_icvar, ndims=2, nparams=0, ic=None, ic_factory=_icf_heat1d, bc=0.0,
                         domain=(0, 1), features=[9, 7, 1], activation='Tanh', layout='fafaf',
                         variables={'amp': 0.7, 'shift': 0.2, 'src': 0.1}, ranges=[(0, 1), (0, 1)], log_scale=-0.2),
    # residual layouts (reference docstring model_torch.py:142-156: 'faR fa fa+ f')
    'poisson_skip': dict(equation=_poisson2d, ndims=2, nparams=0, ic=None, bc=1, domain=(0, 1),
                         features=[8, 6, 8, 1], activation='Tanh', layout='faR fa fa+ f', ranges=[(0, 1), (0, 1)]),
    'heat_resnet': dict(equation=_heat1d, ndims=2, nparams=0, ic=_ic_sin, bc=0, domain=(0, 1),
                        features=[7, 7, 7, 1], activation='Sigmoid', layout='fa R fa+ R fa+ f',
                        ranges=[(0, 1), (0, 1)], log_scale=0.1),
    # mixed derivatives: carried by the extra direction e_x + e_y (polarisation)
    'mixed2d': dict(equation=_mixed2d, ndims=2, nparams=0, ic=None, bc=0.3, domain=[(0, 2), (-1, 1)],
                    features=[9, 8, 1], activation='Tanh', layout='fafaf', ranges=[(0, 2), (-1, 1)]),
    'mixed_ic': dict(equation=_mixed_ic, ndims=3, nparams=0, ic=_ic_sincos, bc=0, domain=(0, 1),
                     features=[10, 6, 1], activation='Sigmoid', layout='fafaf',
                     ranges=[(0, 1), (0, 1), (0, 1)], log_scale=0.2),
    'nonlinear': dict(equation=_nonlinear, ndims=2, nparams=0, ic=None, bc=None, domain=(0, 1),
                      features=[7, 5, 1], activation='Sigmoid', layout='fafaf', ranges=[(0, 1), (0, 1)]),
    # activations outside the tanh / sigmoid family (reference docstring :150-151: callables and nn.* names)
    'poisson_sin': dict(equation=_poisson2d, ndims=2, nparams=0, ic=None, bc=1, domain=(0, 1),
                        features=[9, 11, 1], activation=Sin, layout='fafaf', ranges=[(0, 1), (0, 1)]),
    'heat_softplus': dict(equation=_heat2d, ndims=3, nparams=0, ic=_ic_heat, bc=0, domain=(0, 1),
                          features=[10, 9, 1], activation='Softplus', layout='fafaf',
                          ranges=[(0, 1), (0, 1), (0, .5)]),
    'burgers_silu': dict(equation=_burgers, ndims=2, nparams=0, ic=_ic_burgers, bc=0.5,
                         domain=[(-1, 2), (0, 3)], features=[8, 9, 1], activation='SiLU', layout='fafaf',
                         ranges=[(-1, 2), (0, 3)], log_scale=0.3),
    'wave1d_gelu': dict(equation=_wave1d, ndims=2, nparams=0, ic=_ic_sin, bc=0, domain=(0, 1),
                        features=[12, 10, 1], activation='GELU', layout='fafaf', ranges=[(0, 1), (0, 1)]),
    'mixed_acts_skip': dict(equation=_mixed2d, ndims=2, nparams=0, ic=None, bc=0.3, domain=[(0, 2), (-1, 1)],
                            features=[8, 8, 8, 1], activation=[Sin, 'GELU', 'Tanh'], layout='fa R fa fa+ f',
                            ranges=[(0, 2), (-1, 1)]),
    # five / six derivative directions (HI_DIRECTION below)
    'hess3d': dict(equation=_hess3d, ndims=3, nparams=0, ic=None, bc=0.2, domain=[(0, 1), (-1, 1), (0, 2)],
                   features=[12, 10, 1], activation='Tanh', layout='fafaf', ranges=[(0, 1), (-1, 1), (0, 2)]),
    'heat4d': dict(equation=_heat4d, ndims=5, nparams=0, ic=_ic_heat4d, bc=0, domain=(0, 1),
                   features=[11, 9, 1], activation='Sigmoid', layout='fafaf', ranges=[(0, 1)] * 4 + [(0, .5)],
                   log_scale=0.15),
    'lap6d': dict(equation=_lap6d, ndims=6, nparams=0, ic=None, bc=1, domain=(0, 1),
                  features=[10, 8, 1], activation='Tanh', layout='fafaf', ranges=[(0, 1)] * 6),
    'hess3d_var': dict(equation=_hess3d_var, ndims=3, nparams=0, ic=None, bc=-0.1, domain=(0, 1),
                       features=[8, 8, 8, 1], activation=['GELU', 'Tanh', 'Sigmoid'], layout='fa R fa fa+ f',
                       variables={'kappa': 0.6}, ranges=[(0, 1)] * 3),
    # derivatives of order 3 / 4 (HI_ORDER below)
    'kdv': dict(equation=_kdv, ndims=2, nparams=0, ic=_ic_kdv, bc=0.1, domain=[(-1, 2), (0, 1.5)],
                features=[9, 7, 1], activation='Tanh', layout='fafaf', ranges=[(-1, 2), (0, 1.5)], log_scale=0.2),
    'beam': dict(equation=_beam, ndims=2, nparams=0, ic=_ic_beam, bc=0.0, domain=(0, 1),
                 features=[8, 6, 1], activation='Sigmoid', layout='fafaf', variables={'load': 0.7},
                 ranges=[(0, 1), (0, 1)], log_scale=-0.1),
    'ks': dict(equation=_ks, ndims=2, nparams=0, ic=0.4, bc=None, domain=[(0, 3), (0, 1)],
               features=[10, 8, 6, 1], activation=['Tanh', 'Sigmoid', 'Tanh'], layout='fafafaf',
               ranges=[(0, 3), (0, 1)]),
    'ode3': dict(equation=_ode3, ndims=1, nparams=0, ic=None, bc=0.5, domain=[(0, 2)],
                 features=[7, 5, 1], activation='Tanh', layout='fafaf', ranges=[(0, 2)]),
    'plate': dict(equation=_plate, ndims=3, nparams=0, ic=_ic_plate, bc=0, domain=(0, 1),
                  features=[8, 7, 1], activation='Tanh', layout='fafaf', ranges=[(0, 1), (0, 1), (0, .5)],
                  log_scale=0.1),
    'kdv_icvar': dict(equation=_kdv_icvar, ndims=2, nparams=0, ic=None, ic_factory=_icf_kdv, bc=0.0, domain=[(0, 2), (0, 1)],
                      features=[9, 7, 1], activation='Tanh', layout='fafaf',
                      variables={'amp': 0.7, 'shift': 0.2, 'speed': 1.5}, ranges=[(0, 2), (0, 1)], log_scale=0.1),
    'biharmonic': dict(equation=_biharmonic, ndims=2, nparams=0, ic=None, bc=0.0, domain=(0, 1),
                       features=[10, 8, 1], activation=['Tanh', Sin], layout='fafaf', ranges=[(0, 1), (0, 1)]),
    # the z-stored activation family on the whole-jet path (derivatives up to the fifth from the pre-activation)
    'kdv_silu': dict(equation=_kdv, ndims=2, nparams=0, ic=_ic_kdv, bc=0.1, domain=[(-1, 2), (0, 1.5)],
                     features=[9, 7, 1], activation=['SiLU', 'Softplus'], layout='fafaf', ranges=[(-1, 2), (0, 1.5)],
                     log_scale=0.2),
    'ks_gelu': dict(equation=_ks, ndims=2, nparams=0, ic=0.4, bc=None, domain=[(0, 3), (0, 1)],
                    features=[10, 8, 6, 1], activation=['GELU', 'SiLU', 'Softplus'], layout='fafafaf',
                    ranges=[(0, 3), (0, 1)]),
    # residual layouts under derivatives of order 3 / 4: a two-layer block, and two chained one-layer blocks
    'kdv_resnet': dict(equation=_kdv, ndims=2, nparams=0, ic=_ic_kdv, bc=0.1, domain=[(-1, 2), (0, 1.5)],
                       features=[8, 8, 8, 1], activation=['Tanh', 'SiLU', 'Sigmoid'], layout='fa R fa fa+ f',
                       ranges=[(-1, 2), (0, 1.5)], log_scale=0.2),
    'ks_resnet': dict(equation=_ks, ndims=2, nparams=0, ic=0.4, bc=None, domain=[(0, 3), (0, 1)],
                      features=[7, 7, 7, 1], activation=['Tanh', Sin, 'Tanh'], layout='fa R fa+ R fa+ f',
                      ranges=[(0, 3), (0, 1)]),
}

# problems that need the five- / six-direction kernels; the GPU tests of those kernels live in their own file
HI_DIRECTION = ('hess3d', 'heat4d', 'lap6d', 'hess3d_var')
# problems with derivatives of order 3 / 4 (whole-jet kernels); GPU tests in the same file
HI_ORDER = ('kdv', 'beam', 'ks', 'ode3', 'plate', 'biharmonic', 'kdv_icvar', 'kdv_silu', 'ks_gelu', 'kdv_resnet', 'ks_resnet')

GOLDEN_BATCH = {'poisson2d': 100, 'ode_param': 256, 'heat2d': 128, 'heat_param': 96, 'wave3d': 64,
                'ode_var': 77, 'ode_tanh': 33, 'burgers': 130, 'nonlinear': 64, 'heat1d_icvar': 90, 'poisson_skip': 70, 'heat_resnet': 65, 'mixed2d': 80, 'mixed_ic': 75,
                'poisson_sin': 85, 'heat_softplus': 72, 'burgers_silu': 66, 'wave1d_gelu': 91, 'mixed_acts_skip': 60,
                'hess3d': 70, 'heat4d': 66, 'lap6d': 75, 'hess3d_var': 68,
                'kdv': 72, 'beam': 69, 'ks': 65, 'ode3': 40, 'plate': 67, 'biharmonic': 71, 'kdv_icvar': 74,
                'kdv_silu': 73, 'ks_gelu': 62, 'kdv_resnet': 70, 'ks_resnet': 61}

# problems with a short recorded Adam trajectory: name -> (niters, batch, lr)
GOLDEN_TRAJ = {'poisson2d': (40, 100, 0.005), 'ode_param': (25, 128, 0.01), 'heat2d': (12, 64, 0.001),
               'burgers': (20, 64, 0.01), 'ode_var': (20, 50, 0.05), 'heat1d_icvar': (20, 48, 0.02), 'heat_resnet': (15, 40, 0.01), 'mixed_ic': (15, 40, 0.01),
               'poisson_sin': (20, 64, 0.005), 'burgers_silu': (15, 48, 0.01), 'mixed_acts_skip': (12, 40, 0.01),
               'wave3d': (12, 96, 0.001), 'heat4d': (12, 48, 0.01), 'hess3d_var': (12, 40, 0.01),
               'kdv': (15, 48, 0.005), 'plate': (10, 40, 0.005), 'kdv_icvar': (15, 48, 0.01),
               'kdv_silu': (15, 48, 0.005), 'kdv_resnet': (15, 48, 0.005)}
# (no trajectory for 'beam' and 'biharmonic': the reference's own fp32 fit is not reproducible there — nested autograd of
#  order 4 returns losses of 1.78 and 921.7 (beam), 97.3 (biharmonic) at steps where fp64 gives 0.177, 0.169 and 5.86;
#  tests/test_emul.py holds the fused math to the fp64 oracle along those fits instead)


def make_points(name, batch, seed):
    """ Deterministic explicit points: uniform in the problem's per-column ranges, fp32. """
    cfg = PROBLEMS[name]
    rng = np.random.RandomState(seed)
    cols = [rng.uniform(lo, hi, size=(batch, 1)) for lo, hi in cfg['ranges']]
    return np.concatenate(cols, axis=1).astype(np.float32)


def layer_plan(name):
    """ (activation per dense layer, skip source per dense layer) parsed from the layout string. """
    cfg = PROBLEMS[name]
    acts, skips, stack = [], [], []
    layout = cfg['layout'].replace(' ', '')
    spec = cfg['activation']
    spec = list(spec) if isinstance(spec, (list, tuple)) else [spec] * layout.count('a')
    names = [(a if isinstance(a, str) else a.__name__).lower() for a in spec]
    i_a = 0
    for letter in layout:
        if letter == 'f':
            acts.append('none'); skips.append(None)
        elif letter == 'a':
            acts[-1] = names[i_a]
            i_a += 1
        elif letter == 'R':
            stack.append(len(acts) - 1)
        elif letter == '+':
            skips[-1] = stack.pop()
    return acts, skips


def make_ic(name, V):
    """ initial_condition argument of the problem (callable / number / None); problems whose initial
    condition uses trainable variables build it from the V token of the implementation under test. """
    cfg = PROBLEMS[name]
    if 'ic_factory' in cfg:
        return cfg['ic_factory'](V)
    return cfg['ic']


def has_ic(name):
    cfg = PROBLEMS[name]
    return cfg['ic'] is not None or 'ic_factory' in cfg


def bind(name, D, V):
    """ Equation callable with the reference signature `equation(u, *xs)`. """
    eq = PROBLEMS[name]['equation']
    return lambda u, *xs: eq(u, *xs, D=D, V=V)


def reshape_and_concat_cases(n_cases=200, seed=0):
    """ Deterministic argument mixes for `Solver.reshape_and_concat` (how `predict` and constraints read numbers /
    arrays / lists / tensors): a list of argument lists. """
    rng = np.random.RandomState(seed)
    cases = []
    for _ in range(n_cases):
        n = int(rng.choice([1, 2, 5, 16]))
        args = []
        for _ in range(int(rng.randint(1, 5))):
            kind = int(rng.randint(7))
            if kind == 0:
                args.append(float(np.round(rng.uniform(-3, 3), 3)))
            elif kind == 1:
                args.append(int(rng.randint(-3, 4)))
            elif kind == 2:
                args.append(rng.uniform(-1, 1, size=n).astype(np.float32))
            elif kind == 3:
                args.append(rng.uniform(-1, 1, size=(n, 1)))
            elif kind == 4:
                args.append(list(np.round(rng.uniform(-1, 1, size=n), 3)))
            elif kind == 5:
                args.append(torch.tensor(rng.uniform(-1, 1, size=n), dtype=torch.float32))
            else:
                args.append(torch.tensor(rng.uniform(-1, 1, size=(n, 1)), dtype=torch.float32))
        cases.append(args)
    return cases
