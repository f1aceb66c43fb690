""" TEST INFRASTRUCTURE ONLY — generate tests/golden/*.npz from the UNMODIFIED reference.

Run in the build container only (needs /root/reference):

    python oracle/make_golden.py [problem names …]

It imports `/root/reference/pydens/model_torch.py` as is (through oracle/batchflow_standin, the
stand-in for the un-vendored `batchflow`), builds every problem of tests/problems.py with the
reference `Solver`, and records, for fixed explicit points:

    params   flat parameters in the engine layout (W_0, b_0, …, log_scale, V…; padded to 4)
    points   [B, total] fp32
    residual, loss, grads    — from the reference's own model / D / MSELoss / backward
    u        model output (Solver.predict) on the same points
    traj_*   (some problems) losses + final params of the reference's own `Solver.fit`
             fed by a sampler that replays recorded batches

The files are small and committed; nothing at test/bench time reads /root/reference.
"""
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, os.path.join(HERE, 'batchflow_standin'))
sys.path.insert(0, '/root/reference')
sys.path.insert(0, os.path.join(ROOT, 'tests'))

import pydens as ref                                     # noqa: E402  (the unmodified reference)
from pydens import model_torch as ref_mt                 # noqa: E402
import problems as P                                     # noqa: E402

ref_mt.tqdm = lambda x, *a, **k: x                       # silence the progress bar only


def ref_V(name, init):
    return ref.V(name, data=torch.Tensor([init]))


def flat_of(solver, var_names, grads=False):
    model = solver.model
    linears = [m for m in model.conv_block.modules() if isinstance(m, torch.nn.Linear)]
    parts = []
    for lin in linears:
        for p in (lin.weight, lin.bias):
            t = p.grad if grads else p
            parts.append(torch.zeros_like(p).reshape(-1) if t is None else t.detach().reshape(-1))
    extra = [model.log_scale] + [getattr(model, n) for n in var_names]
    for p in extra:
        t = p.grad if grads else p
        parts.append(torch.zeros_like(p).reshape(-1) if t is None else t.detach().reshape(-1))
    flat = torch.cat(parts)
    pad = (-flat.numel()) % 4
    return torch.cat([flat, flat.new_zeros(pad)]).numpy().astype(np.float32)


class Replay:
    """ Sampler replaying recorded batches (reference fit calls .sample(batch_size), :433). """

    def __init__(self, batches):
        self.batches, self.i = batches, 0

    def sample(self, size):
        b = self.batches[self.i]
        self.i += 1
        assert b.shape[0] == size
        return b


def build(name, seed=0):
    cfg = P.PROBLEMS[name]
    torch.manual_seed(seed)
    solver = ref.Solver(P.bind(name, ref.D, ref_V), ndims=cfg['ndims'], nparams=cfg['nparams'],
                        initial_condition=P.make_ic(name, ref_V), boundary_condition=cfg['bc'], domain=cfg['domain'],
                        layout=cfg['layout'], features=cfg['features'], activation=cfg['activation'])
    if 'log_scale' in cfg:
        with torch.no_grad():
            solver.model.log_scale.fill_(cfg['log_scale'])
    return solver


def evaluate(solver, pts):
    """ One evaluation of the reference's loop body (:435-448, :460) on explicit points. """
    for p in solver.model.parameters():
        p.grad = None
    xs = [torch.from_numpy(pts[:, i:i + 1].copy()) for i in range(pts.shape[1])]
    for x in xs:
        x.requires_grad_()
    xs_concat = solver.reshape_and_concat(xs)
    u_hat = solver.ctx.run(solver.model, xs_concat)
    residual = solver.ctx.run(solver.equation, u_hat, *xs)
    loss = torch.nn.MSELoss()(residual, torch.zeros_like(xs[0]))
    loss.backward()
    return residual.detach().numpy().reshape(-1), float(loss.detach())


def main():
    outdir = os.path.join(ROOT, 'tests', 'golden')
    os.makedirs(outdir, exist_ok=True)
    only = set(sys.argv[1:])                              # optional: problem names to (re)generate
    for name, cfg in P.PROBLEMS.items():
        if only and name not in only:
            continue
        var_names = list(cfg.get('variables', {}))
        solver = build(name)
        pts = P.make_points(name, P.GOLDEN_BATCH[name], seed=123)
        params = flat_of(solver, var_names)
        residual, loss = evaluate(solver, pts)
        grads = flat_of(solver, var_names, grads=True)
        u = solver.predict(*[pts[:, i] for i in range(pts.shape[1])]).reshape(-1)
        out = dict(params=params, points=pts, residual=residual.astype(np.float32),
                   loss=np.float32(loss), grads=grads, u=u.astype(np.float32))
        if name in P.GOLDEN_TRAJ:
            niters, batch, lr = P.GOLDEN_TRAJ[name]
            solver = build(name)
            batches = [P.make_points(name, batch, seed=1000 + i) for i in range(niters)]
            solver.fit(niters=niters, batch_size=batch, sampler=Replay(batches), lr=lr)
            out.update(traj_losses=np.asarray(solver.losses, dtype=np.float32),
                       traj_params=flat_of(solver, var_names),
                       traj_meta=np.asarray([niters, batch, lr], dtype=np.float64))
        path = os.path.join(outdir, name + '.npz')
        np.savez_compressed(path, **out)
        print('%-12s B=%-4d P=%-6d loss=%.6e  |grad|=%.4e  -> %s' % (
            name, pts.shape[0], params.size, loss, float(np.linalg.norm(grads)), os.path.relpath(path, ROOT)))
    if not only or 'reshape_and_concat' in only:
        reshape_and_concat(outdir)


def reshape_and_concat(outdir):
    """ The reference's `Solver.reshape_and_concat` on P.reshape_and_concat_cases(): per case whether it raised,
    the output shape, and the values (fp64, concatenated). """
    cases = P.reshape_and_concat_cases()
    rejected, shapes, values = [], [], []
    for args in cases:
        try:
            want = ref.Solver.reshape_and_concat(list(args))
        except Exception:                                  # noqa: BLE001  (the reference rejects the mix)
            rejected.append(True)
            shapes.append((0, 0))
            continue
        rejected.append(False)
        shapes.append(tuple(want.shape))
        values.append(want.detach().to(torch.float64).reshape(-1).numpy())
    path = os.path.join(outdir, 'reshape_and_concat.npz')
    np.savez_compressed(path, rejected=np.asarray(rejected), shapes=np.asarray(shapes, dtype=np.int64),
                        values=np.concatenate(values))
    print('reshape_and_concat: %d cases, %d rejected -> %s' % (len(cases), sum(rejected), os.path.relpath(path, ROOT)))


if __name__ == '__main__':
    main()
