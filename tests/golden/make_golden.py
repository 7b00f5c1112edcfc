"""Generate the golden vectors under tests/golden/ by running the REFERENCE (google-research/
torchsde v0.2.6, a source tree named by TSDE_REFERENCE_SRC) on the CPU.

    TSDE_REFERENCE_SRC=/path/to/torchsde-0.2.6 python tests/golden/make_golden.py

The reference cannot travel to the GPU box, so its outputs are committed as small .npz fixtures
together with this script.  `trampoline` (a pure-python dependency of the reference that is not
installed and cannot be downloaded here) is provided by oracle/refshim/trampoline.py.

What is recorded
  solver_*.npz   reference `sdeint` output for one (problem, method, dtype) with the Brownian
                 increments it consumed (so any solver can be replayed on identical increments);
  bridge_*.npz   reference Brownian-bridge / merge / Davie-Foster outputs for fixed inputs and fixed
                 normals (its `_randn` is monkey-patched to serve recorded arrays);
  adjoint_*.npz  reference `sdeint_adjoint` (reversible_heun / adjoint_reversible_heun) gradients.
"""
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, os.path.join(ROOT, 'oracle', 'refshim'))
REFERENCE = os.environ.get('TSDE_REFERENCE_SRC')
if not REFERENCE:
    sys.exit("make_golden.py: set TSDE_REFERENCE_SRC to a torchsde v0.2.6 source tree (the directory holding torchsde/)")
sys.path.insert(0, REFERENCE)
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402
import torchsde  # noqa: E402  (the reference)
from torchsde._brownian import brownian_interval as ref_bi  # noqa: E402

from tests import problems  # noqa: E402

assert torchsde.__version__ == '0.2.6'


class Recorder:
    """Wraps a reference BrownianInterval and logs every query + answer."""

    def __init__(self, bm):
        self.bm = bm
        self.shape = bm.shape
        self.levy_area_approximation = bm.levy_area_approximation
        self.log = []

    def __call__(self, ta, tb=None, return_U=False, return_A=False):
        A = None
        if self.bm._have_A:
            W, U, A = self.bm(ta, tb, return_U=True, return_A=True)
        elif self.bm._have_H:
            W, U = self.bm(ta, tb, return_U=True)
        else:
            W, U = self.bm(ta, tb), None
        self.log.append((float(ta), float(tb), W.numpy().copy(), None if U is None else U.numpy().copy(),
                         None if A is None else A.numpy().copy()))
        if return_U:
            return (W, U, A) if return_A else (W, U)
        return (W, A) if return_A else W


def solver_case(name, kind, method, sde_type, d, m, dtype, B=4, ts=None, dt=0.05, options=None, seed=0):
    torch.manual_seed(1234 + seed)
    tdt = torch.float64 if dtype == 'f64' else torch.float32
    sde = problems.make(kind, d, m, sde_type, dtype=tdt, seed=seed)
    y0 = (0.1 + 0.5 * torch.rand(B, d, dtype=torch.float64)).to(tdt)
    ts = torch.tensor(ts, dtype=tdt)
    levy = 'space-time' if method == 'srk' else 'none'
    bm_m = d if kind == 'gbm' else m
    bm = torchsde.BrownianInterval(float(ts[0]), float(ts[-1]), size=(B, bm_m), dtype=tdt, entropy=77 + seed,
                                   levy_area_approximation=levy)
    rec = Recorder(bm)
    with torch.no_grad():
        out = torchsde.sdeint(sde, y0, ts, bm=rec, method=method, dt=dt, options=options,
                              extra=(method == 'reversible_heun'))
    if method == 'reversible_heun':
        ys, extra = out
    else:
        ys, extra = out, ()
    save = dict(y0=y0.numpy(), ts=ts.numpy(), dt=np.float64(dt), ys=ys.numpy(),
                ta=np.array([r[0] for r in rec.log]), tb=np.array([r[1] for r in rec.log]),
                W=np.stack([r[2] for r in rec.log]),
                kind=kind, method=method, sde_type=sde_type, d=d, m=m, dtype=dtype, seed=seed,
                grad_free=bool(options and options.get('grad_free')))
    if rec.log[0][3] is not None:
        save['U'] = np.stack([r[3] for r in rec.log])
    for i, e in enumerate(extra):
        save[f'extra{i}'] = e.numpy()
    np.savez_compressed(os.path.join(HERE, f'solver_{name}.npz'), **save)
    print('wrote', name, ys.shape, len(rec.log), 'increments')


def all_solver_cases():
    aligned = [0.0, 0.1, 0.2, 0.3]
    ragged = np.linspace(0.0, 0.3, 5).tolist()  # spacing 0.075 vs dt 0.05: exercises linear_interp
    cases = []
    for dtype in ('f64', 'f32'):
        for method, opts in (('euler', None), ('milstein', None), ('milstein', {'grad_free': True}), ('srk', None)):
            tag = method + ('_gf' if opts else '')
            cases.append((f'gbm_ito_{tag}_{dtype}', 'gbm', method, 'ito', 6, 6, dtype, aligned, opts))
        for method in ('milstein', 'heun', 'midpoint', 'euler_heun', 'reversible_heun'):
            cases.append((f'gbm_strat_{method}_{dtype}', 'gbm', method, 'stratonovich', 8, 8, dtype, aligned, None))
    cases.append(('gbm_ito_milstein_ragged_f64', 'gbm', 'milstein', 'ito', 6, 6, 'f64', ragged, None))
    cases.append(('gbm_ito_srk_ragged_f32', 'gbm', 'srk', 'ito', 8, 8, 'f32', ragged, None))
    for method, opts in (('euler', None), ('milstein', None), ('milstein', {'grad_free': True}), ('srk', None)):
        tag = method + ('_gf' if opts else '')
        cases.append((f'scalar_ito_{tag}_f64', 'scalar', method, 'ito', 5, 1, 'f64', aligned, opts))
    for method in ('milstein', 'heun', 'midpoint', 'euler_heun', 'reversible_heun'):
        cases.append((f'scalar_strat_{method}_f64', 'scalar', method, 'stratonovich', 5, 1, 'f64', aligned, None))
    for (d, m) in ((3, 2), (4, 8)):
        for method in ('euler', 'milstein', 'srk'):
            cases.append((f'additive{d}x{m}_ito_{method}_f64', 'additive', method, 'ito', d, m, 'f64', aligned, None))
        cases.append((f'general{d}x{m}_ito_euler_f64', 'general', 'euler', 'ito', d, m, 'f64', aligned, None))
        for method in ('heun', 'midpoint', 'euler_heun', 'reversible_heun'):
            cases.append((f'general{d}x{m}_strat_{method}_f64', 'general', method, 'stratonovich', d, m, 'f64',
                          aligned, None))
            cases.append((f'additive{d}x{m}_strat_{method}_f64', 'additive', method, 'stratonovich', d, m, 'f64',
                          aligned, None))
    cases.append(('general4x8_ito_euler_f32', 'general', 'euler', 'ito', 4, 8, 'f32', ragged, None))
    cases.append(('additive4x8_ito_srk_f32', 'additive', 'srk', 'ito', 4, 8, 'f32', aligned, None))
    for i, (name, kind, method, sde_type, d, m, dtype, ts, opts) in enumerate(cases):
        solver_case(name, kind, method, sde_type, d, m, dtype, ts=ts, options=opts, seed=i % 5)


def ito_diagonal_fixture():
    """diagnostics/ito_diagonal.py:26-53, run A (B=16, ts=linspace(0,2,10), dt=0.1) with the
    reference's own NeuralDiagonal(d=5), seeds as diagnostics/utils.py:123-127."""
    import random
    from tests import problems as my_problems
    import importlib.util
    spec = importlib.util.spec_from_file_location('ref_problems', os.path.join(REFERENCE, 'tests', 'problems.py'))
    ref_problems = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(ref_problems)
    torch.set_default_dtype(torch.float64)
    torch.manual_seed(1147481649)
    np.random.seed(1147481649)
    random.seed(1147481649)
    B, d = 16, 5
    t0, t1, steps, dt = 0., 2., 10, 1e-1
    ts = torch.linspace(t0, t1, steps=steps)
    sde = ref_problems.NeuralDiagonal(d=d)
    y0 = torch.full((B, d), fill_value=0.1)
    mine = my_problems.MLPDiagonal(d)
    mine.load_state_dict(sde.state_dict())
    for method, opts, tag in (('euler', None, 'euler'), ('milstein', None, 'milstein'),
                              ('milstein', dict(grad_free=True), 'milstein_gf'), ('srk', None, 'srk')):
        bm = torchsde.BrownianInterval(t0=t0, t1=t1, size=(B, d), dtype=y0.dtype,
                                       levy_area_approximation='space-time', entropy=1147481649)
        rec = Recorder(bm)
        with torch.no_grad():
            ys = torchsde.sdeint(sde, y0, ts, rec, method=method, dt=dt, options=opts)
            ys_mine_def = torchsde.sdeint(mine, y0, ts, Recorder(torchsde.BrownianInterval(
                t0=t0, t1=t1, size=(B, d), dtype=y0.dtype, levy_area_approximation='space-time',
                entropy=1147481649)), method=method, dt=dt, options=opts)
        assert torch.equal(ys, ys_mine_def)  # tests/problems.MLPDiagonal == reference NeuralDiagonal
        save = dict(y0=y0.numpy(), ts=ts.numpy(), dt=np.float64(dt), ys=ys.numpy(),
                    ta=np.array([r[0] for r in rec.log]), tb=np.array([r[1] for r in rec.log]),
                    W=np.stack([r[2] for r in rec.log]), U=np.stack([r[3] for r in rec.log]),
                    method=method, grad_free=bool(opts), d=d)
        for k, v in sde.state_dict().items():
            save['param.' + k] = v.numpy()
        np.savez_compressed(os.path.join(HERE, f'ito_diagonal_{tag}.npz'), **save)
        print('wrote ito_diagonal', tag)
    torch.set_default_dtype(torch.float32)


def bridge_cases():
    """Bridge / merge / Levy-area formulas of the reference with its normals pinned."""
    rng = np.random.RandomState(7)
    for levy in ('none', 'space-time', 'davie', 'foster'):
        for dtype, tdt in (('f64', torch.float64), ('f32', torch.float32)):
            B, m = 5, 3
            served = {}

            def fake_randn(size, dtype_, device, seed, _served=served, _tdt=tdt):
                key = (tuple(size), int(seed))
                if key not in _served:
                    _served[key] = torch.from_numpy(rng.randn(*size)).to(_tdt)
                return _served[key]

            orig = ref_bi._randn
            ref_bi._randn = fake_randn
            try:
                W0 = torch.from_numpy(rng.randn(B, m)).to(tdt)
                H0 = torch.from_numpy(rng.randn(B, m) * 0.3).to(tdt)
                bm = torchsde.BrownianInterval(0.0, 1.0, size=(B, m), dtype=tdt, entropy=5,
                                               levy_area_approximation=levy, W=W0, H=H0)
                queries = [(0.0, 0.3), (0.3, 0.45), (0.45, 1.0), (0.1, 0.2), (0.2, 0.7), (0.05, 0.95)]
                outs = []
                for (a, b) in queries:
                    r = bm(a, b, return_U=levy != 'none', return_A=levy in ('davie', 'foster'))
                    outs.append(r if isinstance(r, tuple) else (r,))
                # dump the tree: every split node with its normals
                nodes = []

                def walk(node, path):
                    if node._midway is None:
                        return
                    x1 = served.get(((B, m), int(node._W_seed)))
                    x2 = served.get(((B, m), int(node._H_seed)))
                    nodes.append((path, node._start, node._midway, node._end, x1, x2,
                                  int(node._left_a_seed), int(node._right_a_seed)))
                    walk(node._left_child, path + 'L')
                    walk(node._right_child, path + 'R')

                walk(bm, '')
                save = dict(W0=W0.numpy(), H0=H0.numpy(), levy=levy, queries=np.array(queries),
                            top_a_seed=int(bm._top_a_seed))
                for i, o in enumerate(outs):
                    for j, x in enumerate(o):
                        save[f'out{i}_{j}'] = x.numpy()
                save['n_nodes'] = len(nodes)
                for i, (path, s, mid, e, x1, x2, las, ras) in enumerate(nodes):
                    save[f'node{i}_path'] = path
                    save[f'node{i}_t'] = np.array([s, mid, e])
                    if x1 is not None:
                        save[f'node{i}_x1'] = x1.numpy()
                    if x2 is not None:
                        save[f'node{i}_x2'] = x2.numpy()
                    save[f'node{i}_aseeds'] = np.array([las, ras], dtype=np.int64)
                for (size, seed), val in served.items():
                    if len(size) == 3:
                        save[f'anoise_{seed}'] = val.numpy()
                np.savez_compressed(os.path.join(HERE, f'bridge_{levy}_{dtype}.npz'), **save)
                print('wrote bridge', levy, dtype, len(nodes), 'nodes')
            finally:
                ref_bi._randn = orig


def adjoint_cases():
    for name, kind, d, m in (('gbm', 'gbm', 6, 6), ('general', 'general', 4, 8), ('scalar', 'scalar', 5, 1),
                             ('additive', 'additive', 3, 2)):
        torch.manual_seed(99)
        tdt = torch.float64
        sde = problems.make(kind, d, m, 'stratonovich', dtype=tdt, seed=3)
        B = 4
        y0 = (0.1 + 0.5 * torch.rand(B, d, dtype=tdt)).requires_grad_(True)
        ts = torch.tensor([0.0, 0.1, 0.2, 0.3], dtype=tdt)
        bm_m = d if kind == 'gbm' else m
        bm = torchsde.BrownianInterval(0.0, 0.3, size=(B, bm_m), dtype=tdt, entropy=11)
        rec = Recorder(bm)
        ys = torchsde.sdeint_adjoint(sde, y0, ts, bm=rec, method='reversible_heun',
                                     adjoint_method='adjoint_reversible_heun', dt=0.05)
        weights = torch.linspace(0.5, 1.5, ys.numel(), dtype=tdt).reshape(ys.shape)
        loss = (ys * weights).sum()
        loss.backward()
        save = dict(y0=y0.detach().numpy(), ts=ts.numpy(), dt=np.float64(0.05), ys=ys.detach().numpy(),
                    weights=weights.numpy(), grad_y0=y0.grad.numpy(), kind=kind, d=d, m=m,
                    ta=np.array([r[0] for r in rec.log]), tb=np.array([r[1] for r in rec.log]),
                    W=np.stack([r[2] for r in rec.log]))
        for n, p in sde.named_parameters():
            save['grad.' + n] = p.grad.numpy()
        np.savez_compressed(os.path.join(HERE, f'adjoint_{name}.npz'), **save)
        print('wrote adjoint', name)


def generic_adjoint_cases():
    """sdeint_adjoint through the augmented AdjointSDE (adjoint_sde.py) with the default adjoint methods
    (adjoint.py:281-296)."""
    cases = [('gbm_ito_euler', 'gbm', 'ito', 'euler', None, 6, 6), ('gbm_ito_srk', 'gbm', 'ito', 'srk', None, 5, 5),
             ('general_ito_euler', 'general', 'ito', 'euler', None, 4, 3),
             ('scalar_ito_milstein', 'scalar', 'ito', 'milstein', None, 5, 1),
             ('additive_ito_srk', 'additive', 'ito', 'srk', None, 3, 2),
             ('general_strat_midpoint', 'general', 'stratonovich', 'midpoint', None, 4, 3),
             ('gbm_strat_heun', 'gbm', 'stratonovich', 'heun', None, 6, 6),
             ('additive_strat_euler_heun', 'additive', 'stratonovich', 'euler_heun', 'heun', 3, 2),
             ('scalar_strat_midpoint_eh', 'scalar', 'stratonovich', 'midpoint', 'euler_heun', 5, 1)]
    for i, (name, kind, sde_type, method, adjoint_method, d, m) in enumerate(cases):
        torch.manual_seed(77 + i)
        tdt = torch.float64
        sde = problems.make(kind, d, m, sde_type, dtype=tdt, seed=i + 1)
        B = 3
        y0 = (0.1 + 0.5 * torch.rand(B, d, dtype=tdt)).requires_grad_(True)
        ts = torch.tensor([0.0, 0.1, 0.2, 0.3], dtype=tdt)
        levy = 'space-time' if method == 'srk' else 'none'
        bm_m = d if kind == 'gbm' else m
        bm = torchsde.BrownianInterval(0.0, 0.3, size=(B, bm_m), dtype=tdt, entropy=900 + i, levy_area_approximation=levy)
        rec = Recorder(bm)
        ys = torchsde.sdeint_adjoint(sde, y0, ts, bm=rec, method=method, adjoint_method=adjoint_method, dt=0.05)
        weights = torch.linspace(0.5, 1.5, ys.numel(), dtype=tdt).reshape(ys.shape)
        (ys * weights).sum().backward()
        save = dict(y0=y0.detach().numpy(), ts=ts.numpy(), dt=np.float64(0.05), ys=ys.detach().numpy(),
                    weights=weights.numpy(), grad_y0=y0.grad.numpy(), kind=kind, d=d, m=m, sde_type=sde_type,
                    method=method, adjoint_method='' if adjoint_method is None else adjoint_method, seed=i + 1,
                    ta=np.array([r[0] for r in rec.log]), tb=np.array([r[1] for r in rec.log]),
                    W=np.stack([r[2] for r in rec.log]))
        if rec.log[0][3] is not None:
            save['U'] = np.stack([r[3] for r in rec.log])
        for n, p in sde.named_parameters():
            save['grad.' + n] = p.grad.numpy()
        np.savez_compressed(os.path.join(HERE, f'genadj_{name}.npz'), **save)
        print('wrote generic adjoint', name)


def log_ode_cases():
    """methods/log_ode.py with davie / foster Levy area (the recorder also logs A)."""
    for i, (name, kind, d, m, levy) in enumerate((('general_foster', 'general', 4, 3, 'foster'),
                                                  ('general_davie', 'general', 3, 4, 'davie'),
                                                  ('gbm_foster', 'gbm', 5, 5, 'foster'),
                                                  ('additive_davie', 'additive', 3, 2, 'davie'))):
        torch.manual_seed(55 + i)
        tdt = torch.float64
        sde = problems.make(kind, d, m, 'stratonovich', dtype=tdt, seed=i)
        B = 4
        y0 = (0.1 + 0.5 * torch.rand(B, d, dtype=tdt))
        ts = torch.tensor([0.0, 0.1, 0.2, 0.3], dtype=tdt)
        bm_m = d if kind == 'gbm' else m
        bm = torchsde.BrownianInterval(0.0, 0.3, size=(B, bm_m), dtype=tdt, entropy=300 + i, levy_area_approximation=levy)
        rec = Recorder(bm)
        ys = torchsde.sdeint(sde, y0, ts, bm=rec, method='log_ode', dt=0.05)
        save = dict(y0=y0.numpy(), ts=ts.numpy(), dt=np.float64(0.05), ys=ys.detach().numpy(), kind=kind, d=d, m=m,
                    sde_type='stratonovich', method='log_ode', dtype='f64', seed=i, grad_free=False, levy=levy,
                    ta=np.array([r[0] for r in rec.log]), tb=np.array([r[1] for r in rec.log]),
                    W=np.stack([r[2] for r in rec.log]), U=np.stack([r[3] for r in rec.log]),
                    A=np.stack([r[4] for r in rec.log]))
        np.savez_compressed(os.path.join(HERE, f'logode_{name}.npz'), **save)
        print('wrote log_ode', name)


def backprop_cases():
    """Gradients by backpropagation THROUGH the reference solver (plain sdeint under autograd)."""
    cases = [('gbm', 'ito', 'euler', None, 6, 6), ('gbm', 'ito', 'milstein', None, 6, 6),
             ('gbm', 'ito', 'milstein', {'grad_free': True}, 5, 5), ('gbm', 'ito', 'srk', None, 8, 8),
             ('gbm', 'stratonovich', 'heun', None, 6, 6), ('gbm', 'stratonovich', 'midpoint', None, 6, 6),
             ('gbm', 'stratonovich', 'euler_heun', None, 6, 6), ('gbm', 'stratonovich', 'reversible_heun', None, 6, 6),
             ('gbm', 'stratonovich', 'milstein', None, 6, 6),
             ('general', 'ito', 'euler', None, 4, 3), ('general', 'stratonovich', 'heun', None, 4, 8),
             ('general', 'stratonovich', 'reversible_heun', None, 4, 8),
             ('additive', 'ito', 'srk', None, 3, 2), ('additive', 'ito', 'milstein', None, 4, 8),
             ('scalar', 'ito', 'milstein', None, 5, 1), ('scalar', 'ito', 'srk', None, 5, 1),
             ('scalar', 'stratonovich', 'midpoint', None, 5, 1)]
    ragged = np.linspace(0.0, 0.3, 5).tolist()
    for i, (kind, sde_type, method, opts, d, m) in enumerate(cases):
        torch.manual_seed(31 + i)
        tdt = torch.float64
        sde = problems.make(kind, d, m, sde_type, dtype=tdt, seed=i + 2)
        B = 3
        y0 = (0.1 + 0.5 * torch.rand(B, d, dtype=tdt)).requires_grad_(True)
        ts = torch.tensor(ragged if i % 3 == 0 else [0.0, 0.1, 0.2, 0.3], dtype=tdt)
        levy = 'space-time' if method == 'srk' else 'none'
        bm_m = d if kind == 'gbm' else m
        bm = torchsde.BrownianInterval(0.0, 0.3, size=(B, bm_m), dtype=tdt, entropy=600 + i, levy_area_approximation=levy)
        rec = Recorder(bm)
        ys = torchsde.sdeint(sde, y0, ts, bm=rec, method=method, dt=0.05, options=opts)
        weights = torch.linspace(0.5, 1.5, ys.numel(), dtype=tdt).reshape(ys.shape)
        (ys * weights).sum().backward()
        tag = method + ('_gf' if opts else '')
        save = dict(y0=y0.detach().numpy(), ts=ts.numpy(), dt=np.float64(0.05), ys=ys.detach().numpy(),
                    weights=weights.numpy(), grad_y0=y0.grad.numpy(), kind=kind, d=d, m=m, sde_type=sde_type,
                    method=method, grad_free=bool(opts), seed=i + 2,
                    ta=np.array([r[0] for r in rec.log]), tb=np.array([r[1] for r in rec.log]),
                    W=np.stack([r[2] for r in rec.log]))
        if rec.log[0][3] is not None:
            save['U'] = np.stack([r[3] for r in rec.log])
        for n, p in sde.named_parameters():
            save['grad.' + n] = p.grad.numpy()
        np.savez_compressed(os.path.join(HERE, f'backprop_{kind}_{sde_type}_{tag}.npz'), **save)
        print('wrote backprop', kind, sde_type, tag)


def adaptive_cases():
    """Adaptive stepping (base_solver.py:117-142) on identical increments: the recorder logs every proposal's
    three queries; rtol/atol chosen so that proposals get rejected."""
    cases = [('gbm_ito_euler', 'gbm', 'euler', 'ito', 6, 6), ('gbm_ito_srk', 'gbm', 'srk', 'ito', 8, 8),
             ('gbm_ito_milstein', 'gbm', 'milstein', 'ito', 6, 6),
             ('general_strat_heun', 'general', 'heun', 'stratonovich', 4, 8),
             ('additive_strat_midpoint', 'additive', 'midpoint', 'stratonovich', 3, 2),
             ('scalar_strat_reversible_heun', 'scalar', 'reversible_heun', 'stratonovich', 5, 1)]
    import warnings
    for i, (name, kind, method, sde_type, d, m) in enumerate(cases):
        torch.manual_seed(4321 + i)
        tdt = torch.float64
        sde = problems.make(kind, d, m, sde_type, dtype=tdt, seed=i)
        B = 4
        y0 = (0.1 + 0.5 * torch.rand(B, d, dtype=tdt))
        ts = torch.tensor([0.0, 0.4, 1.0], dtype=tdt)
        levy = 'space-time' if method == 'srk' else 'none'
        bm_m = d if kind == 'gbm' else m
        bm = torchsde.BrownianInterval(0.0, 1.0, size=(B, bm_m), dtype=tdt, entropy=500 + i, levy_area_approximation=levy)
        rec = Recorder(bm)
        rtol, atol = 1e-3, 1e-3
        with torch.no_grad(), warnings.catch_warnings():
            warnings.simplefilter('ignore')
            ys = torchsde.sdeint(sde, y0, ts, bm=rec, method=method, dt=0.2, adaptive=True, rtol=rtol, atol=atol,
                                 dt_min=1e-4)
        save = dict(y0=y0.numpy(), ts=ts.numpy(), dt=np.float64(0.2), ys=ys.numpy(), rtol=rtol, atol=atol, dt_min=1e-4,
                    ta=np.array([r[0] for r in rec.log]), tb=np.array([r[1] for r in rec.log]),
                    W=np.stack([r[2] for r in rec.log]), kind=kind, method=method, sde_type=sde_type, d=d, m=m,
                    dtype='f64', seed=i, grad_free=False, n_queries=len(rec.log))
        if rec.log[0][3] is not None:
            save['U'] = np.stack([r[3] for r in rec.log])
        np.savez_compressed(os.path.join(HERE, f'adaptive_{name}.npz'), **save)
        print('wrote adaptive', name, len(rec.log) // 3, 'proposals')


def _rec_save(rec, save):
    save['ta'] = np.array([r[0] for r in rec.log])
    save['tb'] = np.array([r[1] for r in rec.log])
    save['W'] = np.stack([r[2] for r in rec.log])
    if rec.log[0][3] is not None:
        save['U'] = np.stack([r[3] for r in rec.log])
    return save


def variant_cases():
    """User-callable subsets the reference accepts beyond plain f/g (VERDICT r01 missing #5): SRK calling the user's
    g_prod (srk.py:87,102,109), additive SRK with a single Brownian channel, Euler-Heun with f_and_g_prod + g but no
    g_prod (euler_heun.py:38)."""
    cases = [('gbm_srk_f+g+g_prod', 'gbm', 'srk', 'ito', 6, 6, ('f', 'g', 'g_prod')),
             ('scalar_srk_f+g+g_prod', 'scalar', 'srk', 'ito', 5, 1, ('f', 'g', 'g_prod')),
             ('additive_srk_f+g_prod', 'additive', 'srk', 'ito', 4, 3, ('f', 'g_prod')),
             ('additive3x1_srk_f+g', 'additive', 'srk', 'ito', 3, 1, ('f', 'g')),
             ('additive3x1_euler_f+g', 'additive', 'euler', 'ito', 3, 1, ('f', 'g')),
             ('additive3x1_heun_f+g', 'additive', 'heun', 'stratonovich', 3, 1, ('f', 'g')),
             ('general_euler_heun_f_and_g_prod+g', 'general', 'euler_heun', 'stratonovich', 4, 3, ('f_and_g_prod', 'g')),
             ('gbm_euler_heun_f_and_g_prod+g', 'gbm', 'euler_heun', 'stratonovich', 6, 6, ('f_and_g_prod', 'g')),
             ('gbm_euler_heun_f_and_g_prod+f_and_g', 'gbm', 'euler_heun', 'stratonovich', 6, 6,
              ('f_and_g_prod', 'f_and_g', 'g')),
             ('gbm_milstein_f+g+g_prod', 'gbm', 'milstein', 'ito', 6, 6, ('f', 'g', 'g_prod')),
             ('general_heun_f+g_prod', 'general', 'heun', 'stratonovich', 4, 3, ('f', 'g_prod'))]
    for i, (name, kind, method, sde_type, d, m, offered) in enumerate(cases):
        torch.manual_seed(777 + i)
        tdt = torch.float64
        sde = problems.WithProds(problems.make(kind, d, m, sde_type, dtype=tdt, seed=i), offered)
        B = 4
        y0 = 0.1 + 0.5 * torch.rand(B, d, dtype=tdt)
        ts = torch.tensor([0.0, 0.1, 0.2, 0.3], dtype=tdt)
        levy = 'space-time' if method == 'srk' else 'none'
        bm_m = d if kind == 'gbm' else m
        bm = torchsde.BrownianInterval(0.0, 0.3, size=(B, bm_m), dtype=tdt, entropy=900 + i, levy_area_approximation=levy)
        rec = Recorder(bm)
        with torch.no_grad():
            ys = torchsde.sdeint(sde, y0, ts, bm=rec, method=method, dt=0.05)
        save = _rec_save(rec, dict(y0=y0.numpy(), ts=ts.numpy(), dt=np.float64(0.05), ys=ys.numpy(), kind=kind,
                                   method=method, sde_type=sde_type, d=d, m=m, dtype='f64', seed=i,
                                   offered=','.join(offered)))
        np.savez_compressed(os.path.join(HERE, f'variant_{name}.npz'), **save)
        print('wrote variant', name)


def logqp_cases():
    """`logqp=True` (sdeint.py:141-145,284-295; base_sde.py:240-306): ys and the per-interval log-ratio, forward
    solves and the gradient of a loss of both through sdeint_adjoint."""
    cases = [('diag_ito_euler', 'diagonal', 'ito', 'euler', False), ('diag_ito_srk', 'diagonal', 'ito', 'srk', False),
             ('diag_strat_midpoint', 'diagonal', 'stratonovich', 'midpoint', False),
             ('general_strat_heun', 'general', 'stratonovich', 'heun', False),
             ('general_ito_euler', 'general', 'ito', 'euler', False),
             ('diag_strat_reversible_heun_adjoint', 'diagonal', 'stratonovich', 'reversible_heun', True),
             ('general_strat_reversible_heun_adjoint', 'general', 'stratonovich', 'reversible_heun', True),
             ('diag_ito_milstein_adjoint', 'diagonal', 'ito', 'milstein', True)]
    for i, (name, noise, sde_type, method, adjoint) in enumerate(cases):
        torch.manual_seed(4100 + i)
        tdt = torch.float64
        d, m = 4, (4 if noise == 'diagonal' else 3)
        sde = problems.LatentPrior(d, m, noise, sde_type, seed=i, dtype=tdt)
        B = 5
        y0 = (0.1 + 0.5 * torch.rand(B, d, dtype=tdt)).requires_grad_(adjoint)
        ts = torch.tensor([0.0, 0.1, 0.2, 0.3], dtype=tdt)
        levy = 'space-time' if method == 'srk' else 'none'
        # (diagonal noise: the augmented state has d + 1 channels, so does the Brownian motion)
        bm_m = d + 1 if noise == 'diagonal' else m
        bm = torchsde.BrownianInterval(0.0, 0.3, size=(B, bm_m), dtype=tdt, entropy=1300 + i, levy_area_approximation=levy)
        rec = Recorder(bm)
        save = dict(ts=ts.numpy(), dt=np.float64(0.05), noise=noise, sde_type=sde_type, method=method, d=d, m=m,
                    seed=i, adjoint=adjoint)
        if adjoint:
            ys, logqp = torchsde.sdeint_adjoint(sde, y0, ts, bm=rec, method=method, dt=0.05, logqp=True)
            wy = torch.linspace(0.5, 1.5, ys.numel(), dtype=tdt).reshape(ys.shape)
            wl = torch.linspace(1.0, 2.0, logqp.numel(), dtype=tdt).reshape(logqp.shape)
            ((ys * wy).sum() + (logqp * wl).sum()).backward()
            save.update(wy=wy.numpy(), wl=wl.numpy(), grad_y0=y0.grad.numpy())
            for n, p in sde.named_parameters():
                save['grad.' + n] = (torch.zeros_like(p) if p.grad is None else p.grad).numpy()
        else:
            with torch.no_grad():
                ys, logqp = torchsde.sdeint(sde, y0, ts, bm=rec, method=method, dt=0.05, logqp=True)
        save.update(y0=y0.detach().numpy(), ys=ys.detach().numpy(), logqp=logqp.detach().numpy())
        np.savez_compressed(os.path.join(HERE, f'logqp_{name}.npz'), **_rec_save(rec, save))
        print('wrote logqp', name)


def bpadaptive_cases():
    """Backpropagation through an ADAPTIVE solve (ADVICE r01: the product used to detach silently)."""
    import warnings
    for i, (name, kind, method, sde_type, d, m) in enumerate([('gbm_ito_milstein', 'gbm', 'milstein', 'ito', 5, 5),
                                                             ('general_strat_heun', 'general', 'heun', 'stratonovich', 4, 3),
                                                             ('gbm_ito_srk', 'gbm', 'srk', 'ito', 4, 4)]):
        torch.manual_seed(8100 + i)
        tdt = torch.float64
        sde = problems.make(kind, d, m, sde_type, dtype=tdt, seed=i + 1)
        B = 3
        y0 = (0.1 + 0.5 * torch.rand(B, d, dtype=tdt)).requires_grad_(True)
        ts = torch.tensor([0.0, 0.4, 1.0], dtype=tdt)
        levy = 'space-time' if method == 'srk' else 'none'
        bm_m = d if kind == 'gbm' else m
        bm = torchsde.BrownianInterval(0.0, 1.0, size=(B, bm_m), dtype=tdt, entropy=1500 + i, levy_area_approximation=levy)
        rec = Recorder(bm)
        with warnings.catch_warnings():
            warnings.simplefilter('ignore')
            ys = torchsde.sdeint(sde, y0, ts, bm=rec, method=method, dt=0.2, adaptive=True, rtol=1e-3, atol=1e-3,
                                 dt_min=1e-4)
        weights = torch.linspace(0.5, 1.5, ys.numel(), dtype=tdt).reshape(ys.shape)
        (ys * weights).sum().backward()
        save = dict(y0=y0.detach().numpy(), ts=ts.numpy(), dt=np.float64(0.2), ys=ys.detach().numpy(), rtol=1e-3,
                    atol=1e-3, dt_min=1e-4, weights=weights.numpy(), grad_y0=y0.grad.numpy(), kind=kind, method=method,
                    sde_type=sde_type, d=d, m=m, seed=i + 1)
        for n, p in sde.named_parameters():
            save['grad.' + n] = p.grad.numpy()
        np.savez_compressed(os.path.join(HERE, f'bpadaptive_{name}.npz'), **_rec_save(rec, save))
        print('wrote bpadaptive', name, len(rec.log) // 3, 'proposals')


def gradgrad_cases():
    """Double backward through sdeint_adjoint (adjoint.py:97-113, adjoint_sde.py create_graph paths; the reference's
    tests/utils.py:97-98 gradgradcheck): gradient of a functional of the first-order adjoint gradients."""
    # (the reversible pair is absent on purpose: the reference itself cannot double-backward it — the re-entered
    # Function finds no saved extra state and AdjointReversibleHeun.init_extra_solver_state raises,
    # reversible_heun.py:93-96)
    # (... and so are Ito SDEs — additive ones included, whose adjoint SDE has general noise: the re-entered
    # adjoint's Ito correction needs `f_and_g` of the first AdjointSDE, which the reference does not define,
    # adjoint_sde.py:267-271)
    cases = [('general_strat_midpoint', 'general', 'stratonovich', 'midpoint', None, 3, 2),
             ('gbm_strat_midpoint', 'gbm', 'stratonovich', 'midpoint', None, 4, 4),
             ('scalar_strat_heun', 'scalar', 'stratonovich', 'heun', 'heun', 3, 1)]
    for i, (name, kind, sde_type, method, adjoint_method, d, m) in enumerate(cases):
        torch.manual_seed(5200 + i)
        tdt = torch.float64
        sde = problems.make(kind, d, m, sde_type, dtype=tdt, seed=i + 4)
        params = list(sde.parameters())
        B = 3
        y0 = (0.1 + 0.5 * torch.rand(B, d, dtype=tdt)).requires_grad_(True)
        ts = torch.tensor([0.0, 0.1, 0.2], dtype=tdt)
        bm_m = d if kind == 'gbm' else m
        bm = torchsde.BrownianInterval(0.0, 0.2, size=(B, bm_m), dtype=tdt, entropy=1700 + i)
        rec = Recorder(bm)
        ys = torchsde.sdeint_adjoint(sde, y0, ts, bm=rec, method=method, adjoint_method=adjoint_method, dt=0.05)
        w1 = torch.linspace(0.5, 1.5, ys.numel(), dtype=tdt).reshape(ys.shape)
        loss = (ys * w1).sum()
        first = torch.autograd.grad(loss, [y0] + params, create_graph=True, allow_unused=True)
        first = [torch.zeros_like(x) if g is None else g for g, x in zip(first, [y0] + params)]
        w2 = [torch.linspace(1.0, 2.0, g.numel(), dtype=tdt).reshape(g.shape) for g in first]
        second = sum((g * w).sum() for g, w in zip(first, w2))
        gg = torch.autograd.grad(second, [y0] + params, allow_unused=True)
        gg = [torch.zeros_like(x) if g is None else g for g, x in zip(gg, [y0] + params)]
        save = dict(y0=y0.detach().numpy(), ts=ts.numpy(), dt=np.float64(0.05), ys=ys.detach().numpy(), kind=kind,
                    sde_type=sde_type, method=method, adjoint_method=adjoint_method or '', d=d, m=m, seed=i + 4,
                    w1=w1.numpy(), first_y0=first[0].detach().numpy(), second_y0=gg[0].numpy())
        for (n, _), g1, g2, w in zip(sde.named_parameters(), first[1:], gg[1:], w2[1:]):
            save['first.' + n] = g1.detach().numpy()
            save['second.' + n] = g2.numpy()
        np.savez_compressed(os.path.join(HERE, f'gradgrad_{name}.npz'), **_rec_save(rec, save))
        print('wrote gradgrad', name, len(rec.log), 'queries')


def adjoint_adaptive_cases():
    """sdeint_adjoint with the reversible pair and adjoint_adaptive=True (adjoint.py:245-249: warns, then integrates
    the adjoint adaptively): gradients on identical increments, including the backward pass's data-dependent queries."""
    import warnings
    for i, (name, kind, d, m) in enumerate([('gbm', 'gbm', 5, 5), ('general', 'general', 4, 3), ('scalar', 'scalar', 4, 1)]):
        torch.manual_seed(6100 + i)
        tdt = torch.float64
        sde = problems.make(kind, d, m, 'stratonovich', dtype=tdt, seed=i + 6)
        B = 3
        y0 = (0.1 + 0.5 * torch.rand(B, d, dtype=tdt)).requires_grad_(True)
        ts = torch.tensor([0.0, 0.25, 0.5], dtype=tdt)
        bm_m = d if kind == 'gbm' else m
        bm = torchsde.BrownianInterval(0.0, 0.5, size=(B, bm_m), dtype=tdt, entropy=2100 + i)
        rec = Recorder(bm)
        with warnings.catch_warnings():
            warnings.simplefilter('ignore')
            ys = torchsde.sdeint_adjoint(sde, y0, ts, bm=rec, method='reversible_heun',
                                         adjoint_method='adjoint_reversible_heun', dt=0.125, adjoint_adaptive=True,
                                         adjoint_rtol=1e-2, adjoint_atol=1e-2, dt_min=2e-3)
            n_fwd = len(rec.log)
            weights = torch.linspace(0.5, 1.5, ys.numel(), dtype=tdt).reshape(ys.shape)
            (ys * weights).sum().backward()
        save = dict(y0=y0.detach().numpy(), ts=ts.numpy(), dt=np.float64(0.125), ys=ys.detach().numpy(), kind=kind, d=d,
                    m=m, seed=i + 6, weights=weights.numpy(), grad_y0=y0.grad.numpy(), rtol=1e-2, atol=1e-2,
                    dt_min=2e-3, n_forward_queries=n_fwd)
        for n, p in sde.named_parameters():
            save['grad.' + n] = p.grad.numpy()
        np.savez_compressed(os.path.join(HERE, f'adjadaptive_{name}.npz'), **_rec_save(rec, save))
        print('wrote adjadaptive', name, n_fwd, 'forward +', len(rec.log) - n_fwd, 'backward queries')


if __name__ == '__main__':
    for only in ('variant', 'logqp', 'bpadaptive', 'gradgrad', 'adjadaptive'):
        if only in sys.argv:
            {'variant': variant_cases, 'logqp': logqp_cases, 'bpadaptive': bpadaptive_cases,
             'gradgrad': gradgrad_cases, 'adjadaptive': adjoint_adaptive_cases}[only]()
            sys.exit(0)
    if 'adaptive' in sys.argv:
        adaptive_cases()
        sys.exit(0)
    if 'backprop' in sys.argv:
        backprop_cases()
        sys.exit(0)
    if 'logode' in sys.argv:
        log_ode_cases()
        sys.exit(0)
    if 'genadj' in sys.argv:
        generic_adjoint_cases()
        sys.exit(0)
    all_solver_cases()
    ito_diagonal_fixture()
    bridge_cases()
    adjoint_cases()
    adaptive_cases()
    generic_adjoint_cases()
    log_ode_cases()
    backprop_cases()
    variant_cases()
    logqp_cases()
    bpadaptive_cases()
    gradgrad_cases()
    adjoint_adaptive_cases()
