"""Differential tests of the CPU oracle and of the product's contract against the REFERENCE ITSELF
(google-research/torchsde v0.2.6).

Complements tests/test_oracle_golden.py: instead of ~110 fixed fixtures, seeded random configurations — problem kind,
method, dtype, batch/state/Brownian sizes, time grids with evaluation points off the step grid, dyadic and non-dyadic
dt — are solved by the reference on the CPU while every Brownian query it makes is recorded; the oracle is replayed on
the identical increments and the whole series compared.  The remaining tests compare accept / reject decisions,
exception types, warnings, signatures and call sequences of the product with the reference's.

The reference's side of every comparison is stored in tests/golden/live_reference.npz.xz (an xz-compressed .npz: the
arrays of each test case under '<test>/<case id>/<name>', everything else as JSON under 'outcomes'), so the module
needs no copy of the reference.  To regenerate that file, run the module against a torchsde v0.2.6 source tree; the
tests then compare with the live reference and record its results:

    TSDE_RECORD_REFERENCE=/path/to/torchsde-0.2.6 python -m pytest tests/test_oracle_live_reference.py

Recording merges into the existing file, so that a run of some of the tests (`-k ...`) updates just those cases.  After
renaming or removing cases, delete the file first and record the whole module, so that no stale entries remain.
"""
import io
import json
import lzma
import os
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, 'tests', 'golden', 'live_reference.npz.xz')
REFERENCE = os.environ.get('TSDE_RECORD_REFERENCE')  # record from this reference source tree
if REFERENCE:
    for p in (REFERENCE, os.path.join(ROOT, 'oracle', 'refshim')):
        if p not in sys.path:
            sys.path.insert(0, p)
    import torchsde  # noqa: E402  (the reference)
    assert torchsde.__version__ == '0.2.6', torchsde.__version__
else:
    torchsde = None  # replay the recorded results

from oracle import solvers  # noqa: E402
from . import problems  # noqa: E402

_recorded = {'arrays': {}, 'outcomes': {}}


def _load_golden():
    """(arrays, outcomes) stored in GOLDEN; read once."""
    if not hasattr(_load_golden, 'cache'):
        with open(GOLDEN, 'rb') as f:
            z = np.load(io.BytesIO(lzma.decompress(f.read())), allow_pickle=False)
            arrays = {k: z[k] for k in z.files}
        _load_golden.cache = (arrays, json.loads(str(arrays.pop('outcomes'))))
    return _load_golden.cache


def _plain(x):
    """JSON-representable canonical form of an outcome (tuples become lists, dtypes and other objects their repr)."""
    if isinstance(x, (list, tuple)):
        return [_plain(v) for v in x]
    if isinstance(x, dict):
        return {str(k): _plain(v) for k, v in x.items()}
    if x is None or isinstance(x, (bool, int, float, str)):
        return x
    return repr(x)


def ref_outcome(key, compute):
    """The reference's outcome for `key` in `_plain` form: `compute()` on the live reference (and recorded) when
    regenerating, the recorded value otherwise."""
    if torchsde is not None:
        value = json.loads(json.dumps(_plain(compute())))
        _recorded['outcomes'][key] = value
        return value
    return _load_golden()[1][key]


def ref_arrays(request, compute):
    """The reference's arrays for this test case: `compute()` returns a dict of arrays (and scalars / strings) from the
    live reference when regenerating; otherwise they are read back from GOLDEN."""
    prefix = request.node.originalname + '/' + (request.node.callspec.id if hasattr(request.node, 'callspec') else '') + '/'
    if torchsde is not None:
        out = {k: np.asarray(v) for k, v in compute().items()}
        _recorded['arrays'].update({prefix + k: v for k, v in out.items()})
        return out
    arrays = _load_golden()[0]
    return {k[len(prefix):]: v for k, v in arrays.items() if k.startswith(prefix)}


@pytest.fixture(scope='module', autouse=True)
def _write_recorded_results():
    """When regenerating: merge what this run recorded into GOLDEN."""
    yield
    if torchsde is None:
        return
    arrays, outcomes = {}, {}
    if os.path.exists(GOLDEN):
        arrays, outcomes = _load_golden()
    arrays = dict(arrays, **_recorded['arrays'])
    outcomes = dict(outcomes, **_recorded['outcomes'])
    buf = io.BytesIO()
    np.savez(buf, outcomes=np.asarray(json.dumps(outcomes, sort_keys=True, separators=(',', ':'))), **arrays)
    with open(GOLDEN, 'wb') as f:
        f.write(lzma.compress(buf.getvalue(), preset=9 | lzma.PRESET_EXTREME))


# (method, options) x (sde_type) x (noise kinds) that the reference accepts (its own compatibility matrix:
# methods/*.py class attributes, tests/test_sdeint.py:124-136)
MENU = [
    ('euler', None, 'ito', ('gbm', 'scalar', 'additive', 'general')),
    ('milstein', None, 'ito', ('gbm', 'scalar', 'additive')),
    ('milstein', {'grad_free': True}, 'ito', ('gbm', 'scalar')),
    ('srk', None, 'ito', ('gbm', 'scalar', 'additive')),
    ('milstein', None, 'stratonovich', ('gbm', 'scalar')),
    ('heun', None, 'stratonovich', ('gbm', 'scalar', 'additive', 'general')),
    ('midpoint', None, 'stratonovich', ('gbm', 'scalar', 'additive', 'general')),
    ('euler_heun', None, 'stratonovich', ('gbm', 'scalar', 'additive', 'general')),
    ('reversible_heun', None, 'stratonovich', ('gbm', 'scalar', 'additive', 'general')),
]


class _Recorder:
    """Logs every query the reference solver makes and the tensors it got back."""

    def __init__(self, bm):
        self.bm, self.shape, self.levy_area_approximation = bm, bm.shape, bm.levy_area_approximation
        self.log = []

    def __call__(self, ta, tb=None, return_U=False, return_A=False):
        if self.levy_area_approximation == 'none':
            W, U = self.bm(ta, tb), None
        else:
            W, U = self.bm(ta, tb, return_U=True)
        self.log.append((float(ta), float(tb), W.numpy().copy(), None if U is None else U.numpy().copy()))
        return (W, U) if return_U else W


def _draw(rng):
    method, opts, sde_type, kinds = MENU[rng.randint(len(MENU))]
    kind = kinds[rng.randint(len(kinds))]
    dtype = (torch.float64, torch.float32)[rng.randint(2)]
    B = int(rng.randint(1, 6))
    d = int(rng.randint(1, 7))
    m = 1 if kind == 'scalar' else (d if kind == 'gbm' else int(rng.randint(1, 6)))
    n_out = int(rng.randint(2, 6))
    t0 = float(rng.choice([0.0, 0.25, -0.5]))
    gaps = rng.uniform(0.03, 0.2, size=n_out - 1)
    ts = t0 + np.concatenate([[0.0], np.cumsum(gaps)])
    if rng.randint(2):
        ts = np.round(ts * 16) / 16 + np.arange(n_out) / 64.0   # dyadic points: many coincide with the step grid
    dt = float(rng.choice([2.0 ** -4, 2.0 ** -5, 0.05, 0.03]))
    return method, opts, sde_type, kind, dtype, B, d, m, ts, dt


def _log_arrays(rec):
    """The queries a `_Recorder` logged, as arrays: ta, tb, W and (with Levy area) U."""
    out = dict(ta=np.array([r[0] for r in rec.log]), tb=np.array([r[1] for r in rec.log]),
               W=np.stack([r[2] for r in rec.log]))
    if rec.log[0][3] is not None:
        out['U'] = np.stack([r[3] for r in rec.log])
    return out


@pytest.mark.parametrize('seed', range(100))
def test_oracle_equals_live_reference(request, seed):
    rng = np.random.RandomState(1000 + seed)
    method, opts, sde_type, kind, dtype, B, d, m, ts, dt = _draw(rng)
    torch.manual_seed(seed)
    sde = problems.make(kind, d, m, sde_type, dtype=dtype, seed=seed)
    y0 = (0.1 + 0.5 * torch.rand(B, d, dtype=torch.float64)).to(dtype)
    tst = torch.tensor(ts, dtype=dtype)
    levy = 'space-time' if method == 'srk' else 'none'

    def reference():
        bm = torchsde.BrownianInterval(float(tst[0]), float(tst[-1]), size=(B, m), dtype=dtype, entropy=seed,
                                       levy_area_approximation=levy)
        rec = _Recorder(bm)
        with torch.no_grad():
            out = torchsde.sdeint(sde, y0, tst, bm=rec, method=method, dt=dt, options=opts,
                                  extra=method == 'reversible_heun')
        ys, extra = (out if method == 'reversible_heun' else (out, ()))
        return dict(_log_arrays(rec), ys=ys.numpy(), **{f'extra{i}': e.numpy() for i, e in enumerate(extra)})

    r = ref_arrays(request, reference)
    ref = r['ys']
    ref_extra = [r[f'extra{i}'] for i in range(sum(k.startswith('extra') for k in r))]
    replay = problems.ReplayBM(r['ta'], r['tb'], r['W'], r.get('U'), levy=levy)
    solver = solvers.make(method, problems.NumpySDE(sde), replay, dt, opts or {})
    ys, extra = solver.integrate(y0.numpy(), tst.numpy())
    what = f"{method} {opts} {sde_type} {kind} {dtype} B={B} d={d} m={m} ts={ts} dt={dt}"
    assert ys.shape == ref.shape and ys.dtype == ref.dtype, what
    # SRK (diagonal) and derivative-free Milstein use sqrt(dt).  The reference takes it with torch's CPU sqrt of a 0-d
    # tensor, which on AVX-512 builds is not correctly rounded in fp64 (sqrt(2^-5) comes out one ulp low), the oracle
    # with the IEEE square root: those two methods are compared to a few ulps, everything else on GBM bit for bit.
    uses_sqrt = method == 'srk' or bool(opts and opts.get('grad_free'))
    if kind == 'gbm' and not uses_sqrt:      # IEEE +,* only, same op order: bit for bit
        assert np.array_equal(ys, ref), f"{what}: max abs diff {np.abs(ys - ref).max()}"
    elif kind == 'gbm':
        eps = np.finfo(ref.dtype).eps
        np.testing.assert_allclose(ys, ref, rtol=16 * eps, atol=0, err_msg=what)
    elif dtype == torch.float64:
        np.testing.assert_allclose(ys, ref, rtol=1e-12, atol=1e-14, err_msg=what)
    else:
        np.testing.assert_allclose(ys, ref, rtol=5e-6, atol=1e-6, err_msg=what)
    for a, b in zip(extra, ref_extra):
        np.testing.assert_allclose(a, b, rtol=1e-5 if dtype == torch.float32 else 1e-11,
                                   atol=1e-6 if dtype == torch.float32 else 1e-13, err_msg=what)


@pytest.mark.parametrize('seed', range(24))
def test_oracle_adaptive_equals_live_reference(request, seed):
    """Adaptive branch (base_solver.py:117-142, adaptive_stepping.py): same proposals, same accept/reject history,
    same series as the reference on the increments it consumed."""
    import warnings
    rng = np.random.RandomState(5000 + seed)
    method, opts, sde_type, kinds = MENU[rng.randint(len(MENU))]
    kind = kinds[rng.randint(len(kinds))]
    dtype = torch.float64
    B, d = int(rng.randint(1, 5)), int(rng.randint(1, 6))
    m = 1 if kind == 'scalar' else (d if kind == 'gbm' else int(rng.randint(1, 5)))
    ts = np.concatenate([[0.0], np.cumsum(rng.uniform(0.1, 0.5, size=int(rng.randint(1, 4))))])
    dt0 = float(rng.choice([0.3, 0.2, 0.125]))
    rtol, atol = float(rng.choice([1e-2, 1e-3, 3e-4])), float(rng.choice([1e-2, 1e-3, 3e-4]))
    torch.manual_seed(seed)
    sde = problems.make(kind, d, m, sde_type, dtype=dtype, seed=seed)
    y0 = 0.1 + 0.5 * torch.rand(B, d, dtype=dtype)
    tst = torch.tensor(ts, dtype=dtype)
    levy = 'space-time' if method == 'srk' else 'none'

    def reference():
        bm = torchsde.BrownianInterval(float(tst[0]), float(tst[-1]), size=(B, m), dtype=dtype, entropy=seed,
                                       levy_area_approximation=levy)
        rec = _Recorder(bm)
        with torch.no_grad(), warnings.catch_warnings():
            warnings.simplefilter('ignore')
            ys = torchsde.sdeint(sde, y0, tst, bm=rec, method=method, dt=dt0, adaptive=True, rtol=rtol, atol=atol,
                                 dt_min=1e-4, options=opts)
        return dict(_log_arrays(rec), ys=ys.numpy())

    r = ref_arrays(request, reference)
    replay = problems.ReplayBM(r['ta'], r['tb'], r['W'], r.get('U'), levy=levy)
    solver = solvers.make(method, problems.NumpySDE(sde), replay, dt0, opts or {})
    ys, _, n = solvers.integrate_adaptive(solver, y0.numpy(), tst.numpy(), rtol, atol, 1e-4)
    what = f"{method} {opts} {sde_type} {kind} B={B} d={d} m={m} ts={ts} dt={dt0} rtol={rtol} atol={atol}"
    assert 3 * n == len(r['ta']), what          # three Brownian queries per proposal: identical history
    np.testing.assert_allclose(ys, r['ys'], rtol=1e-11, atol=1e-13, err_msg=what)


@pytest.mark.parametrize('levy', ['none', 'space-time', 'davie', 'foster'])
@pytest.mark.parametrize('seed', range(6))
def test_oracle_bridge_equals_live_reference(request, seed, levy):
    """Brownian bridge / merge / Davie-Foster formulas (brownian_interval.py:78-103,188-241,643-672) on random query
    sequences: the reference's `_randn` is patched to serve recorded normals, its interval tree is dumped after the
    queries, and the oracle recomputes every answer from the same normals."""
    from .test_oracle_golden import _tree_eval
    rng = np.random.RandomState(9000 + seed)
    tdt = (torch.float64, torch.float32)[seed % 2]
    B, m = int(rng.randint(1, 5)), int(rng.randint(1, 5))

    def reference():
        """The tree dump (normals, node times and seeds) as `case`, the answers as out{query}_{W, U, A}."""
        from torchsde._brownian import brownian_interval as ref_bi
        served = {}

        def fake_randn(size, dtype_, device, seed_):
            key = (tuple(size), int(seed_))
            if key not in served:
                served[key] = torch.from_numpy(rng.randn(*size)).to(tdt)
            return served[key]

        orig = ref_bi._randn
        ref_bi._randn = fake_randn
        try:
            W0 = torch.from_numpy(rng.randn(B, m)).to(tdt)
            H0 = torch.from_numpy(rng.randn(B, m) * 0.3).to(tdt)
            bm = torchsde.BrownianInterval(0.0, 1.0, size=(B, m), dtype=tdt, entropy=5, levy_area_approximation=levy,
                                           W=W0, H=H0)
            queries = []
            for _ in range(int(rng.randint(3, 9))):
                a, b = np.sort(np.round(rng.uniform(0.0, 1.0, size=2) * 64) / 64)
                if b > a:
                    queries.append((float(a), float(b)))
            case = {}
            for i, (a, b) in enumerate(queries):
                r = bm(a, b, return_U=levy != 'none', return_A=levy in ('davie', 'foster'))
                for j, x in enumerate(r if isinstance(r, tuple) else (r,)):
                    case[f'out{i}_{j}'] = x.numpy()
            case.update(W0=W0.numpy(), H0=H0.numpy(), queries=np.array(queries), top_a_seed=int(bm._top_a_seed))
            nodes = []

            def walk(node, path):
                if node._midway is None:
                    return
                nodes.append((path, node))
                walk(node._left_child, path + 'L')
                walk(node._right_child, path + 'R')

            walk(bm, '')
            case['n_nodes'] = len(nodes)
            for i, (path, node) in enumerate(nodes):
                case[f'node{i}_path'] = path
                case[f'node{i}_t'] = np.array([node._start, node._midway, node._end])
                x1 = served.get(((B, m), int(node._W_seed)))
                x2 = served.get(((B, m), int(node._H_seed)))
                if x1 is not None:
                    case[f'node{i}_x1'] = x1.numpy()
                if x2 is not None:
                    case[f'node{i}_x2'] = x2.numpy()
                case[f'node{i}_aseeds'] = np.array([int(node._left_a_seed), int(node._right_a_seed)], dtype=np.int64)
            for (size, sd), val in served.items():
                if len(size) == 3:
                    case[f'anoise_{sd}'] = val.numpy()
        finally:
            ref_bi._randn = orig
        return case

    case = ref_arrays(request, reference)
    res = _tree_eval(case, levy)
    tol = dict(rtol=1e-5, atol=1e-5) if tdt == torch.float32 else dict(rtol=1e-12, atol=1e-13)
    assert len(res) == len(case['queries'])
    for i, (W, U, A) in enumerate(res):
        np.testing.assert_allclose(W, case[f'out{i}_0'], **tol)
        if levy != 'none':
            np.testing.assert_allclose(U, case[f'out{i}_1'], **tol)
        if levy in ('davie', 'foster'):
            np.testing.assert_allclose(A, case[f'out{i}_2'], **tol)


@pytest.mark.parametrize('seed', range(40))
def test_host_planned_grid_equals_the_grid_the_reference_walks(request, seed):
    """The product plans the time grid once on the host (torchsde_b200/_core/schedule.py) instead of evaluating
    `while curr_t < out_t` / `min(curr_t + dt, ts[-1])` on device tensors (base_solver.py:107-147).  The plan must be the
    grid the reference actually walks — including the rounding of the accumulated `curr_t + dt` in fp32 (1001 steps
    for dt = 1e-3 on [0, 1]) and the clipped last step: compared here, bit for bit, with the intervals the live
    reference queries its Brownian motion on."""
    from torchsde_b200._core import schedule
    rng = np.random.RandomState(7000 + seed)
    dtype = (torch.float32, torch.float64)[seed % 2]
    n_out = int(rng.randint(2, 6))
    t0 = float(rng.choice([0.0, 1.0, -0.3]))
    ts = t0 + np.concatenate([[0.0], np.cumsum(rng.uniform(0.02, 0.4, size=n_out - 1))])
    if seed % 3 == 0:
        ts = np.array([0.0, 1.0])
    dt = float(rng.choice([1e-3, 1e-2, 0.03, 2.0 ** -6, 0.1, 0.25])) if seed % 3 else 1e-3 * (1 + seed % 2 * 9)
    tst = torch.tensor(ts, dtype=dtype)

    def reference():
        sde = problems.make('gbm', 1, 1, 'ito', dtype=dtype, seed=0)
        bm = torchsde.BrownianInterval(float(tst[0]), float(tst[-1]), size=(1, 1), dtype=dtype, entropy=1)
        rec = _Recorder(bm)
        with torch.no_grad():
            torchsde.sdeint(sde, torch.ones(1, 1, dtype=dtype), tst, bm=rec, method='euler', dt=dt)
        log = _log_arrays(rec)
        return dict(ta=log['ta'], tb=log['tb'])

    r = ref_arrays(request, reference)
    sched = schedule.build_schedule(tst, dt)
    assert sched.n_steps == len(r['ta']), (ts, dt, dtype)
    for (a, b), ra, rb in zip(sched.steps, r['ta'], r['tb']):
        assert float(a) == ra and float(b) == rb, (ts, dt, dtype)
    if seed % 3 == 0 and dtype == torch.float32 and dt == 1e-3:
        assert sched.n_steps == 1001


@pytest.mark.parametrize('sde_type', ['ito', 'stratonovich'])
@pytest.mark.parametrize('method', ['blah', None, 'euler', 'milstein', 'srk', 'euler_heun', 'heun', 'midpoint', 'log_ode',
                                    'reversible_heun'])
@pytest.mark.parametrize('kind', ['gbm', 'scalar', 'additive', 'general'])
@pytest.mark.parametrize('levy', [None, 'none', 'space-time', 'davie', 'foster'])
def test_contract_errors_equal_the_live_reference(request, sde_type, method, kind, levy):
    """`sdeint` must reject exactly the (sde_type, noise_type, method, Levy-area) combinations the reference rejects,
    with the same exception type (ValueError).  The product is given CPU tensors: a combination it accepts gets past
    every contract check and then stops at the CUDA requirement (RuntimeError) — there is no CPU fallback."""
    import warnings
    import torchsde_b200 as tsde
    d, m = 3, {'gbm': 3, 'scalar': 1}.get(kind, 2)
    sde = problems.make(kind, d, m, sde_type, dtype=torch.float64)
    y0 = torch.ones(4, d, dtype=torch.float64)
    ts = [0.0, 0.1]

    def outcome(mod):
        bm = None if levy is None else mod.BrownianInterval(0.0, 0.1, size=(4, m), dtype=torch.float64,
                                                            levy_area_approximation=levy,
                                                            **({'device': 'cuda'} if mod is tsde else {}))
        try:
            with warnings.catch_warnings(), torch.no_grad():
                warnings.simplefilter('ignore')
                mod.sdeint(sde, y0, ts, bm=bm, method=method, dt=0.05)
        except ValueError:
            return 'ValueError'
        except (RuntimeError, NotImplementedError) as e:
            return 'accepted' if mod is tsde and ('CUDA' in str(e) or 'not implemented' in str(e)) else type(e).__name__
        return 'accepted'

    assert _plain(outcome(tsde)) == ref_outcome(request.node.name, lambda: outcome(torchsde)), \
        (sde_type, method, kind, levy)


_ADJ_METHODS = [None, 'euler', 'milstein', 'srk', 'midpoint', 'heun', 'euler_heun', 'reversible_heun', 'log_ode']
_ADJ_ADJOINTS = [None, 'euler', 'milstein', 'srk', 'midpoint', 'heun', 'euler_heun', 'adjoint_reversible_heun', 'log_ode',
                 'blah']


@pytest.mark.parametrize('sde_type', ['ito', 'stratonovich'])
@pytest.mark.parametrize('kind', ['gbm', 'scalar', 'additive', 'general'])
def test_adjoint_contract_errors_equal_the_live_reference(request, sde_type, kind):
    """`sdeint_adjoint`: 90 (method, adjoint_method) pairs per (sde_type, noise type).  The reference is run forward AND
    backward on the CPU (it builds its adjoint solver only in `backward`); the product, given CPU tensors, stops at the
    CUDA requirement once every contract check has passed.  They must agree on ValueError vs accepted, except for two
    documented cases:
      * adjoint_method='adjoint_reversible_heun' with a non-reversible forward method: the reference accepts the call
        and then dies inside `backward` with RuntimeError("Please report a bug to torchsde."); the product rejects the
        pair up front with a ValueError;
      * adjoint_method='milstein' on non-diagonal noise: NotImplementedError from the adjoint SDE's
        `g_prod_and_gdg_prod` at backward time in both (adjoint_sde.py:332-377) — not reachable without a GPU here.
    """
    import warnings
    import torchsde_b200 as tsde
    d, m = 3, {'gbm': 3, 'scalar': 1}.get(kind, 2)
    sde = problems.make(kind, d, m, sde_type, dtype=torch.float64)

    def outcome(mod, method, adj):
        y0 = torch.ones(2, d, dtype=torch.float64, requires_grad=True)
        try:
            with warnings.catch_warnings():
                warnings.simplefilter('ignore')
                ys = mod.sdeint_adjoint(sde, y0, [0.0, 0.1], method=method, adjoint_method=adj, dt=0.05)
                ys.sum().backward()
        except ValueError:
            return 'ValueError'
        except (RuntimeError, NotImplementedError) as e:
            if mod is tsde and ('CUDA' in str(e) or 'not implemented' in str(e)):
                return 'accepted'
            return type(e).__name__
        return 'accepted'

    for method in _ADJ_METHODS:
        for adj in _ADJ_ADJOINTS:
            ours = outcome(tsde, method, adj)
            ref = ref_outcome(f'{request.node.name}/{method}/{adj}', lambda: outcome(torchsde, method, adj))
            if ours == ref:
                continue
            if adj == 'adjoint_reversible_heun' and method != 'reversible_heun':
                assert (ours, ref) == ('ValueError', 'RuntimeError'), (sde_type, kind, method, adj, ours, ref)
            elif adj == 'milstein' and kind != 'gbm':
                assert (ours, ref) == ('accepted', 'NotImplementedError'), (sde_type, kind, method, adj, ours, ref)
            else:
                raise AssertionError((sde_type, kind, method, adj, ours, ref))


class _BadShape(torch.nn.Module):
    """Diagonal-noise SDE whose callables return deliberately wrong shapes."""
    noise_type, sde_type = 'diagonal', 'ito'

    def __init__(self, f_shape, g_shape):
        super().__init__()
        self.f_shape, self.g_shape = f_shape, g_shape

    def f(self, t, y):
        return torch.zeros(self.f_shape, dtype=y.dtype)

    def g(self, t, y):
        return torch.zeros(self.g_shape, dtype=y.dtype)


def _malformed_calls():
    good = problems.make('gbm', 3, 3, 'ito', dtype=torch.float64)
    gen = problems.make('general', 3, 2, 'ito', dtype=torch.float64)
    y0 = torch.ones(4, 3, dtype=torch.float64)
    yield 'y0 1-d', dict(sde=good, y0=y0[0], ts=[0.0, 0.1])
    yield 'y0 3-d', dict(sde=good, y0=y0[None], ts=[0.0, 0.1])
    yield 'y0 not a tensor', dict(sde=good, y0=[[1.0, 1.0, 1.0]], ts=[0.0, 0.1])
    yield 'ts decreasing', dict(sde=good, y0=y0, ts=[0.1, 0.0])
    yield 'ts repeated', dict(sde=good, y0=y0, ts=[0.0, 0.0, 0.1])
    yield 'ts 2-d tensor', dict(sde=good, y0=y0, ts=torch.tensor([[0.0, 0.1]], dtype=torch.float64))
    yield 'ts of strings', dict(sde=good, y0=y0, ts=['a', 'b'])
    yield 'ts single point', dict(sde=good, y0=y0, ts=[0.0])
    yield 'ts requires grad', dict(sde=good, y0=y0, ts=torch.tensor([0.0, 0.1], dtype=torch.float64, requires_grad=True))
    yield 'dt requires grad', dict(sde=good, y0=y0, ts=[0.0, 0.1], dt=torch.tensor(0.05, requires_grad=True))
    yield 'bm batch mismatch', dict(sde=good, y0=y0, ts=[0.0, 0.1], bm=(5, 3))
    yield 'bm channel mismatch', dict(sde=good, y0=y0, ts=[0.0, 0.1], bm=(4, 2))
    yield 'bm rank 1', dict(sde=good, y0=y0, ts=[0.0, 0.1], bm=(4,))
    yield 'general bm channel mismatch', dict(sde=gen, y0=y0, ts=[0.0, 0.1], bm=(4, 3))
    yield 'f wrong batch', dict(sde=_BadShape((5, 3), (4, 3)), y0=y0, ts=[0.0, 0.1])
    yield 'f wrong state', dict(sde=_BadShape((4, 2), (4, 3)), y0=y0, ts=[0.0, 0.1])
    yield 'g wrong state', dict(sde=_BadShape((4, 3), (4, 2)), y0=y0, ts=[0.0, 0.1])
    yield 'g rank 3 for diagonal', dict(sde=_BadShape((4, 3), (4, 3, 3)), y0=y0, ts=[0.0, 0.1])
    yield 'f rank 1', dict(sde=_BadShape((3,), (4, 3)), y0=y0, ts=[0.0, 0.1])
    yield 'unknown noise type', dict(sde=type('S', (torch.nn.Module,), dict(noise_type='weird', sde_type='ito', f=good.f, g=good.g))(), y0=y0, ts=[0.0, 0.1])
    yield 'unknown sde type', dict(sde=type('S', (torch.nn.Module,), dict(noise_type='diagonal', sde_type='weird', f=good.f, g=good.g))(), y0=y0, ts=[0.0, 0.1])
    yield 'no noise_type attribute', dict(sde=type('S', (torch.nn.Module,), dict(sde_type='ito', f=good.f, g=good.g))(), y0=y0, ts=[0.0, 0.1])
    yield 'no drift', dict(sde=type('S', (torch.nn.Module,), dict(noise_type='diagonal', sde_type='ito', g=good.g))(), y0=y0, ts=[0.0, 0.1])
    yield 'no diffusion', dict(sde=type('S', (torch.nn.Module,), dict(noise_type='diagonal', sde_type='ito', f=good.f))(), y0=y0, ts=[0.0, 0.1])
    yield 'logqp without h', dict(sde=good, y0=y0, ts=[0.0, 0.1], logqp=True)
    yield 'names to a missing method', dict(sde=good, y0=y0, ts=[0.0, 0.1], names={'drift': 'nope'})
    yield 'well-formed', dict(sde=good, y0=y0, ts=[0.0, 0.1])


@pytest.mark.parametrize('label', [lab for lab, _ in _malformed_calls()])
def test_malformed_calls_fail_like_the_live_reference(request, label):
    """Shape / type / attribute violations of the user-SDE protocol (sdeint.py:115-258): same exception type as the
    reference (a call the reference accepts must reach the product's CUDA requirement)."""
    import warnings
    import torchsde_b200 as tsde
    kwargs = dict(_malformed_calls())[label]

    def outcome(mod):
        kw = dict(kwargs)
        if 'bm' in kw:
            kw['bm'] = mod.BrownianInterval(0.0, 0.1, size=kw['bm'], dtype=torch.float64,
                                            **({'device': 'cuda'} if mod is tsde else {}))
        kw.setdefault('dt', 0.05)
        try:
            with warnings.catch_warnings(), torch.no_grad():
                warnings.simplefilter('ignore')
                mod.sdeint(**kw)
        except (RuntimeError, NotImplementedError) as e:
            if mod is tsde and ('CUDA' in str(e) or 'not implemented' in str(e)):
                return 'accepted'
            return type(e).__name__
        except Exception as e:  # noqa: BLE001 - the exception TYPE is what is compared
            return type(e).__name__
        return 'accepted'

    assert _plain(outcome(tsde)) == ref_outcome(request.node.name, lambda: outcome(torchsde)), label


_BI_BAD = {
    'no size no W': dict(t0=0.0, t1=1.0),
    't0 > t1': dict(t0=1.0, t1=0.0, size=(2, 3)),
    't0 == t1': dict(t0=1.0, t1=1.0, size=(2, 3)),
    'tensor t0 ok': dict(t0=torch.tensor(0.0), t1=torch.tensor(1.0), size=(2, 3)),
    'non-scalar t0': dict(t0=torch.tensor([0.0, 0.5]), t1=1.0, size=(2, 3)),
    'bad levy': dict(t0=0.0, t1=1.0, size=(2, 3), levy_area_approximation='wrong'),
    'integer dtype': dict(t0=0.0, t1=1.0, size=(2, 3), dtype=torch.int64),
    'W given': dict(t0=0.0, t1=1.0, W=torch.zeros(2, 3)),
    'W of integer dtype': dict(t0=0.0, t1=1.0, W=torch.zeros(2, 3, dtype=torch.int32)),
    'W and size disagree': dict(t0=0.0, t1=1.0, size=(2, 4), W=torch.zeros(2, 3)),
    'W and dtype disagree': dict(t0=0.0, t1=1.0, dtype=torch.float64, W=torch.zeros(2, 3, dtype=torch.float32)),
    'H without levy': dict(t0=0.0, t1=1.0, W=torch.zeros(2, 3), H=torch.zeros(2, 3)),
    'H with levy': dict(t0=0.0, t1=1.0, W=torch.zeros(2, 3), H=torch.zeros(2, 3), levy_area_approximation='space-time'),
    'H shape mismatch': dict(t0=0.0, t1=1.0, W=torch.zeros(2, 3), H=torch.zeros(2, 4), levy_area_approximation='space-time'),
    'halfway tree': dict(t0=0.0, t1=1.0, size=(2, 3), halfway_tree=True),
    'dt hint': dict(t0=0.0, t1=1.0, size=(2, 3), dt=0.1),
    'scalar size': dict(t0=0.0, t1=1.0, size=()),
    'rank-1 size': dict(t0=0.0, t1=1.0, size=(5,)),
    'entropy given': dict(t0=0.0, t1=1.0, size=(2, 3), entropy=7),
    'pool and cache sizes': dict(t0=0.0, t1=1.0, size=(2, 3), pool_size=4, cache_size=None),
    'tol': dict(t0=0.0, t1=1.0, size=(2, 3), tol=1e-3),
}


@pytest.mark.parametrize('label', sorted(_BI_BAD))
def test_brownian_interval_constructor_like_the_live_reference(request, label):
    """Constructor contract of BrownianInterval (brownian_interval.py:394-494): accepts / rejects the same arguments
    with the same exception type, and reports the same shape / dtype / levy / flags."""
    import torchsde_b200 as tsde
    kwargs = _BI_BAD[label]

    def outcome(mod):
        kw = dict(kwargs)
        try:
            bm = mod.BrownianInterval(**kw)
        except Exception as e:  # noqa: BLE001
            return type(e).__name__
        return ('ok', tuple(bm.shape), bm.dtype, bm.levy_area_approximation, bm.halfway_tree, bm.dt, bm.tol,
                bm.pool_size, bm.cache_size)

    assert _plain(outcome(tsde)) == ref_outcome(request.node.name, lambda: outcome(torchsde)), label


def test_public_signatures_equal_the_live_reference(request):
    """Drop-in boundary (SURVEY §8b): same exported names, same parameter names, order, kinds and defaults."""
    import inspect
    import torchsde_b200 as tsde
    names = ['sdeint', 'sdeint_adjoint', 'BrownianInterval', 'BrownianPath', 'BrownianTree', 'ReverseBrownian',
             'brownian_interval_like', 'BaseBrownian', 'BaseSDE', 'SDEIto', 'SDEStratonovich']

    def signatures(mod):
        """{name: [(function name, [(parameter, kind, default), ...]) for the function or __init__ / __call__]}"""
        out = {}
        for name in names:
            obj = getattr(mod, name)
            fns = [obj]
            if inspect.isclass(obj):
                fns = [obj.__init__]
                if hasattr(obj, '__call__') and name != 'BaseSDE' and not name.startswith('SDE'):
                    fns.append(obj.__call__)
            out[name] = [(getattr(f, '__name__', ''), [(p.name, p.kind, p.default)
                                                       for p in inspect.signature(f).parameters.values()])
                         for f in fns]
        return out

    ours = _plain(signatures(tsde))
    ref = ref_outcome(request.node.name, lambda: signatures(torchsde))
    for name in names:
        assert len(ours[name]) == len(ref[name]), name
        for (_, po), (fname, pr) in zip(ours[name], ref[name]):
            assert po == pr, f"{name}.{fname}: {po} != {pr}"
    # read-only properties of a Brownian motion (brownian_interval.py:744-785)
    for prop in ('shape', 'dtype', 'device', 'entropy', 'levy_area_approximation', 'dt', 'tol', 'pool_size', 'cache_size',
                 'halfway_tree'):
        assert isinstance(getattr(tsde.BrownianInterval, prop), property), prop
    assert callable(tsde.BrownianInterval.size) and callable(tsde.BrownianInterval.display_binary_tree)


_DERIVED = {
    'path': ('BrownianPath', dict(t0=0.0, w0=torch.zeros(2, 3))),
    'path window': ('BrownianPath', dict(t0=0.5, w0=torch.zeros(2, 3, dtype=torch.float64), window_size=4)),
    'path bad t0': ('BrownianPath', dict(t0=torch.tensor([0.0, 1.0]), w0=torch.zeros(2, 3))),
    'path int w0': ('BrownianPath', dict(t0=0.0, w0=torch.zeros(2, 3, dtype=torch.int64))),
    'tree': ('BrownianTree', dict(t0=0.0, w0=torch.zeros(2, 3))),
    'tree t1 w1': ('BrownianTree', dict(t0=0.0, w0=torch.zeros(2, 3), t1=2.0, w1=torch.ones(2, 3))),
    'tree t1 before t0': ('BrownianTree', dict(t0=1.0, w0=torch.zeros(2, 3), t1=0.5)),
    'tree w1 shape': ('BrownianTree', dict(t0=0.0, w0=torch.zeros(2, 3), t1=1.0, w1=torch.ones(2, 4))),
    'tree options': ('BrownianTree', dict(t0=0.0, w0=torch.zeros(2, 3), entropy=3, tol=1e-4, pool_size=8, cache_depth=5,
                                          safety=0.1)),
    'like': ('brownian_interval_like', dict(y=torch.zeros(4, 5, dtype=torch.float64))),
    'like overrides': ('brownian_interval_like', dict(y=torch.zeros(4, 5), t0=0.5, t1=2.0, size=(4, 2),
                                                       levy_area_approximation='space-time')),
}


@pytest.mark.parametrize('label', sorted(_DERIVED))
def test_derived_brownians_construct_like_the_live_reference(request, label):
    """BrownianPath / BrownianTree / brownian_interval_like (derived.py:52-205): same acceptance, exception types and
    reported shape / dtype / Levy-area mode."""
    import warnings
    import torchsde_b200 as tsde
    name, kwargs = _DERIVED[label]

    def outcome(mod):
        try:
            with warnings.catch_warnings():
                warnings.simplefilter('ignore')
                bm = getattr(mod, name)(**kwargs)
        except Exception as e:  # noqa: BLE001
            return type(e).__name__
        return ('ok', tuple(bm.shape), bm.dtype, bm.levy_area_approximation)

    assert _plain(outcome(tsde)) == ref_outcome(request.node.name, lambda: outcome(torchsde)), label


@pytest.mark.parametrize('sde_type', ['ito', 'stratonovich'])
@pytest.mark.parametrize('kind', ['gbm', 'scalar', 'additive', 'general'])
def test_adjoint_sde_glue_equals_the_live_reference(request, kind, sde_type):
    """`_core/adjoint_sde.AdjointSDE` (the augmented backward SDE of the generic adjoint, adjoint_sde.py:23-377) is
    autograd glue around the user's f and g — pure torch ops, so it runs on the CPU: every product it hands to the
    solvers (drift, diffusion-vector product, both at once, Milstein's pair for diagonal noise) is compared with the
    reference's AdjointSDE on random augmented states, including the Ito corrections."""
    from torchsde_b200._core import base_sde as our_base
    from torchsde_b200._core.adjoint_sde import AdjointSDE as OurAdjointSDE
    rng = torch.Generator().manual_seed(11)
    B, d = 3, 4
    m = {'gbm': d, 'scalar': 1}.get(kind, 2)
    sde = problems.make(kind, d, m, sde_type, dtype=torch.float64, seed=2)
    params = [p for p in sde.parameters() if p.requires_grad]
    y = 0.1 + torch.rand(B, d, generator=rng, dtype=torch.float64)
    adj_y = torch.randn(B, d, generator=rng, dtype=torch.float64)
    aug = [y, adj_y] + [torch.randn(p.shape, generator=rng, dtype=torch.float64) for p in params]
    shapes = [t.size() for t in aug]
    flat = torch.cat([t.reshape(-1) for t in aug]).unsqueeze(0)
    t = torch.tensor(-0.3, dtype=torch.float64)
    bm_m = d if kind == 'gbm' else m
    v = torch.randn(B, bm_m, generator=rng, dtype=torch.float64)
    v2 = torch.randn(B, bm_m, generator=rng, dtype=torch.float64) if kind == 'gbm' else None

    def products(adjoint_sde):
        out = dict(noise_type=adjoint_sde.noise_type, sde_type=adjoint_sde.sde_type)
        with torch.no_grad():
            out['f'] = adjoint_sde.f(t, flat).numpy()
            out['g_prod'] = adjoint_sde.g_prod(t, flat, v).numpy()
            out['f_and_g_prod.f'], out['f_and_g_prod.g_prod'] = (x.numpy() for x in adjoint_sde.f_and_g_prod(t, flat, v))
            if kind == 'gbm':
                out['gdg.g_prod'], out['gdg.gdg_prod'] = (x.numpy() for x in
                                                          adjoint_sde.g_prod_and_gdg_prod(t, flat, v, v2))
        return out

    def reference():
        from torchsde._core import base_sde as ref_base
        from torchsde._core.adjoint_sde import AdjointSDE as RefAdjointSDE
        return products(RefAdjointSDE(ref_base.ForwardSDE(sde), params, shapes))

    ref = ref_arrays(request, reference)
    ours = products(OurAdjointSDE(our_base.ForwardSDE(sde), params, shapes))
    assert ours.pop('noise_type') == str(ref.pop('noise_type')) and ours.pop('sde_type') == str(ref.pop('sde_type'))
    assert sorted(ours) == sorted(ref)
    tol = dict(rtol=1e-12, atol=1e-13)
    for name in ours:
        np.testing.assert_allclose(ours[name], ref[name], err_msg=name, **tol)


class _WithPrior(torch.nn.Module):
    """f, g and a prior drift h — what `logqp=True` needs (sdeint.py:141-145)."""

    def __init__(self, base):
        super().__init__()
        self.base = base
        self.noise_type, self.sde_type = base.noise_type, base.sde_type

    def f(self, t, y):
        return self.base.f(t, y)

    def g(self, t, y):
        return self.base.g(t, y)

    def h(self, t, y):
        return -0.5 * y + torch.sin(t)


@pytest.mark.parametrize('kind', ['gbm', 'scalar', 'additive', 'general'])
def test_logqp_augmentation_equals_the_live_reference(request, kind):
    """SDELogqp (base_sde.py:240-306): drift / diffusion of the state augmented with the KL integrand, diagonal branch
    (stable division) and general branch (pseudo-inverse) — pure torch, compared on the CPU."""
    from torchsde_b200._core import base_sde as our_base
    d, m = 4, {'gbm': 4, 'scalar': 1}.get(kind, 3)
    sde = _WithPrior(problems.make(kind, d, m, 'ito', dtype=torch.float64, seed=4))
    gen = torch.Generator().manual_seed(3)
    y = torch.cat([0.2 + torch.rand(5, d, generator=gen, dtype=torch.float64), torch.zeros(5, 1, dtype=torch.float64)], dim=1)
    t = torch.tensor(0.4, dtype=torch.float64)

    def evaluate(base):
        aug = base.SDELogqp(sde)
        out = dict(noise_type=aug.noise_type, sde_type=aug.sde_type)
        with torch.no_grad():
            out['f'] = aug.f(t, y).numpy()
            out['g'] = aug.g(t, y).numpy()
            out['f_and_g.f'], out['f_and_g.g'] = (x.numpy() for x in aug.f_and_g(t, y))
        try:
            base.SDELogqp(problems.make(kind, d, m, 'ito'))
            out['without_h'] = 'accepted'
        except AttributeError:
            out['without_h'] = 'AttributeError'
        return out

    def reference():
        from torchsde._core import base_sde as ref_base
        return evaluate(ref_base)

    ref = ref_arrays(request, reference)
    ours = evaluate(our_base)
    assert str(ref['without_h']) == 'AttributeError'   # an SDE without `h` is rejected by both
    for key in ('noise_type', 'sde_type', 'without_h'):
        assert ours.pop(key) == str(ref.pop(key)), key
    assert sorted(ours) == sorted(ref)
    tol = dict(rtol=1e-12, atol=1e-13)
    for name in ours:
        np.testing.assert_allclose(ours[name], ref[name], err_msg=name, **tol)


from .test_host_dry_run import dry  # noqa: E402,F401  (fixture: recording stand-in for the C library)


class _Partial(torch.nn.Module):
    """General-noise SDE that exposes only a chosen subset of the five callables of the user-SDE protocol."""
    noise_type = 'general'

    def __init__(self, which, sde_type):
        super().__init__()
        self.sde_type = sde_type
        self.w = torch.nn.Parameter(torch.rand(3, 2, generator=torch.Generator().manual_seed(1)))
        self.offered = tuple(which)

    def __getattr__(self, name):
        if name in ('f', 'g', 'f_and_g', 'g_prod', 'f_and_g_prod'):
            if name in self.__dict__.get('offered', ()):
                return getattr(self, '_' + name)
            raise AttributeError(name)
        return super().__getattr__(name)

    def _f(self, t, y):
        return -y

    def _g(self, t, y):
        return torch.tanh(y).unsqueeze(-1) * self.w

    def _f_and_g(self, t, y):
        return self._f(t, y), self._g(t, y)

    def _g_prod(self, t, y, v):
        return (self._g(t, y) * v.unsqueeze(1)).sum(-1)

    def _f_and_g_prod(self, t, y, v):
        return self._f(t, y), self._g_prod(t, y, v)


_SUBSETS = [('f', 'g'), ('f_and_g',), ('f', 'g_prod'), ('f_and_g_prod',), ('f', 'g', 'g_prod'), ('f_and_g', 'f_and_g_prod'),
            ('g',), ('f',), ('g_prod',), ('f', 'g', 'f_and_g', 'g_prod', 'f_and_g_prod')]


@pytest.mark.parametrize('method,sde_type', [('euler', 'ito'), ('heun', 'stratonovich'), ('midpoint', 'stratonovich'),
                                             ('euler_heun', 'stratonovich'), ('reversible_heun', 'stratonovich')])
@pytest.mark.parametrize('which', _SUBSETS, ids=lambda w: '+'.join(w))
def test_partial_sde_protocols_behave_like_the_live_reference(request, dry, which, method, sde_type):  # noqa: F811
    """Which subsets of {f, g, f_and_g, g_prod, f_and_g_prod} suffice for which solver, and how a missing callable
    surfaces (ValueError from the contract check, or RuntimeError "Method `g` has not been provided…" at call time,
    base_sde.py:78-85): the product — dry-run on the CPU — must accept, reject and word it exactly like the reference."""
    import warnings
    import torchsde_b200 as tsde
    ts, dt = [0.0, 0.09375, 0.25], 0.0625

    def outcome(mod):
        sde = _Partial(which, sde_type)
        kw = {} if mod is torchsde else {'device': 'cpu'}
        try:
            with warnings.catch_warnings(), torch.no_grad():
                warnings.simplefilter('ignore')
                ys = mod.sdeint(sde, torch.ones(4, 3), ts, method=method, dt=dt,
                                bm=mod.BrownianInterval(0., .25, size=(4, 2), **kw))
            return ('ok', tuple(ys.shape))
        except (ValueError, RuntimeError) as e:
            return (type(e).__name__, str(e))

    ours, ref = _plain(outcome(tsde)), ref_outcome(request.node.name, lambda: outcome(torchsde))
    if method == 'euler_heun' and 'f_and_g_prod' in which and not {'g', 'g_prod'} & set(which):
        # One deliberate superset: Euler-Heun's second diffusion product g(t0, y').dW.  The reference asks `g_prod` for
        # it, whose default needs `g` (RuntimeError when the SDE offers neither); the product obtains it from the user's
        # `f_and_g_prod` — same value, so an SDE that only provides the fused callable still solves.
        assert ours[0] == 'ok' and ref[0] == 'RuntimeError'
        return
    assert ours[0] == ref[0], (which, method, ours, ref)
    if ours[0] == 'RuntimeError':
        assert ours[1] == ref[1]


@pytest.mark.parametrize('query', [(0.5, 0.2), (-1.0, 0.5), (0.5, 2.0), (-2.0, -1.0), (0.3, 0.3), (0.25, None), (0.0, 1.0),
                                   (torch.tensor(0.1), torch.tensor(0.6))], ids=str)
@pytest.mark.parametrize('levy', ['none', 'space-time', 'foster'])
def test_query_contract_equals_the_live_reference(request, dry, query, levy):  # noqa: F811
    """`BrownianInterval.__call__` (brownian_interval.py:589-687): reversed times raise RuntimeError, times outside
    [t0, t1] warn and are clamped, `tb=None` is a point query from t0, and the tuple returned for every
    (return_U, return_A) combination has the same arity and shapes.  (Values are a GPU matter; dry run here.)"""
    import warnings
    import torchsde_b200 as tsde
    ta, tb = query

    def outcome(mod):
        kw = {} if mod is torchsde else {'device': 'cpu'}
        bm = mod.BrownianInterval(0.0, 1.0, size=(3, 2), dtype=torch.float64, levy_area_approximation=levy, **kw)
        results = []
        for want_u in (False, True):
            for want_a in (False, True):
                if (want_u and levy == 'none') or (want_a and levy != 'foster'):
                    continue
                with warnings.catch_warnings(record=True) as caught:
                    warnings.simplefilter('always')
                    try:
                        out = bm(ta, tb, return_U=want_u, return_A=want_a)
                    except (RuntimeError, ValueError) as e:
                        results.append((want_u, want_a, type(e).__name__))
                        continue
                out = out if isinstance(out, tuple) else (out,)
                results.append((want_u, want_a, tuple(tuple(o.shape) for o in out),
                                sorted({w.category.__name__ for w in caught})))
        return results

    assert _plain(outcome(tsde)) == ref_outcome(request.node.name, lambda: outcome(torchsde))


def _warning_cases():
    yield 'unused kwarg', 'sdeint', dict(method='euler', foo=1)
    yield 'adaptive euler, non-additive noise', 'sdeint', dict(method='euler', adaptive=True)
    yield 'plain', 'sdeint', dict(method='euler')
    yield 'adjoint unused kwarg', 'sdeint_adjoint', dict(method='euler', bar=2)
    yield 'reversible forward, generic adjoint', 'sdeint_adjoint', dict(method='reversible_heun', adjoint_method='midpoint')
    yield 'reversible pair, ts off the step grid', 'sdeint_adjoint', dict(method='reversible_heun', ts=[0.0, 0.1, 0.25])
    yield 'reversible pair, aligned', 'sdeint_adjoint', dict(method='reversible_heun')
    yield 'reversible pair, adaptive', 'sdeint_adjoint', dict(method='reversible_heun', adaptive=True)


@pytest.mark.parametrize('label', [c[0] for c in _warning_cases()])
def test_warnings_equal_the_live_reference(request, dry, label):  # noqa: F811
    """User-facing warnings of sdeint / sdeint_adjoint (misc.py:26-31, sdeint.py:270-274, adjoint.py:240-256): same
    categories, same first sentence."""
    import warnings
    import torchsde_b200 as tsde
    _, fn, kwargs = next(c for c in _warning_cases() if c[0] == label)
    kwargs = dict(kwargs)
    ts = kwargs.pop('ts', [0.0, 0.125, 0.25])
    sde_type = 'stratonovich' if kwargs.get('method') == 'reversible_heun' else 'ito'

    def collect(mod):
        sde = problems.make('gbm', 3, 3, sde_type, dtype=torch.float32)
        kw = {} if mod is torchsde else {'device': 'cpu'}
        bm = mod.BrownianInterval(0.0, 0.25, size=(4, 3), dtype=torch.float32, **kw)
        with warnings.catch_warnings(record=True) as caught:
            warnings.simplefilter('always')
            try:
                getattr(mod, fn)(sde, torch.ones(4, 3), ts, bm=bm, dt=0.0625, **kwargs)
            except NotImplementedError:
                pass
        return sorted((w.category.__name__, str(w.message)[:40]) for w in caught
                      if 'torchsde' in str(w.filename) or 'sdeint' in str(w.message) or True)

    ours, ref = _plain(collect(tsde)), ref_outcome(request.node.name, lambda: collect(torchsde))
    assert [c for c, _ in ours] == [c for c, _ in ref], (ours, ref)
    assert ours == ref, (ours, ref)


class _LoggingBM:
    """Duck-typed Brownian motion (the reference accepts any object with this call signature, base_solver.py:54-57):
    returns zeros and logs how it was asked."""

    def __init__(self, shape, levy, dtype=torch.float32):
        self.shape, self.levy_area_approximation, self.dtype = shape, levy, dtype
        self.device = torch.device('cpu')
        self.log = []

    def __call__(self, ta, tb=None, return_U=False, return_A=False):
        self.log.append((round(float(ta), 9), None if tb is None else round(float(tb), 9), bool(return_U), bool(return_A)))
        W = torch.zeros(self.shape, dtype=self.dtype)
        out = [W]
        if return_U:
            out.append(torch.zeros_like(W))
        if return_A:
            out.append(torch.zeros(*self.shape, self.shape[-1], dtype=self.dtype))
        return out[0] if len(out) == 1 else tuple(out)


@pytest.mark.parametrize('kind,sde_type,method,levy', [
    ('gbm', 'ito', 'euler', 'none'), ('gbm', 'ito', 'milstein', 'none'), ('gbm', 'ito', 'srk', 'space-time'),
    ('additive', 'ito', 'srk', 'space-time'), ('general', 'stratonovich', 'heun', 'none'),
    ('scalar', 'stratonovich', 'midpoint', 'none'), ('gbm', 'stratonovich', 'euler_heun', 'none'),
    ('general', 'stratonovich', 'reversible_heun', 'none'), ('general', 'stratonovich', 'log_ode', 'foster')])
def test_brownian_queries_are_made_like_the_live_reference(request, dry, kind, sde_type, method, levy):  # noqa: F811
    """With a user-supplied (duck-typed) Brownian object the solver must ask for exactly the increments the reference
    asks for — same intervals, same order, once per step, same return_U / return_A flags — in the forward pass and in
    the backward pass of `sdeint_adjoint`."""
    import warnings
    import torchsde_b200 as tsde
    d, m = 3, {'gbm': 3, 'scalar': 1}.get(kind, 2)
    ts, dt = [0.0, 0.09375, 0.25], 0.0625

    def run(mod, adjoint):
        sde = problems.make(kind, d, m, sde_type, dtype=torch.float32)
        bm = _LoggingBM((4, m), levy)
        with warnings.catch_warnings():
            warnings.simplefilter('ignore')
            if adjoint:
                ys = mod.sdeint_adjoint(sde, torch.ones(4, d, requires_grad=True), ts, bm=bm, method=method, dt=dt)
                ys.sum().backward()
            else:
                with torch.no_grad():
                    mod.sdeint(sde, torch.ones(4, d), ts, bm=bm, method=method, dt=dt)
        return bm.log

    assert _plain(run(tsde, False)) == ref_outcome(request.node.name + '/forward', lambda: run(torchsde, False))
    if method not in ('srk', 'log_ode'):
        assert _plain(run(tsde, True)) == ref_outcome(request.node.name + '/adjoint', lambda: run(torchsde, True))


class _CallLogSDE(torch.nn.Module):
    """Time-dependent toy SDE that logs every evaluation the solver requests: (callable, time)."""

    def __init__(self, noise_type, sde_type, m):
        super().__init__()
        self.noise_type, self.sde_type, self.m = noise_type, sde_type, m
        self.p = torch.nn.Parameter(torch.ones(1))
        self.log = []

    def f(self, t, y):
        self.log.append(('f', round(float(t), 9)))
        return -y * self.p * torch.cos(t)

    def g(self, t, y):
        self.log.append(('g', round(float(t), 9)))
        base = 0.1 * y * self.p / (1 + t)
        if self.noise_type == 'diagonal':
            return base
        return base.unsqueeze(-1).expand(-1, -1, self.m).contiguous()


@pytest.mark.parametrize('noise,sde_type,method,levy', [
    ('diagonal', 'ito', 'euler', 'none'), ('diagonal', 'ito', 'milstein', 'none'),
    ('diagonal', 'stratonovich', 'milstein', 'none'), ('diagonal', 'ito', 'srk', 'space-time'),
    ('additive', 'ito', 'srk', 'space-time'), ('general', 'stratonovich', 'heun', 'none'),
    ('general', 'stratonovich', 'midpoint', 'none'), ('diagonal', 'stratonovich', 'euler_heun', 'none'),
    ('general', 'stratonovich', 'reversible_heun', 'none'), ('diagonal', 'stratonovich', 'reversible_heun', 'none')])
def test_user_callables_are_evaluated_like_the_live_reference(request, dry, noise, sde_type, method, levy):  # noqa: F811
    """The solver calls *up* into the user's f and g: for every tableau the sequence of (callable, stage time) is the
    reference's, call for call.  SRK is the one designed difference: the reference re-evaluates earlier stages inside
    its inner loop (10 f + 6 g per srid2 step, methods/srk.py:70-75), the product evaluates each distinct
    (callable, time, stage) once — fewer calls, the same set."""
    d, m = 3, (3 if noise == 'diagonal' else 2)
    ts, dt = [0.0, 0.09375, 0.25], 0.0625
    import torchsde_b200 as tsde

    def calls(mod):
        sde = _CallLogSDE(noise, sde_type, m)
        with torch.no_grad():
            mod.sdeint(sde, torch.ones(4, d), ts, bm=_LoggingBM((4, m), levy), method=method, dt=dt)
        return sde.log

    ours = calls(tsde)
    ref = [tuple(c) for c in ref_outcome(request.node.name, lambda: calls(torchsde))]
    if method == 'srk':
        assert set(ours) == set(ref) and len(ours) < len(ref)
    else:
        assert ours == ref


class _PlainSDE:
    """Not an nn.Module: parameters must be named explicitly for the adjoint (adjoint.py:228-231)."""
    noise_type, sde_type = 'diagonal', 'ito'

    def __init__(self):
        self.c = torch.ones(3, requires_grad=True)
        self.frozen = torch.ones(3)

    def f(self, t, y):
        return -self.c * y * self.frozen

    def g(self, t, y):
        return 0.1 * y


@pytest.mark.parametrize('label', ['missing', 'empty tuple', 'explicit', 'with a frozen tensor', 'module default'])
def test_adjoint_params_contract_equals_the_live_reference(request, dry, label):  # noqa: F811
    import warnings
    import torchsde_b200 as tsde

    def outcome(mod):
        plain = _PlainSDE()
        sde, kw = plain, {}
        if label == 'empty tuple':
            kw = dict(adjoint_params=())
        elif label == 'explicit':
            kw = dict(adjoint_params=(plain.c,))
        elif label == 'with a frozen tensor':
            kw = dict(adjoint_params=(plain.c, plain.frozen))
        elif label == 'module default':
            sde = problems.make('gbm', 3, 3, 'ito', dtype=torch.float32)
        y0 = torch.ones(4, 3, requires_grad=True)
        bkw = {} if mod is torchsde else {'device': 'cpu'}
        try:
            with warnings.catch_warnings():
                warnings.simplefilter('ignore')
                ys = mod.sdeint_adjoint(sde, y0, [0.0, 0.125, 0.25], method='euler', dt=0.0625,
                                        bm=mod.BrownianInterval(0., .25, size=(4, 3), **bkw), **kw)
                ys.sum().backward()
        except Exception as e:  # noqa: BLE001
            return type(e).__name__
        return ('ok', y0.grad is not None, plain.c.grad is not None, plain.frozen.grad is not None)

    assert _plain(outcome(tsde)) == ref_outcome(request.node.name, lambda: outcome(torchsde)), label


@pytest.mark.parametrize('cls,kwargs', [('BrownianPath', dict(t0=0.0, w0=torch.zeros(3, 2))),
                                        ('BrownianTree', dict(t0=0.0, w0=torch.zeros(3, 2), t1=1.0)),
                                        ('BrownianTree', dict(t0=0.0, w0=torch.zeros(3, 2), t1=1.0, w1=torch.ones(3, 2)))],
                         ids=['path', 'tree', 'tree with w1'])
@pytest.mark.parametrize('query', [(0.5, None), (0.25, 0.75), (0.0, None), (1.0, None), (0.75, 0.25), (1.5, None),
                                   (-0.5, None)], ids=str)
def test_derived_brownian_queries_equal_the_live_reference(request, dry, cls, kwargs, query):  # noqa: F811
    """BrownianPath / BrownianTree (derived.py:52-172): point queries return w0 + W(t0, t); interval queries the
    increment; same shapes, errors and warnings as the reference (values are a GPU matter)."""
    import warnings
    import torchsde_b200 as tsde
    ta, tb = query

    def outcome(mod):
        with warnings.catch_warnings(record=True) as caught:
            warnings.simplefilter('always')
            bm = getattr(mod, cls)(**kwargs)
            try:
                out = bm(ta) if tb is None else bm(ta, tb)
            except Exception as e:  # noqa: BLE001
                return type(e).__name__
        return (tuple(out.shape), out.dtype, sorted({w.category.__name__ for w in caught}))

    assert _plain(outcome(tsde)) == ref_outcome(request.node.name, lambda: outcome(torchsde))


def test_reverse_brownian_equals_the_live_reference(request, dry):  # noqa: F811
    """ReverseBrownian (derived.py:22-49): time reversal (ta, tb) -> base(-tb, -ta), attribute forwarding."""
    import torchsde_b200 as tsde

    def outcome(mod):
        kw = {} if mod is torchsde else {'device': 'cpu'}
        base = mod.BrownianInterval(0.0, 1.0, size=(3, 2), levy_area_approximation='space-time', **kw)
        rev = mod.ReverseBrownian(base)
        w, u = rev(-0.75, -0.25, return_U=True)
        return (tuple(w.shape), tuple(u.shape), tuple(rev.shape), rev.dtype, rev.levy_area_approximation,
                rev.base_brownian is base)

    assert _plain(outcome(tsde)) == ref_outcome(request.node.name, lambda: outcome(torchsde))
