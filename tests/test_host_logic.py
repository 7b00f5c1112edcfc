"""CPU-only tests: host logic of the package (no kernel is launched) and the C-ABI surface."""
import ctypes
import os
import re

import pytest
import torch

import torchsde_b200 as tsde
from torchsde_b200 import _cabi
from torchsde_b200._brownian import interval as bi
from torchsde_b200._core import schedule
from . import problems

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


# ---- C ABI ---------------------------------------------------------------------------------
def _declared_symbols():
    text = open(os.path.join(ROOT, 'include', 'torchsde_b200.h')).read()
    text = re.sub(r'/\*.*?\*/', '', text, flags=re.S)
    return sorted(set(re.findall(r'\b(tsde_[a-z0-9_]+)\s*\(', text)))


def test_cabi_loads_and_exports_every_declared_symbol():
    if not os.path.exists(_cabi.LIB_PATH):
        import __graft_entry__
        __graft_entry__.build()
    lib = ctypes.CDLL(_cabi.LIB_PATH)
    names = _declared_symbols()
    assert len(names) >= 28
    for n in names:
        assert hasattr(lib, n), f"{n} declared in include/torchsde_b200.h but not exported"
    # the ctypes binding covers every declared compute entry point, with matching arity
    assert set(_cabi.SIGNATURES) == set(names) - {'tsde_abi_version', 'tsde_error_string', 'tsde_kernel_launches'}
    assert _cabi.lib().tsde_abi_version() == 1


def test_struct_layout_matches_header():
    assert ctypes.sizeof(_cabi.Launch) == 40
    assert ctypes.sizeof(_cabi.Noise) == 80
    assert _cabi.Noise.cell_id.offset == 32 and _cabi.Noise.h.offset == 56


def test_no_cpu_fallback():
    sde = problems.GBMDiagonal(4, 'ito', dtype=torch.float32)
    y0 = torch.ones(3, 4)
    with pytest.raises(RuntimeError, match='CUDA'):
        tsde.sdeint(sde, y0, [0.0, 0.1], dt=0.05, method='euler',
                    bm=problems.ReplayBM([0.0], [0.05], [torch.zeros(3, 4)]))
    with pytest.raises(RuntimeError, match='CUDA'):
        tsde.BrownianInterval(0.0, 1.0, size=(2, 2))(0.0, 0.5)


def test_product_does_not_import_oracle():
    import subprocess, sys
    code = "import sys, torchsde_b200; assert not any(m == 'oracle' or m.startswith('oracle.') for m in sys.modules)"
    subprocess.run([sys.executable, '-c', code], check=True, cwd=ROOT)
    for dirpath, _, files in os.walk(os.path.join(ROOT, 'torchsde_b200')):
        for f in files:
            if f.endswith('.py'):
                assert 'oracle' not in open(os.path.join(dirpath, f)).read().replace('oracle/', '')


# ---- schedule (base_solver.py:107-147) ----------------------------------------------------------
def _reference_grid(ts, dt):
    """The reference's loop on 0-d tensors, verbatim control flow."""
    curr_t = ts[0]
    steps, outs = [], []
    prev_t = curr_t
    for out_t in ts[1:]:
        while curr_t < out_t:
            next_t = min(curr_t + dt, ts[-1])
            prev_t = curr_t
            steps.append((float(curr_t), float(next_t)))
            curr_t = next_t
        outs.append((len(steps) - 1, float(prev_t), float(curr_t), float(out_t)))
    return steps, outs


@pytest.mark.parametrize('dtype', [torch.float32, torch.float64])
@pytest.mark.parametrize('ts,dt', [([0.0, 1.0], 1e-3), ([0.0, 0.075, 0.15, 0.225, 0.3], 0.05),
                                   ([0.0, 0.25, 1.0], 2.0 ** -4), ([0.0, 0.01, 0.02], 0.05), ([1.0, 2.5], 0.7)])
def test_schedule_matches_reference_loop(dtype, ts, dt):
    t = torch.tensor(ts, dtype=dtype)
    s = schedule.build_schedule(t, dt)
    steps, outs = _reference_grid(t, dt)
    assert [(float(a), float(b)) for a, b in s.steps] == steps
    assert s.bounds == [steps[0][0]] + [b for _, b in steps]
    for o, (k, prev_t, curr_t, out_t) in zip(s.outputs, outs):
        assert o.step == k and o.aligned == (curr_t == out_t)
    if dtype == torch.float32 and ts == [0.0, 1.0]:
        assert s.n_steps == 1001  # fp32 accumulation leaves a sliver step (SURVEY §7.0)


def test_schedule_rejects_stalled_time():
    with pytest.raises(ValueError):
        schedule.build_schedule(torch.tensor([1e8, 1e8 + 16], dtype=torch.float32), 1e-3)


# ---- contract errors (sdeint.py:115-281, base_solver.py:49-58, test_sdeint.py:124-136) ---------
def _bm(levy, m=3):
    return tsde.BrownianInterval(0.0, 0.3, size=(4, m), dtype=torch.float64, device='cuda',
                                 levy_area_approximation=levy)


@pytest.mark.parametrize('sde_type', ['ito', 'stratonovich'])
@pytest.mark.parametrize('method', ['blah', 'euler', 'milstein', 'srk', 'euler_heun', 'heun', 'midpoint', 'log_ode',
                                    'reversible_heun'])
@pytest.mark.parametrize('kind', ['gbm', 'scalar', 'additive', 'general'])
@pytest.mark.parametrize('levy', [None, 'none', 'space-time', 'davie', 'foster'])
def test_error_matrix(sde_type, method, kind, levy):
    """Which (sde_type, noise_type, method, levy) combinations must raise ValueError; evaluated on
    CPU tensors: a legal combination gets past all checks and then stops at the CUDA requirement."""
    d, m = 3, {'gbm': 3, 'scalar': 1}.get(kind, 2)
    sde = problems.make(kind, d, m, sde_type, dtype=torch.float64)
    should_fail = False
    if sde_type == 'ito':
        should_fail |= method not in ('euler', 'srk', 'milstein')
    else:
        should_fail |= method not in ('euler_heun', 'heun', 'midpoint', 'log_ode', 'milstein', 'reversible_heun')
    if method in ('milstein', 'srk') and kind == 'general':
        should_fail = True
    if method == 'srk' and levy == 'none':
        should_fail = True
    if method == 'log_ode' and levy in ('none', 'space-time'):
        should_fail = True
    y0 = torch.ones(4, d, dtype=torch.float64)
    bm = None if levy is None else _bm(levy, m)
    if should_fail:
        with pytest.raises(ValueError):
            tsde.sdeint(sde, y0, [0.0, 0.3], bm=bm, method=method, dt=0.05)
    else:
        with pytest.raises((RuntimeError, NotImplementedError), match='CUDA|not implemented'):
            tsde.sdeint(sde, y0, [0.0, 0.3], bm=bm, method=method, dt=0.05)


def test_contract_messages():
    sde = problems.GBMDiagonal(3, 'ito')
    y0 = torch.ones(4, 3, dtype=torch.float64)
    with pytest.raises(ValueError, match='2-dimensional'):
        tsde.sdeint(sde, y0[0], [0.0, 1.0])
    with pytest.raises(ValueError, match='strictly increasing'):
        tsde.sdeint(sde, y0, [0.0, 0.0])
    with pytest.raises(ValueError, match='torch.Tensor'):
        tsde.sdeint(sde, [1.0], [0.0, 1.0])
    with pytest.raises(ValueError, match='Batch sizes'):
        tsde.sdeint(sde, y0, [0.0, 1.0], bm=tsde.BrownianInterval(0., 1., size=(5, 3), device='cuda'))
    with pytest.raises(ValueError, match='must not require gradient'):
        tsde.sdeint(sde, y0, torch.tensor([0.0, 1.0], dtype=torch.float64, requires_grad=True))
    with pytest.warns(UserWarning, match='Unexpected arguments'):
        with pytest.raises(RuntimeError):
            tsde.sdeint(sde, y0, [0.0, 1.0], method='euler', bogus=1)

    class NoNoise(torch.nn.Module):
        sde_type = 'ito'
    with pytest.raises(ValueError, match='noise_type'):
        tsde.sdeint(NoNoise(), y0, [0.0, 1.0])
    with pytest.raises(ValueError, match='adjoint parameters'):
        tsde.sdeint_adjoint(object(), y0, [0.0, 1.0])
    with pytest.raises(ValueError, match='only be used for adjoint_method'):
        tsde.sdeint(problems.GBMDiagonal(3, 'stratonovich'), y0, [0.0, 1.0], method='adjoint_reversible_heun')


# ---- interval tree (pure host logic) ----------------------------------------------------------
def _pieces(bm, ta, tb):
    out = []
    for p in bm._locate(ta, tb):
        if isinstance(p, bi._Node):
            out.append((p.start, p.end))
        else:
            g, i, j = p
            out.append((g.bounds[i], g.bounds[j], j - i))
    return out


def test_locate_binary_tree_like_reference():
    bm = tsde.BrownianInterval(0.0, 1.0, size=(2, 2), device='cuda')
    assert _pieces(bm, 0.0, 1.0) == [(0.0, 1.0)]
    assert _pieces(bm, 0.3, 0.6) == [(0.3, 0.6)]
    # root split at 0.3, right child split at 0.6
    assert bm._root.mid == 0.3 and bm._root.right.mid == 0.6
    assert _pieces(bm, 0.1, 0.8) == [(0.1, 0.3), (0.3, 0.6), (0.6, 0.8)]
    assert _pieces(bm, 0.0, 0.3) == [(0.0, 0.3)]      # an existing node answers as a whole
    assert _pieces(bm, 0.0, 0.2) == [(0.0, 0.1), (0.1, 0.2)]
    ids = set()
    stack = [bm._root]
    while stack:
        n = stack.pop()
        ids.add(n.id)
        if n.kind == bi._BINARY:
            stack += [n.left, n.right]
    assert len(ids) == 11  # all node ids distinct


def test_locate_grid_cells():
    bm = tsde.BrownianInterval(0.0, 1.0, size=(2, 2), device='cuda', dt=0.125)
    bm._bind_uniform(0.125)
    assert bm._root.kind == bi._GRID and len(bm._root.bounds) == 9
    assert _pieces(bm, 0.25, 0.75) == [(0.25, 0.75, 4)]
    assert _pieces(bm, 0.0, 1.0) == [(0.0, 1.0)]
    assert _pieces(bm, 0.125, 0.25) == [(0.125, 0.25, 1)]
    assert _pieces(bm, 0.3, 0.6) == [(0.3, 0.375), (0.375, 0.5, 1), (0.5, 0.6)]
    assert _pieces(bm, 0.26, 0.3) == [(0.26, 0.3)]
    assert _pieces(bm, 0.25, 0.3) == [(0.25, 0.3)]
    assert _pieces(bm, 0.25, 0.28) == [(0.25, 0.26), (0.26, 0.28)]
    assert _pieces(bm, 0.3, 0.5) == [(0.3, 0.375), (0.375, 0.5, 1)]


def test_bind_grid_rules():
    mk = lambda **kw: tsde.BrownianInterval(0.0, 1.0, size=(2, 2), device='cuda', **kw)  # noqa
    bounds = [0.0, 0.25, 0.5, 1.0]
    b = mk().bind_grid(bounds)
    assert b is not None and b.first == [0, 1, 2] and b.count == [1, 1, 1]
    bm = mk()
    assert bm.bind_grid([k / 8 for k in range(9)]) is not None
    nested = bm.bind_grid([0.0, 0.5, 0.625, 1.0])           # coarser, nested: runs of cells
    assert nested.first == [0, 4, 5] and nested.count == [4, 1, 3]
    assert bm.bind_grid([0.0, 0.3, 1.0]) is None            # not nested -> ordinary queries
    sub = bm.bind_grid([0.25, 0.5])                          # sub-range of an existing grid
    assert sub.first == [2] and sub.count == [2]
    assert mk(halfway_tree=True, tol=1e-6).bind_grid(bounds) is None
    assert tsde.BrownianInterval(0.0, 1.0, W=torch.zeros(2, 2)).bind_grid(bounds) is None
    rev = b.reversed()
    nz = _cabi.Noise()
    rev.fill(nz, 0, False, 0)
    assert nz.cell_id == (b.node.cell_base + 2) & ((1 << 64) - 1) and nz.h == 0.5
    assert bi.key_from_entropy(5) != bi.key_from_entropy(6) and bi.key_from_entropy(2 ** 70 + 5) != bi.key_from_entropy(5)


def test_halfway_tree_structure_is_query_order_independent():
    a = tsde.BrownianInterval(0.0, 1.0, size=(2,), device='cuda', halfway_tree=True, tol=1e-3)
    b = tsde.BrownianInterval(0.0, 1.0, size=(2,), device='cuda', halfway_tree=True, tol=1e-3)
    qs = [(0.125, 0.5), (0.3, 0.7), (0.0, 0.06)]
    pa = [[(p.start, p.end, p.id) for p in a._locate(a._round(x), a._round(y))] for x, y in qs]
    pb = [[(p.start, p.end, p.id) for p in b._locate(b._round(x), b._round(y))] for x, y in reversed(qs)][::-1]
    assert pa == pb


def test_bench_reference_arm_prints_one_contract_line():
    """`bench.py --impl reference` (the CPU arm the driver runs next to ours): one JSON line with the contract's keys."""
    import json
    import subprocess
    import sys
    env = dict(os.environ, TSDE_BENCH_B='2048', TSDE_BENCH_REF_BUDGET_S='2')
    out = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--impl', 'reference', '--steps', '1',
                          '--warmup', '0'], check=True, cwd=ROOT, env=env, capture_output=True, text=True).stdout
    lines = [ln for ln in out.splitlines() if ln.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d['impl'] == 'reference' and d['unit'] == 'traj-steps/s' and d['higher_is_better'] is True
    for key in ('metric', 'value', 'n_gpus', 'steps', 'warmup', 'ms_per_step', 'scaling', 'dtype', 'data', 'config'):
        assert key in d, key
    assert d['value'] > 0 and d['e2e']['value'] == d['value'] and d['e2e']['h2d_bytes_per_step'] == 0
    cb = d['cpu_baseline']
    # the reference itself where build() has staged it under oracle/_ref (git-ignored, travels with a copy of the
    # working tree); the numpy port only where that directory is absent
    staged = os.path.isdir(os.path.join(ROOT, 'oracle', '_ref', 'pkg', 'torchsde'))
    assert cb['kind'] == ('reference' if staged else 'port') and cb['cores'] >= 1
    assert d['config']['workload'] == 'cfg2' and d['config']['method'] == 'milstein' 


def test_header_is_plain_c():
    """The drop-in boundary is a C ABI: the header must compile as C (no C++, no torch types), warning-free."""
    import shutil
    import subprocess
    gcc = shutil.which('gcc')
    if gcc is None:
        pytest.skip("no gcc")
    hdr = os.path.join(ROOT, 'include', 'torchsde_b200.h')
    r = subprocess.run([gcc, '-std=c99', '-fsyntax-only', '-Wall', '-Wextra', '-Werror', '-x', 'c', hdr],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr


def test_schedule_cache_is_keyed_by_the_value_of_dt():
    """A fresh dt tensor per call may reuse the id of a dead one: the cached time grid must follow dt's value."""
    import gc
    from torchsde_b200._core import schedule
    ts = torch.tensor([0.0, 1.0])
    reused = False
    for _ in range(50):
        dt1 = torch.tensor(0.1)
        ident = id(dt1)
        assert schedule.get_schedule(ts, dt1).n_steps == 10
        del dt1
        gc.collect()
        dt2 = torch.tensor(0.05)
        reused = reused or id(dt2) == ident
        assert schedule.get_schedule(ts, dt2).n_steps == 20
        assert schedule.get_schedule(ts, 0.25).n_steps == 4
        if reused:
            break
    # same value, different dtype of dt: the grid is accumulated in the promoted dtype -> separate entries
    a = schedule.get_schedule(ts, torch.tensor(0.1, dtype=torch.float32))
    b = schedule.get_schedule(ts, torch.tensor(0.1, dtype=torch.float64))
    assert a is not b


def test_graph_plan_key_follows_the_sde_tensors():
    """A captured graph bakes in the addresses of the SDE's parameters: the plan key must change when they are
    replaced (`.double()`, re-assignment) and stay put under in-place updates (optimiser steps)."""
    from torchsde_b200._core.graph import _tensor_signature
    sde = problems.GBMDiagonal(4, 'ito', dtype=torch.float32)
    s0 = _tensor_signature(sde)
    assert len(s0) == len(list(sde.parameters())) > 0
    with torch.no_grad():
        for p in sde.parameters():
            p.add_(0.5)                                   # what an optimiser step does
    sde.load_state_dict(sde.state_dict())
    assert _tensor_signature(sde) == s0
    sde.mu = torch.nn.Parameter(sde.mu.detach().clone())  # new storage
    assert _tensor_signature(sde) != s0
    assert _tensor_signature(sde.double()) != s0

    class Plain:                                          # SDEs need not be nn.Modules (sdeint.py:124-243)
        noise_type, sde_type = 'diagonal', 'ito'

        def __init__(self):
            self.c = torch.ones(3)
            self.name = 'x'
    obj = Plain()
    s1 = _tensor_signature(obj)
    assert len(s1) == 1
    obj.c = torch.ones(3)
    assert _tensor_signature(obj) != s1 or obj.c.data_ptr() == s1[0][0]
    assert _tensor_signature(object()) == ()


def test_plan_cache_tolerates_unhashable_sde_objects():
    import weakref
    from torchsde_b200._core.graph import plans_of

    class Slotted:
        __slots__ = ('x',)

    class NoHash:
        def __eq__(self, other):
            return True

    cache = weakref.WeakKeyDictionary()
    assert plans_of(cache, Slotted()) is None and plans_of(cache, NoHash()) is None
    mod = problems.GBMDiagonal(2, 'ito')
    d = plans_of(cache, mod)
    assert d == {} and plans_of(cache, mod) is d


def test_cabi_rejects_malformed_calls_without_touching_the_device():
    """Contract violations are TSDE_EINVAL from every compute entry point — a null launch descriptor, a valid one with
    null operands, negative sizes — checked before any CUDA call (so this runs on a machine without a GPU, in a child
    process because a regression here is a segfault).  An empty launch is a no-op (0)."""
    import subprocess
    import sys
    import textwrap
    code = textwrap.dedent('''
        import ctypes, sys
        sys.path.insert(0, %r)
        import torch
        from torchsde_b200 import _cabi
        lib = _cabi.lib()
        EINVAL = -22

        def args_for(name, launch):
            out = []
            for t in _cabi.SIGNATURES[name]:
                if t is _cabi._D:
                    out.append(0.0)
                elif t is _cabi._L:
                    out.append(launch)
                elif t in (_cabi._I, ctypes.c_int64, ctypes.c_uint64):
                    out.append(0)
                else:
                    out.append(None)
            return out

        ok = _cabi.make_launch(torch.float32, _cabi.NOISE_DIAGONAL, 4, 8, 8, 0)
        negative = _cabi.make_launch(torch.float32, _cabi.NOISE_DIAGONAL, -1, 8, 8, 0)
        no_width = _cabi.make_launch(torch.float64, _cabi.NOISE_GENERAL, 4, 8, 0, 0)
        for name in _cabi.SIGNATURES:
            for launch in (None, ctypes.byref(ok), ctypes.byref(negative), ctypes.byref(no_width)):
                rc = getattr(lib, name)(*args_for(name, launch))
                assert rc == EINVAL, (name, rc)
        # an empty launch (rows == 0) is a valid no-op for every entry point, whatever its operands: the tensors of an
        # empty batch have no storage, their data pointers are null
        for dtype, noise_type, m in ((torch.float32, _cabi.NOISE_DIAGONAL, 8), (torch.float64, _cabi.NOISE_GENERAL, 4)):
            empty = _cabi.make_launch(dtype, noise_type, 0, 8, m, 0)
            for name in _cabi.SIGNATURES:
                rc = getattr(lib, name)(*args_for(name, ctypes.byref(empty)))
                # (entry points that exist for one noise layout only still reject the other one)
                assert rc in (0, EINVAL), (name, rc)
                if rc == EINVAL:
                    other = _cabi.make_launch(dtype, 1 - noise_type, 0, 8, 8 if noise_type else 4, 0)
                    assert getattr(lib, name)(*args_for(name, ctypes.byref(other))) == 0, name
        empty = _cabi.make_launch(torch.float32, _cabi.NOISE_DIAGONAL, 0, 8, 8, 0)
        buf = (ctypes.c_float * 64)()
        p = ctypes.addressof(buf)
        nz = _cabi.Noise()
        nz.source, nz.w = _cabi.SRC_MEMORY, p
        assert lib.tsde_step_euler(ctypes.byref(empty), ctypes.byref(nz), p, p, p, 0.1, p) == 0
        assert lib.tsde_linear_interp(ctypes.byref(empty), p, p, 0.5, 0.5, p) == 0
        # wrong dtype code, diagonal noise with m != d, Milstein on general noise
        bad_dtype = _cabi.make_launch(torch.float32, _cabi.NOISE_DIAGONAL, 4, 8, 8, 0)
        bad_dtype.dtype = 7
        assert lib.tsde_step_euler(ctypes.byref(bad_dtype), ctypes.byref(nz), p, p, p, 0.1, p) == EINVAL
        skew = _cabi.make_launch(torch.float32, _cabi.NOISE_DIAGONAL, 4, 8, 4, 0)
        assert lib.tsde_step_euler(ctypes.byref(skew), ctypes.byref(nz), p, p, p, 0.1, p) == EINVAL
        general = _cabi.make_launch(torch.float32, _cabi.NOISE_GENERAL, 4, 8, 4, 0)
        assert lib.tsde_milstein_vjp_seed(ctypes.byref(general), ctypes.byref(nz), p, 0.1, 1, p) == EINVAL
        # noise descriptor: unknown source code, counter source without a key, (W, U) requested from memory without U
        for noise_type, m in ((_cabi.NOISE_DIAGONAL, 8), (_cabi.NOISE_GENERAL, 4)):
            launch = _cabi.make_launch(torch.float32, noise_type, 4, 8, m, 0)
            bad = _cabi.Noise()
            bad.source, bad.w = 99, p
            assert lib.tsde_step_euler(ctypes.byref(launch), ctypes.byref(bad), p, p, p, 0.1, p) == EINVAL
            bad.source, bad.key = _cabi.SRC_COUNTER, None
            assert lib.tsde_step_euler(ctypes.byref(launch), ctypes.byref(bad), p, p, p, 0.1, p) == EINVAL
        need_u = _cabi.Noise()
        need_u.source, need_u.w, need_u.want_u, need_u.u = _cabi.SRC_MEMORY, p, 1, None
        assert lib.tsde_step_srk_diag(ctypes.byref(ok), ctypes.byref(need_u), p, p, p, p, p, p, p, p, 0.1, 10.0, 0.3, 0.3,
                                      p) == EINVAL
        # launch flags: unknown bits; a batch-broadcast g on a row-wise (diagonal / m == 1) launch or on the
        # reversible-Heun pair, whose g operands are saved and differentiated
        flagged = _cabi.Noise()
        flagged.source, flagged.w, flagged.flags = _cabi.SRC_MEMORY, p, 2
        assert lib.tsde_step_euler(ctypes.byref(general), ctypes.byref(flagged), p, p, p, 0.1, p) == EINVAL
        flagged.flags = _cabi.FLAG_G_BROADCAST
        assert lib.tsde_step_euler(ctypes.byref(ok), ctypes.byref(flagged), p, p, p, 0.1, p) == EINVAL
        scalar = _cabi.make_launch(torch.float32, _cabi.NOISE_GENERAL, 4, 8, 1, 0)
        assert lib.tsde_step_euler(ctypes.byref(scalar), ctypes.byref(flagged), p, p, p, 0.1, p) == EINVAL
        assert lib.tsde_reversible_heun_z(ctypes.byref(general), ctypes.byref(flagged), p, p, p, p, 0.1, p) == EINVAL
        assert b'invalid argument' in lib.tsde_error_string(EINVAL)
        print('validated', len(_cabi.SIGNATURES))
    ''' % ROOT)
    r = subprocess.run([sys.executable, '-c', code], capture_output=True, text=True)
    assert r.returncode == 0 and f'validated {len(_cabi.SIGNATURES)}' in r.stdout, (r.returncode, r.stdout[-300:], r.stderr[-600:])


def test_c_client_of_the_abi(tmp_path):
    """The boundary is usable from plain C: tests/c/abi_client.c includes the public header, dlopens the library and
    checks version, struct sizes, diagnostics and argument validation (everything that needs no GPU)."""
    import shutil
    import subprocess
    gcc = shutil.which('gcc')
    if gcc is None:
        pytest.skip("no gcc")
    _cabi.lib()  # make sure the library is built
    exe = str(tmp_path / 'abi_client')
    subprocess.run([gcc, '-std=c99', '-Wall', '-Wextra', '-Werror', '-I', os.path.join(ROOT, 'include'),
                    os.path.join(ROOT, 'tests', 'c', 'abi_client.c'), '-o', exe, '-ldl'], check=True)
    r = subprocess.run([exe, _cabi.LIB_PATH], capture_output=True, text=True)
    assert r.returncode == 0 and 'c client ok, abi 1' in r.stdout, (r.returncode, r.stdout, r.stderr)


def test_bench_clock_sampler_reports_the_timed_window_only():
    """bench.py starts `nvidia-smi -lms` before the warm-up (so that its start-up does not run against the first timed
    steps) and reports only samples taken after `mark()`; throttle reasons outside the window do not count, an empty
    window falls back to the last sample."""
    import importlib.util
    import time
    spec = importlib.util.spec_from_file_location('bench_under_test', os.path.join(ROOT, 'bench.py'))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)

    class _Done:
        def terminate(self):
            pass

        def wait(self, timeout=None):
            return 0

    s = bench.ClockSampler(0)
    s.proc = _Done()
    t = time.monotonic()
    warm = '1500, 1965, Not Active, Not Active, Active, Not Active'   # sw_thermal_slowdown during the warm-up only
    timed = '1965, 1965, Not Active, Not Active, Not Active, Active'  # sw_power_cap inside the window: kept and noted
    s.lines = [(t - 2.0, warm), (t - 1.0, warm)]
    s.t_mark = t
    s.lines += [(t + 0.1, timed), (t + 0.3, timed)]
    got = s.stop()
    assert got == {'sm_mhz': 1965.0, 'sm_max_mhz': 1965.0, 'samples': 2, 'reasons': ['sw_power_cap']}
    empty = bench.ClockSampler(0)
    empty.proc = _Done()
    empty.lines = [(t - 2.0, warm)]
    empty.t_mark = t
    assert empty.stop()['samples'] == 1 and empty.stop()['sm_mhz'] == 1500.0
