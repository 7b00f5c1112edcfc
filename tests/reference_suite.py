#!/usr/bin/env python
"""Run the REFERENCE's own, unmodified test-suite against torchsde_b200 on a GPU (SURVEY §4 / §7 step 0).

    python tests/reference_suite.py [extra pytest args]        # on a CUDA box

`__graft_entry__.build()` stages the reference's tests/ under the git-ignored oracle/_ref/tests/reference_tests where
TSDE_REFERENCE_SRC names a reference source tree (oracle/stage_reference.py; they cannot be committed: reference
sources).  This runner puts an import alias `torchsde -> torchsde_b200`
(tests/as_torchsde) first on sys.path and runs them.  The reference parametrises most tests over ['cpu', 'cuda'];
this package has no CPU path by design, so the CPU parametrisations are deselected and only counted; tests without a
`device` parameter get the GPU as torch's default device (tests/as_torchsde/refsuite_plugin.py).  Output: the
pytest summary plus one JSON line {passed, failed, skipped, deselected_cpu, seconds}.
"""
import json
import os
import re
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle.stage_reference import TESTS as SUITE  # noqa: E402
ALIAS = os.path.join(ROOT, 'tests', 'as_torchsde')


def main():
    if not os.path.isdir(SUITE):
        print(json.dumps({"unavailable": "oracle/_ref/tests/reference_tests is absent (run build() with TSDE_REFERENCE_SRC "
                                         "naming a torchsde v0.2.6 source tree)"}))
        return 0
    env = dict(os.environ, PYTHONPATH=os.pathsep.join([ALIAS, ROOT]))
    # CPU parametrisations: ids contain 'cpu' or 'device0' (devices = [cpu, gpu] lists)
    deselect = 'not cpu and not device0'
    # the suite is host-bound (thousands of small eager solves at dt = 1e-3): spread it over worker processes sharing
    # the GPU (pytest-xdist; REFSUITE_WORKERS=0 runs it in-process)
    workers = os.environ.get('REFSUITE_WORKERS', '16')
    cmd = [sys.executable, '-m', 'pytest', SUITE, '-q', '-p', 'no:cacheprovider', '-p', 'refsuite_plugin', '--rootdir', SUITE,
           '-k', deselect,
           '-x' if '--x' in sys.argv else '--maxfail=100000'] + [a for a in sys.argv[1:] if a != '--x']
    if workers not in ('0', ''):
        cmd += ['-n', workers]
    t0 = time.time()
    out = subprocess.run(cmd, env=env, capture_output=True, text=True)
    text = out.stdout + out.stderr
    log = os.environ.get('REFSUITE_LOG')
    if log:
        open(log, 'w').write(text)
    print(text[-6000:])
    summary = {"seconds": round(time.time() - t0, 1), "returncode": out.returncode}
    for key in ('passed', 'failed', 'skipped', 'deselected', 'error', 'errors', 'warnings'):
        m = re.search(r'(\d+) ' + key, text.splitlines()[-1] if text.strip() else '')
        if m:
            summary[key] = int(m.group(1))
    failed = sorted(set(re.findall(r'^FAILED (\S+)', text, flags=re.M)))
    summary['failed_tests'] = failed[:60]
    print(json.dumps(summary))
    return 0


if __name__ == '__main__':
    sys.exit(main())
