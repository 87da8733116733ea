#!/usr/bin/env python3
"""Run the REFERENCE'S OWN unittest suite (/root/reference/test/*.py, 85 CLI-level tests, SURVEY.md section 4) against

    reference   the unmodified CLI on the reference's own C++                (baseline)
    patch       the unmodified CLI with porechop_b200.patch                  (python -m porechop_b200)
    flat        porechop_b200.flat_cli                                       (python -m porechop_b200.flat_cli)

and report, per mode, which tests pass.  The parity target is the BASELINE'S outcome set (three of the reference's tests
fail against the reference itself at this commit, SURVEY.md 0.10), not "all green".

    python tests/refsuite/run_reference_suite.py [--modes reference,patch,flat] [--engine oracle|sim|cuda] [-k substring] [--jobs N]

The suite is copied to a scratch directory (the reference tree is read-only and the tests write next to themselves);
`porechop-runner.py` there is tests/refsuite/runner.py.  Needs the reference checkout: authoring container only.
"""
import argparse
import json
import os
import re
import shutil
import subprocess
import sys
import tempfile

HERE = os.path.dirname(os.path.abspath(__file__))
REPO = os.path.dirname(os.path.dirname(HERE))


def run_mode(mode, engine, ref, pattern, jobs):
    with tempfile.TemporaryDirectory() as d:
        shutil.copytree(os.path.join(ref, 'test'), os.path.join(d, 'test'))
        shutil.copy(os.path.join(HERE, 'runner.py'), os.path.join(d, 'porechop-runner.py'))
        os.chmod(os.path.join(d, 'porechop-runner.py'), 0o755)
        env = dict(os.environ, PB200_SUITE_MODE=mode, PB200_SUITE_ENGINE=engine, PB200_SUITE_REPO=REPO, PB200_SUITE_REF=ref,
                   PYTHONPATH=ref + os.pathsep + os.environ.get('PYTHONPATH', ''), PYTHONWARNINGS='ignore')
        mods = sorted(f[:-3] for f in os.listdir(os.path.join(d, 'test')) if f.startswith('test_') and f.endswith('.py'))
        procs = []
        for m in mods:                       # one unittest process per test module, `jobs` at a time
            cmd = [sys.executable, '-m', 'unittest', '-v', 'test.' + m] + (['-k', pattern] if pattern else [])
            procs.append((m, cmd))
        results = {}
        running = []

        def reap(p_m):
            m, p = p_m
            _, err = p.communicate()
            current = None                   # unittest -v: "name (id)[\n docstring] ... ok|FAIL|ERROR|skipped"
            for line in err.decode(errors='replace').splitlines():
                mt = re.match(r'^(test_\w+) \((\S+?)\)', line)
                if mt:
                    current = mt.group(2).split('.', 1)[-1]          # module.Class.test_name
                me = re.search(r'\.\.\. (ok|FAIL|ERROR|skipped.*|expected failure)$', line)
                if me and current:
                    results[current] = me.group(1)
                    current = None
        for m, cmd in procs:
            running.append((m, subprocess.Popen(cmd, cwd=d, env=env, stdout=subprocess.PIPE, stderr=subprocess.PIPE)))
            if len(running) >= jobs:
                reap(running.pop(0))
        for r in running:
            reap(r)
        return results


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--modes', default='reference,patch,flat')
    ap.add_argument('--engine', default='oracle', choices=['oracle', 'sim', 'cuda'])
    ap.add_argument('--ref', default='', help='Porechop checkout (default: tests/helpers.py porechop_checkout())')
    ap.add_argument('-k', default='')
    ap.add_argument('--jobs', type=int, default=max(1, (os.cpu_count() or 2) // 2))
    ap.add_argument('--json', default='')
    a = ap.parse_args()
    if not a.ref:
        sys.path.insert(0, os.path.dirname(HERE))
        from helpers import porechop_checkout
        a.ref = porechop_checkout()
        if not a.ref:
            sys.exit('no Porechop checkout: pass --ref or set PORECHOP_CHECKOUT')
    out = {}
    for mode in a.modes.split(','):
        out[mode] = run_mode(mode, a.engine, a.ref, a.k, a.jobs)
        ok = sorted(k for k, v in out[mode].items() if v == 'ok')
        bad = sorted(k for k, v in out[mode].items() if v != 'ok')
        print('%-9s %d tests: %d ok, %d not ok' % (mode, len(out[mode]), len(ok), len(bad)))
        for k in bad:
            print('            not ok: %s (%s)' % (k, out[mode][k]))
    if 'reference' in out:
        base = out['reference']
        for mode in out:
            if mode != 'reference':
                diff = sorted(k for k in base if out[mode].get(k) != base[k])
                print('%-9s differs from the baseline on %d tests%s' % (mode, len(diff), (': ' + ', '.join(diff)) if diff else ''))
    if a.json:
        with open(a.json, 'w') as f:
            json.dump(out, f, indent=1, sort_keys=True)
    return 0


if __name__ == '__main__':
    sys.exit(main())
