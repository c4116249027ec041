"""-m gpu: every case of tests/kernel_ledger.py on the device -- the kernels it launched must be the ledger's, every
output within the elementwise fp64 bound, guard bands and inputs untouched, a second run bit-equal (float-atomic
outputs: 1e-6).  The cases of a switch set run in a process of their own (the library reads the switches once)."""
import json
import math
import os
import subprocess
import sys

import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
import kernel_ledger as KL  # noqa: E402

pytestmark = pytest.mark.gpu
_RESULTS = {}


def _results(name, tmp_dir):
    if name not in _RESULTS:
        if name == "default":
            _RESULTS[name] = KL.run_set("default")
        else:
            out = os.path.join(tmp_dir, f"ledger_{name}.json")
            env = dict(os.environ)
            env.update(KL.ENV_SETS[name])
            p = subprocess.run([sys.executable, os.path.join(HERE, "kernel_ledger.py"), "--set", name, "--out", out],
                               env=env, capture_output=True, text=True, timeout=1800)
            sys.stderr.write(p.stderr[-3000:])
            assert p.returncode == 0, f"switch set {name}: worker failed"
            with open(out) as f:
                _RESULTS[name] = json.load(f)
    return _RESULTS[name]


def _check(res):
    bad = {cid: r["failures"] for cid, r in res.items() if r["failures"]}
    assert not bad, "\n".join(f"{cid}: {f}" for cid, f in sorted(bad.items()))


def test_default_cases(tmp_path_factory):
    _check(_results("default", str(tmp_path_factory.mktemp("ledger"))))


@pytest.mark.parametrize("name", [n for n in KL.ENV_SETS if n != "default"])
def test_switch_set(name, tmp_path_factory):
    _check(_results(name, str(tmp_path_factory.mktemp("ledger"))))


def test_every_reachable_kernel_seen(tmp_path_factory):
    tmp = str(tmp_path_factory.mktemp("ledger"))
    res = {}
    for name in KL.ENV_SETS:
        res.update(_results(name, tmp))
    rows, unseen = [], []
    for k, e in sorted(KL.LEDGER.items()):
        if KL.entry_kind(e) == "unreachable":
            rows.append((k, "unreachable: " + e[1], "", ""))
            continue
        ran = [cid for cid in KL.entry_cases(e) if cid in res and k in res[cid]["kernels"]]
        if not ran:
            unseen.append(k)
            continue
        worst = max(ran, key=lambda c: res[c]["worst"])
        rows.append((k, worst, f"{res[worst]['worst']:.3f}", f"{max(res[c]['rel'] for c in ran):.2e}"))
    print(f"\n{'kernel':<62} {'case (worst)':<58} {'err/bound':>9} {'rel()':>9}")
    for r in rows:
        print(f"{r[0]:<62} {r[1]:<58} {r[2]:>9} {r[3]:>9}")
    assert not unseen, f"ledger entries no case launched: {unseen}"
    assert all(r["worst"] <= 1.0 and not math.isnan(r["worst"]) for r in res.values())
