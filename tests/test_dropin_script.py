"""The reference script's calls into the drop-in modules, replayed.  `tests/golden/dropin_script_calls.json` records
(oracle/gen_dropin_calls.py) what the UNMODIFIED noisynet.py did when it ran on a CPU-only host on top of `dropin/`:
its `from hardware_model / quant / plot_histograms import ...` statements (noisynet.py:13-14, models/resnet.py:9-11,
models/mobilenet.py:9, main.py:37), every NoisyConv2d / NoisyLinear / QuantMeasure constructor call of `Net(args)`
(noisynet.py:344-359), the module attributes it read, and its first call into a drop-in forward, which stopped at the
loud no-CPU-fallback error.  The replay runs the same imports, constructors and attribute reads against the current
drop-in modules and checks that the first forward fails the same way, inside OUR module."""
import json
import os
import subprocess
import sys
import textwrap

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FIXTURE = os.path.join(ROOT, "tests", "golden", "dropin_script_calls.json")

RUNNER = textwrap.dedent('''
    import importlib, json, os, sys, traceback
    import torch
    DROPIN = {dropin!r}
    sys.path.insert(0, DROPIN)                         # what a user puts in front of the reference tree
    rec = json.load(open({fixture!r}))
    for src, name, fromlist in rec['imports']:
        m = importlib.import_module(name)
        assert os.path.dirname(os.path.realpath(m.__file__)) == os.path.realpath(DROPIN), (src, name, m.__file__)
        missing = [n for n in fromlist if not hasattr(m, n)]
        assert not missing, (src, name, missing)
    mods = []
    for c in rec['constructors']:
        cls = getattr(importlib.import_module(c['module']), c['cls'])
        assert cls.__module__.startswith('noisynet_b200.'), (c, cls.__module__)
        mods.append(cls(*c['args'], **c['kwargs']))
    for i, kind, name in rec['attributes']:
        assert hasattr(mods[i], name), (rec['constructors'][i]['cls'], name)
    fc = rec['first_call']
    assert fc['method'] == 'forward'
    try:
        mods[fc['instance']](*[torch.zeros(*s) for s in fc['shapes']])
        out = None
    except Exception as e:
        frames = []
        for f in traceback.extract_tb(e.__traceback__):
            path = os.path.realpath(f.filename)
            if os.sep + 'noisynet_b200' + os.sep in path:
                frames.append(['noisynet_b200', path.split(os.sep + 'noisynet_b200' + os.sep)[-1], f.name])
        out = dict(type=type(e).__name__, message=str(e), frames=frames)
    print(json.dumps(out))
''')


def test_recorded_script_calls_reach_our_kernels():
    rec = json.load(open(FIXTURE))
    # the recording covers the CIFAR script's whole model: four quantizers, two convolutions, two linear layers
    assert [c["cls"] for c in rec["constructors"]] == ["QuantMeasure"] * 4 + ["NoisyConv2d"] * 2 + ["NoisyLinear"] * 2
    assert {name for _, name, _ in rec["imports"]} == {"hardware_model", "quant", "plot_histograms"}
    code = RUNNER.format(dropin=os.path.join(ROOT, "dropin"), fixture=FIXTURE)
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-1500:] + r.stderr[-3000:]
    got = json.loads(r.stdout.strip().splitlines()[-1])
    want = rec["error"]
    assert got is not None, "the script's first drop-in forward ran on a CPU tensor without an error"
    assert got["type"] == want["type"] == "NoisyNetLibraryError", got
    assert "there is no CPU fallback" in got["message"] and got["message"] == want["message"], got
    # it failed inside OUR module's forward, at the same place as when the script itself called it
    ours = [f for f in want["frames"] if f[0] == "noisynet_b200"]
    assert ours and ours[0][1] == "hardware_model.py", want["frames"]
    assert got["frames"] == ours, (got["frames"], ours)
