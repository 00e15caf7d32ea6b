#!/usr/bin/env python
"""Mints tests/golden/dropin_script_calls.json: every call the UNMODIFIED reference script (noisynet.py) makes into
the drop-in modules, recorded while the script runs on top of them on a CPU-only host -- the fixture
tests/test_dropin_script.py replays (the reference tree is not part of this repository).  Run where a reference
tree exists (NOISYNET_REFERENCE, default /root/reference), after building the library:

    python oracle/gen_dropin_calls.py            # CPU, ~1 min

Recorded, in order: the `from hardware_model / quant / plot_histograms import ...` statements of the reference files,
the constructor calls of NoisyConv2d / NoisyLinear / QuantMeasure made from the reference, the attributes the reference
reads or assigns on those modules, and the first call into a drop-in forward together with the error it raises (the
library refuses CPU tensors: there is no CPU fallback).
"""
import json
import os
import subprocess
import sys
import tempfile
import textwrap

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = os.environ.get("NOISYNET_REFERENCE", "/root/reference")
OUT = os.path.join(ROOT, "tests", "golden", "dropin_script_calls.json")

ARGV = ["--current", "1", "--act_max", "5", "--w_max1", "0.3", "--LR", "0.005", "--L2_1", "0.0005", "--L2_2", "0.0002",
        "--q_a", "4", "--q_w", "4", "--batch_size", "16", "--nepochs", "1", "--no-augment"]

RUNNER = textwrap.dedent('''
    import builtins, collections.abc, json, os, runpy, sys, traceback, types
    import numpy as np, torch
    REF = os.path.realpath({ref!r})
    sys.path.insert(0, REF)
    sys.path.insert(0, {dropin!r})                     # OUR hardware_model / quant / plot_histograms first
    six = types.ModuleType('torch._six'); six.container_abcs = collections.abc
    sys.modules['torch._six'] = six                    # import rot of the reference under torch 2.x
    mpl = types.ModuleType('matplotlib'); mpl.use = lambda *a, **k: None
    plt = types.ModuleType('matplotlib.pyplot'); mpl.pyplot = plt
    sys.modules['matplotlib'] = mpl; sys.modules['matplotlib.pyplot'] = plt
    torch.Tensor.cuda = lambda self, *a, **k: self
    torch.nn.Module.cuda = lambda self, *a, **k: self
    import hardware_model, quant
    assert 'noisynet_b200' in hardware_model.NoisyConv2d.__module__, hardware_model.__file__
    assert 'noisynet_b200' in quant.QuantMeasure.__module__

    rec = dict(imports=[], constructors=[], attributes=[], first_call=None, error=None)

    def from_ref(depth):
        f = sys._getframe(depth + 1)
        return os.path.realpath(f.f_code.co_filename).startswith(REF + os.sep)

    def plain(v):
        if isinstance(v, (bool, int, float, str)) or v is None:
            return v
        if isinstance(v, (np.integer, np.floating, np.bool_)):
            return v.item()
        if isinstance(v, (list, tuple)):
            return [plain(x) for x in v]
        raise TypeError("unrecorded argument type %s" % type(v))

    _imp = builtins.__import__
    def imp(name, globals=None, locals=None, fromlist=(), level=0):
        src = (globals or {{}}).get('__file__') or ''
        if level == 0 and name in ('hardware_model', 'quant', 'plot_histograms') and \\
                os.path.realpath(src).startswith(REF + os.sep):
            e = [os.path.relpath(os.path.realpath(src), REF), name, list(fromlist or ())]
            if e not in rec['imports']:
                rec['imports'].append(e)
        return _imp(name, globals, locals, fromlist, level)
    builtins.__import__ = imp

    classes = [('hardware_model', hardware_model.NoisyConv2d), ('hardware_model', hardware_model.NoisyLinear),
               ('hardware_model', hardware_model.QuantMeasure), ('quant', quant.QuantMeasure)]
    instances = []
    for modname, cls in classes:
        def wrap(cls=cls, modname=modname):
            init, ga, sa, fwd = cls.__init__, cls.__getattribute__, cls.__setattr__, cls.forward
            def __init__(self, *a, **k):
                if from_ref(1):
                    object.__setattr__(self, '_rec_index', len(rec['constructors']))
                    rec['constructors'].append(dict(module=modname, cls=cls.__name__, args=plain(list(a)),
                                                    kwargs={{n: plain(v) for n, v in k.items()}}))
                init(self, *a, **k)
            def __getattribute__(self, name):
                if not name.startswith(('_rec', '__')) and from_ref(1):
                    i = object.__getattribute__(self, '__dict__').get('_rec_index')
                    if i is not None and [i, 'get', name] not in rec['attributes']:
                        rec['attributes'].append([i, 'get', name])
                return ga(self, name)
            def __setattr__(self, name, value):
                i = self.__dict__.get('_rec_index')
                if i is not None and from_ref(1) and [i, 'set', name] not in rec['attributes']:
                    rec['attributes'].append([i, 'set', name])
                sa(self, name, value)
            def forward(self, *a, **k):
                i = self.__dict__.get('_rec_index')
                if rec['first_call'] is None and i is not None:
                    rec['first_call'] = dict(instance=i, method='forward',
                                             shapes=[list(t.shape) for t in a if isinstance(t, torch.Tensor)])
                return fwd(self, *a, **k)
            cls.__init__, cls.__getattribute__, cls.__setattr__, cls.forward = __init__, __getattribute__, __setattr__, forward
        wrap()

    sys.argv = ['noisynet.py'] + {argv!r}
    try:
        runpy.run_path(os.path.join(REF, 'noisynet.py'), run_name='__main__')
    except Exception as e:
        frames = []
        for f in traceback.extract_tb(e.__traceback__):
            path = os.path.realpath(f.filename)
            if path.startswith(REF + os.sep):
                frames.append(['reference', os.path.relpath(path, REF), f.name])
            elif os.sep + 'noisynet_b200' + os.sep in path:
                frames.append(['noisynet_b200', path.split(os.sep + 'noisynet_b200' + os.sep)[-1], f.name])
        rec['error'] = dict(type=type(e).__name__, message=str(e), frames=frames)
    json.dump(rec, open('calls.json', 'w'), indent=1)
''')


def main():
    with tempfile.TemporaryDirectory() as tmp:
        os.makedirs(os.path.join(tmp, "data"))
        np.savez(os.path.join(tmp, "data", "cifar_RGB_4bit.npz"), np.zeros((50000, 3072), np.uint8),
                 np.zeros(50000, np.int64), np.zeros((10000, 3072), np.uint8), np.zeros(10000, np.int64))
        code = RUNNER.format(ref=REF, dropin=os.path.join(ROOT, "dropin"), argv=ARGV)
        env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
        r = subprocess.run([sys.executable, "-c", code], cwd=tmp, capture_output=True, text=True, timeout=600, env=env)
        path = os.path.join(tmp, "calls.json")
        if not os.path.isfile(path):
            sys.stderr.write(r.stdout[-2000:] + r.stderr[-4000:])
            raise SystemExit("reference run failed")
        rec = json.load(open(path))
    rec["argv"] = ARGV
    if rec["error"] is None or rec["first_call"] is None:
        raise SystemExit("the reference run did not reach a drop-in forward: %s" % json.dumps(rec)[:2000])
    with open(OUT, "w") as f:
        json.dump(rec, f, indent=1)
        f.write("\n")
    print("%d imports, %d constructors, %d attribute accesses; first call: %s; error: %s"
          % (len(rec["imports"]), len(rec["constructors"]), len(rec["attributes"]), rec["first_call"], rec["error"]["type"]))
    print("wrote", OUT)


if __name__ == "__main__":
    main()
