"""Developer tool: run the `-m gpu` tests on a machine WITHOUT a GPU, with the C-ABI library replaced by the
prototype-checking recorder of tests/test_abi_calls_cpu.py (no compute) and CUDA touch points stubbed.  Python-level errors in the tests
or in the host code they drive (wrong keyword, missing attribute, bad shape) show up as non-assertion exceptions BEFORE a GPU call is
spent on them; numeric assertions are expected to stop a test (nothing is computed), tensor comparisons are neutralised to get further.
Usage: python tools/gated_tests_dryrun.py [--all]   ->  "python errors: 0" is the goal (--all: the validated tests too;
tests/test_gpu_tests_dryrun_cpu.py runs that as part of the CPU suite)."""
import os, sys, traceback, inspect, itertools
os.environ['B200RL_UNVALIDATED'] = '1'
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, 'tests'))
import torch
import test_agent_host_cpu as H
from test_abi_calls_cpu import _Recorder
from rl_games_b200 import ops, _lib
rec = _Recorder(_lib.lib); ops.lib = rec
real_device = torch.device
class _Meta(type):
    def __instancecheck__(cls, obj): return isinstance(obj, real_device)
class _Dev(metaclass=_Meta):
    def __new__(cls, *a, **k):
        if a and isinstance(a[0], str) and a[0].startswith('cuda'): return real_device('cpu')
        return real_device(*a, **k)
torch.device = _Dev
def on_cpu(fn):
    def w(*a, **k):
        if isinstance(k.get('device'), str) and k['device'].startswith('cuda'): k['device'] = 'cpu'
        return fn(*a, **k)
    return w
for n in ('empty','zeros','ones','full','tensor','arange','randn','rand','empty_like','zeros_like','full_like'):
    setattr(torch, n, on_cpu(getattr(torch, n)))
_to = torch.Tensor.to
def to(self, *a, **k):
    a = tuple('cpu' if isinstance(x, str) and x.startswith('cuda') else x for x in a)
    if isinstance(k.get('device'), str) and k['device'].startswith('cuda'): k['device'] = 'cpu'
    return _to(self, *a, **k)
torch.Tensor.to = to
torch.cuda.is_available = lambda: True
torch.cuda.set_device = lambda d: None
torch.cuda.synchronize = lambda *a: None
torch.cuda.current_device = lambda: 0
torch.cuda.Event = H._Event
torch.cuda.current_stream = lambda *a: H._Stream()
torch.Tensor.pin_memory = lambda self: self
class _G:
    def __init__(self): pass
    def replay(self): pass
import contextlib
torch.cuda.CUDAGraph = _G
@contextlib.contextmanager
def _graph(g): yield
torch.cuda.graph = _graph
ops._need_cuda = lambda *ts: None
import pytest
torch.testing.assert_close = lambda *a, **k: None
torch.equal = lambda a, b: True
_pa = pytest.approx
class _Any:
    def __eq__(self, o): return True
    def __req__(self, o): return True
pytest.approx = lambda *a, **k: _Any()
# every GPU test module in tests/, so that a new one is covered without being listed here; the two-GPU module launches worker processes
# on real devices and has nothing to run without them
import glob
mods = sorted(os.path.basename(f)[:-3] for f in glob.glob(os.path.join(ROOT, 'tests', 'test_*_gpu.py')))
mods = [m for m in mods if m != 'test_multigpu_gpu']
# tests that need a real device object even to get going (CUDA generator, IPC allocation): nothing to learn from them here
NEEDS_DEVICE = {'test_fused_allreduce_adam_world1_matches_adam_step', 'test_gae_full_size_properties'}
bad = 0
for mn in mods:
    m = __import__(mn)
    for name, fn in inspect.getmembers(m, inspect.isfunction):
        if not name.startswith('test_'): continue
        marks = getattr(fn, 'pytestmark', []) + list(getattr(m, 'pytestmark', []) if isinstance(getattr(m, 'pytestmark', []), list) else [getattr(m, 'pytestmark')])
        gated = any(mk.name == 'skipif' and 'UNVALIDATED' in str(mk.kwargs.get('reason', '')) + str(mk.args) or (mk.name == 'skipif' and 'hardware' in str(mk.kwargs.get('reason', ''))) for mk in marks)
        if not gated and '--all' not in sys.argv: continue
        if name in NEEDS_DEVICE: continue
        params = [mk for mk in marks if mk.name == 'parametrize']
        names, values = [], [[]]
        for mk in params:
            ns = [x.strip() for x in mk.args[0].split(',')]
            vals = mk.args[1]
            values = [v + (list(x) if len(ns) > 1 else [x]) for v in values for x in vals]
            names += ns
        sig = inspect.signature(fn).parameters
        for vs in values:
            kw = dict(zip(names, vs))
            if 'ops' in sig: kw['ops'] = ops
            if 'tmp_path' in sig:
                import pathlib, tempfile; kw['tmp_path'] = pathlib.Path(tempfile.mkdtemp())
            try:
                fn(**kw)
                print('ran through ', mn, name, {k: v for k, v in kw.items() if k not in ('ops',)})
            except AssertionError as e:
                print('numeric stage', mn, name, list(kw.values())[:2])
            except Exception as e:
                bad += 1
                print('PYTHON ERROR ', mn, name, {k: v for k, v in kw.items() if k != 'ops'}, type(e).__name__, str(e)[:200])
                tb = traceback.extract_tb(e.__traceback__)
                for fr in tb[-3:]: print('      ', fr.filename.split('/')[-1], fr.lineno, fr.line)
print('python errors:', bad)
