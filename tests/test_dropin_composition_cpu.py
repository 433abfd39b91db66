"""`cutie/` (this repo's drop-in shim) composed with a reference checkout on sys.path: modules the shim provides -- the
hot-path surface -- win; everything else (dataset readers, palette, ...) resolves to the reference's own files, so
eval_vos.py-style imports work unchanged with this repo placed AHEAD of the reference on PYTHONPATH.  The reference
checkout is a stand-in with the reference's package layout (hkchengrex/Cutie: `cutie/` without an __init__.py, empty
sub-package __init__.py files) and one-line modules at the paths involved."""
import os
import subprocess
import sys

from tests.conftest import ROOT

# modules of the reference that the shim also provides, and modules only the reference has
SHIM_PROVIDED = ['cutie/inference/inference_core.py', 'cutie/inference/memory_manager.py',
                 'cutie/inference/kv_memory_store.py', 'cutie/inference/object_manager.py', 'cutie/model/cutie.py',
                 'cutie/utils/get_default_model.py']
REFERENCE_ONLY = ['cutie/inference/data/video_reader.py', 'cutie/inference/data/vos_test_dataset.py',
                  'cutie/utils/palette.py']


def _stand_in_reference(root):
    for pkg in ('cutie/inference', 'cutie/inference/data', 'cutie/model', 'cutie/utils'):
        os.makedirs(os.path.join(root, pkg), exist_ok=True)
        open(os.path.join(root, pkg, '__init__.py'), 'w').close()
    for f in SHIM_PROVIDED + REFERENCE_ONLY:
        with open(os.path.join(root, f), 'w') as fh:
            fh.write('"""stand-in for the reference module at this path"""\n')
    return root


PROBE = r'''
import importlib, json
out = {}
for mod in ['cutie.inference.inference_core', 'cutie.inference.memory_manager', 'cutie.inference.kv_memory_store',
            'cutie.inference.object_manager', 'cutie.model.cutie', 'cutie.utils.get_default_model',
            'cutie.inference.data.video_reader', 'cutie.inference.data.vos_test_dataset', 'cutie.utils.palette']:
    out[mod] = importlib.import_module(mod).__file__
from cutie.inference.inference_core import InferenceCore
out['InferenceCore'] = InferenceCore.__module__
print(json.dumps(out))
'''


def test_shim_wins_for_the_hot_path_and_defers_to_the_reference_elsewhere(tmp_path):
    import json
    REF = _stand_in_reference(str(tmp_path / 'reference'))
    env = dict(os.environ, PYTHONPATH=os.pathsep.join([ROOT, REF]))
    r = subprocess.run([sys.executable, '-c', PROBE], capture_output=True, text=True, cwd=str(tmp_path), env=env, timeout=300)
    assert r.returncode == 0, r.stderr[-2000:]
    got = json.loads(r.stdout.strip().splitlines()[-1])
    ours = [m for m, f in got.items() if f.startswith(ROOT + os.sep)]
    theirs = [m for m, f in got.items() if f.startswith(REF + os.sep)]
    assert set(ours) == {'cutie.inference.inference_core', 'cutie.inference.memory_manager', 'cutie.inference.kv_memory_store',
                         'cutie.inference.object_manager', 'cutie.model.cutie', 'cutie.utils.get_default_model'}
    assert set(theirs) == {'cutie.inference.data.video_reader', 'cutie.inference.data.vos_test_dataset', 'cutie.utils.palette'}
    assert got['InferenceCore'] == 'cutie_b200.inference.inference_core'


def test_shim_alone_still_imports():
    env = dict(os.environ, PYTHONPATH=ROOT)
    r = subprocess.run([sys.executable, '-c', 'from cutie.inference.inference_core import InferenceCore; '
                        'from cutie.utils.get_default_model import get_default_model; print(InferenceCore.__module__)'],
                       capture_output=True, text=True, env=env, timeout=300)
    assert r.returncode == 0 and 'cutie_b200.inference.inference_core' in r.stdout, r.stderr[-2000:]
