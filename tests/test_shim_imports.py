"""CPU: import mechanics of the `src_seq` shadow package (no kernels run): shadowed modules resolve to the drop-in
classes, everything else to the reference tree's own files, RE2NN_SHIM=off falls through.  The reference tree is the
stand-in of helpers.stand_in_reference (the reference's layout and names), written to a temporary directory."""
import os
import subprocess
import sys

from helpers import stand_in_reference

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

CODE = r'''
import os, sys
from src_seq.farnn.model_decompose_single import FARNN_S_D_W_I_S, FARNN_S_SF
from src_seq.farnn.model_onehot import FARNN_S_O_I_S, FARNN_S_O_I, FARNN_S_O
from src_seq.farnn.model_decompose import FARNN_S_D_W
from src_seq.farnn.model_decompose_independent import FARNN_S_D_W_I
from src_seq.farnn.priority import PriorityLayer
from src_seq.baselines.crf import CRF
from src_seq.baselines.KD import KD_loss
import src_seq.val, src_seq.utils
mods = [c.__module__ for c in (FARNN_S_D_W_I_S, FARNN_S_SF, FARNN_S_O_I_S, FARNN_S_O_I, FARNN_S_O, FARNN_S_D_W, FARNN_S_D_W_I,
                                PriorityLayer, CRF)]
print('|'.join(mods))
print(src_seq.val.__file__ + '|' + src_seq.utils.__file__ + '|' + KD_loss.__module__)
'''


def _run(shim_on, ref):
    env = dict(os.environ, PYTHONPATH=os.pathsep.join([os.path.join(ROOT, 'shim'), ROOT]), RE2NN_REFERENCE_ROOT=ref,
               RE2NN_SHIM='on' if shim_on else 'off')
    r = subprocess.run([sys.executable, '-c', CODE], env=env, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True,
                       timeout=300)
    assert r.returncode == 0, r.stderr[-2000:]
    return r.stdout.strip().splitlines()[-2:]


def test_shim_resolves_dropins_and_reference_files(tmp_path):
    ref = stand_in_reference(tmp_path)
    mods, files = _run(True, ref)
    assert all(m.startswith('re2nn_seq_b200') for m in mods.split('|')), mods
    val_file, utils_file, kd_mod = files.split('|')
    assert os.path.abspath(val_file).startswith(ref) and os.path.abspath(utils_file).startswith(ref)
    assert kd_mod == 'src_seq.baselines.KD'


def test_shim_off_is_the_reference(tmp_path):
    mods, _ = _run(False, stand_in_reference(tmp_path))
    assert all(m.startswith('src_seq.') for m in mods.split('|')), mods
