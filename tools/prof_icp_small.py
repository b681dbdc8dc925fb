import os, sys
os.environ["OPE_ICP_SMALL"]="1"; os.environ["OPE_PROFILE"]="1"
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, 'oracle'))
import numpy as np, ope_pkg; ope_pkg.load()
from ope_b200 import cuda_lib, synth
import ctypes
ctx = cuda_lib.Context(0)
model = synth.bundled_model()
for f in range(3):
    cl = synth.make_frame(model, 1000+f)[0]
    tr = cuda_lib.PoseTracker(ctx); ctypes.CDLL(None).srand(1)
    r = tr.estimate_final(model.copy(), cl); print("frame", f, "iters", r.icp_iterations, "nsrc", r.n_src_fine, "ntgt", r.n_tgt_fine, "icp ms", tr.stage_ms()[4]); tr.close()
