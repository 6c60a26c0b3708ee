"""Generate tests/golden/solver_ref.npz: the reference's own GPTQ solver (`gptq.py`, imported unmodified) on the seeded layers and
calibration batches of tests/test_gptq_solver.py.

    PYTHONDONTWRITEBYTECODE=1 python tests/golden/make_solver_golden.py <reference checkout>

The reference's table-printing dependency `texttable` and the SNR helper it pulls from `utils` are stubbed (neither touches the result),
and its unconditional torch.cuda.synchronize() is a no-op so that it runs on the CPU.  Its `import quant` resolves to this repository's
package, whose Quantizer reproduces the reference's bit for bit (tests/test_host_modules.py).  Stored per case: a seeded sample of the
Hessian, scale, zero, g_idx, the error and the on-grid weights as uint8 grid codes (they reconstruct the reference's fp32 weights exactly).
"""
import importlib
import os
import sys
import types

import numpy as np
import torch

sys.dont_write_bytecode = True
HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
for p in (os.path.dirname(HERE), ROOT, os.path.join(ROOT, 'gptq-for-llama_b200')):
    sys.path.insert(0, p)
import test_gptq_solver as T  # noqa: E402


def reference_gptq(ref_dir):
    import quant  # noqa: F401  (this repo's package, see above)
    import utils as ours
    tt = types.ModuleType('texttable')

    class Texttable:  # only used to print one line per layer
        def header(self, *a): pass
        def set_cols_dtype(self, *a): pass
        def add_row(self, *a): pass
        def draw(self): return 'a\nb\nc'
    tt.Texttable = Texttable
    shim = types.ModuleType('utils')
    shim.find_layers, shim.DEV = ours.find_layers, ours.DEV
    shim.torch_snr_error = lambda a, b, reduction='mean': ((a - b)**2 / (b**2 + 1e-12)).mean()
    sys.modules.update(texttable=tt, utils=shim)
    sys.modules.pop('gptq', None)
    sys.path.insert(0, ref_dir)
    try:
        ref = importlib.import_module('gptq')
        assert os.path.abspath(ref.__file__).startswith(os.path.abspath(ref_dir))
    finally:
        sys.path.remove(ref_dir)
    torch.cuda.synchronize = lambda *a, **k: None
    return ref


def main(ref_dir):
    ref = reference_gptq(ref_dir)
    out = {}
    for case in T.CASES:
        K = case[0]
        name = T.case_name(*case)
        r = T.run_solver(ref.GPTQ, *case)
        codes = T.grid_codes(r)
        g = r['g_idx'].long()
        assert torch.equal(r['scale'][:, g] * (codes - r['zero'][:, g]), r['W']), name
        assert codes.min() >= 0 and codes.max() <= 2**case[2] - 1
        out.update({f'{name}/H_sample': r['H'].flatten()[T.h_sample_index(K)].numpy(), f'{name}/scale': r['scale'].numpy(),
                    f'{name}/zero': r['zero'].numpy(), f'{name}/g_idx': r['g_idx'].numpy(), f'{name}/codes': codes.numpy().astype(np.uint8),
                    f'{name}/err': np.float64(r['err'])})
    path = os.path.join(HERE, 'solver_ref.npz')
    np.savez_compressed(path, **out)
    print(f'wrote {len(T.CASES)} cases to {path} ({os.path.getsize(path)} bytes)')


if __name__ == '__main__':
    main(sys.argv[1])
