"""Golden Hessians for the window optimiser (SURVEY 8f-2), produced by executing the REFERENCE's own builders:
OptimizerTx / OptimizerRx / OptimizerTxRx .gen_hessian (python/optimization_tools/optimizers.py) on a small system
(N = 64) so that the reference's O(n^2 N^2) loops finish in seconds.

Run:  WOFDM_REFERENCE=<checkout of felipescoelho/w-ofdm-optimization> python -B tests/golden/make_golden_hessian.py"""
import os
import sys

sys.dont_write_bytecode = True
HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(os.environ["WOFDM_REFERENCE"], "python"))
import numpy as np  # noqa: E402
from optimization_tools.optimizers import OptimizerTx, OptimizerRx, OptimizerTxRx  # noqa: E402

N, CP, TTX, TRX, L = 64, 10, 4, 6, 9
rng = np.random.default_rng(2024)
h = (rng.standard_normal(L) + 1j * rng.standard_normal(L)) * np.exp(-np.arange(L) / 3.0)
out = {"N": N, "cp": CP, "tail_tx": TTX, "tail_rx": TRX, "h": h}
for name in ("wtx", "CPwtx"):
    o = OptimizerTx(name, N, CP, TTX)
    out[f"H_{name}"] = o.gen_hessian(o.calculate_chann_matrices(h))
for name in ("wrx", "CPwrx"):
    o = OptimizerRx(name, N, CP, TRX)
    out[f"H_{name}"] = o.gen_hessian(o.calculate_chann_matrices(h))
for name in ("WOLA", "CPW"):
    o = OptimizerTxRx(name, N, CP, TTX, TRX)
    out[f"H_{name}"] = o.gen_hessian(o.calculate_chann_matrices(h))
np.savez_compressed(os.path.join(HERE, "hessian.npz"), **out)
print({k: np.shape(v) for k, v in out.items()})
