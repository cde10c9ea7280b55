"""The reference's GPU X-TDA class (xtddft/XTDA_GPU.py:24-500) on the B200 engine: `XTDA(mol, mf, nstates, so2st)`,
`kernel(x0=None, nstates=None) -> (e, v)`, host-Davidson solver settings of XTDA_GPU.py:393-395."""
from __future__ import annotations

from .XTDA import XTDA as _XTDA


class XTDA(_XTDA):
    def __init__(self, mol, mf, nstates=10, so2st=True, core_idx=None):
        super().__init__(mol, mf, nstates=nstates, basis="orbital", so2st=so2st, use_Davidson=True, core_idx=core_idx)
        self.level_shift = getattr(mf, "level_shift", 0) or 0
        self._settings = "gpu_class"

    def kernel(self, x0=None, nstates=None):
        e = self.Davidson(x0=x0, nstates=nstates)
        return e, self.v
