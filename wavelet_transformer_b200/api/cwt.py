"""Continuous wavelet transform entry point -- mirrors src/cwt.py:39-135.

Same constants, dataclasses and ``run_cwt`` signature as the reference; the
transform itself runs on the GPU through ``pycwt_compat`` (pycwt-shaped facade).
"""

from __future__ import annotations

from dataclasses import dataclass, field
from typing import List, Type

import numpy as np
import numpy.typing as npt

from .. import _shim
from .. import pycwt_compat as wavelet
from .wavelet_helpers import standardize_series

UNITS = "%"
NORMALIZE = True
DT = 1 / 12            # years
S0 = 2 * DT            # smallest scale
DJ = 1 / 12            # twelve sub-octaves per octave
J = 7 / DJ             # seven octaves (float, as in the reference)
MOTHER = wavelet.Morlet(f0=6)
LEVELS = [0.0625, 0.125, 0.25, 0.5, 1, 2, 4, 8, 16]


@dataclass
class DataForCWT:
    """Inputs of a CWT run (src/cwt.py:48-71).  ``t_values`` must be datetime64."""

    t_values: npt.NDArray
    y_values: npt.NDArray
    mother_wavelet: Type
    delta_t: float
    delta_j: float
    initial_scale: float
    levels: List[float]
    time_range: npt.NDArray = field(init=False)

    def __post_init__(self):
        first_year = np.min(self.t_values).astype("datetime64[Y]").astype(int) + 1970
        self.time_range = np.arange(1, self.t_values.size + 1) * self.delta_t + first_year


@dataclass
class ResultsFromCWT:
    """Outputs of a CWT run (src/cwt.py:74-81)."""

    power: npt.NDArray
    period: npt.NDArray
    significance_levels: npt.NDArray
    coi: npt.NDArray


def run_cwt(cwt_data: Type[DataForCWT], normalize: bool = True, standardize: bool = False,
            calculate_significance: bool = True, significance_level: float = 0.95,
            **kwargs) -> Type[ResultsFromCWT]:
    """Power spectrum, Fourier periods, power/significance ratio and COI.

    Behaviour kept from src/cwt.py:85-135: the module constants DT/DJ/S0/J (not
    the dataclass fields) drive the transform; ``normalize`` has no effect
    because the ``standardize`` branch decides the input; ``ar1`` always runs on
    the raw series and raises ``Warning`` when it cannot be bounded."""
    y = cwt_data.y_values
    signal = standardize_series(y, **kwargs) if standardize else y
    alpha, _, _ = wavelet.ar1(y)
    mother = wavelet._as_mother(cwt_data.mother_wavelet)
    if isinstance(mother, wavelet.Morlet):
        # |W|^2 straight from the fused kernel: no complex plane over PCIe, no host abs()**2, and
        # none of the side outputs of pycwt.cwt the reference discards (src/cwt.py:109)
        _, scales, freqs, coi = wavelet._resolve_s0_J(np.size(signal), DT, DJ, S0, J, mother)
        power, _ = _shim.cwt(np.asarray(signal, dtype=float), DT, DJ, S0, int(J), _shim.MORLET, mother.f0)
        power = np.asarray(power, dtype=float)
    else:
        wave, scales, freqs, coi, _, _ = wavelet.cwt(signal, DT, DJ, S0, J, mother)
        power = np.abs(wave) ** 2
    period = 1 / freqs
    ratio = None
    if calculate_significance:
        signif, _ = wavelet.significance(1.0, DT, scales, 0, alpha, significance_level=significance_level,
                                         wavelet=cwt_data.mother_wavelet)
        ratio = power / (np.ones([1, len(cwt_data.t_values)]) * signif[:, None])
    return ResultsFromCWT(power, period, ratio, coi)


def run_cwt_batch(cwt_data_list: List[Type[DataForCWT]], normalize: bool = True, standardize: bool = False,
                  calculate_significance: bool = True, significance_level: float = 0.95,
                  **kwargs) -> List[Type[ResultsFromCWT]]:
    """``run_cwt`` of several equal-length Morlet series as ONE fused CWT+power launch
    (the loop of src/utils/transform_helpers.py:117-124 as a batch).  Per series the result
    equals ``run_cwt``'s; ``ar1`` still raises ``Warning`` for a series it cannot bound."""
    if not cwt_data_list:
        return []
    mother = wavelet._as_mother(cwt_data_list[0].mother_wavelet)
    ys = [np.asarray(d.y_values, dtype=float) for d in cwt_data_list]
    if len({y.size for y in ys}) != 1:
        raise ValueError("run_cwt_batch takes series of equal length")
    alphas = [wavelet.ar1(y)[0] for y in ys]
    signals = np.stack([standardize_series(y, **kwargs) if standardize else y for y in ys])
    n0 = signals.shape[1]
    _, scales, freqs, coi = wavelet._resolve_s0_J(n0, DT, DJ, S0, J, mother)
    power, _ = _shim.cwt(signals, DT, DJ, S0, int(J), _shim.MORLET, mother.f0, f64=True)
    power = np.asarray(power, dtype=float).reshape(len(ys), scales.size, n0)
    period = 1 / freqs
    out = []
    for b, (d, alpha) in enumerate(zip(cwt_data_list, alphas)):
        ratio = None
        if calculate_significance:
            signif, _ = wavelet.significance(1.0, DT, scales, 0, alpha, significance_level=significance_level,
                                             wavelet=mother)
            ratio = power[b] / (np.ones([1, len(d.t_values)]) * signif[:, None])
        out.append(ResultsFromCWT(power[b], period.copy(), ratio, coi.copy()))
    return out


@dataclass
class AveragesFromCWT:
    """Time- and scale-averaged power of one series with their red-noise significance (the pycwt sample's
    glbl_power, glbl_signif, scale_avg and scale_avg_signif; Torrence & Compo 1998 eqs. 22-28)."""

    period: npt.NDArray
    glbl_power: npt.NDArray
    glbl_signif: npt.NDArray
    scale_avg: npt.NDArray
    scale_avg_signif: float


def run_cwt_averages(cwt_data_list: List[Type[DataForCWT]], period_band=(2, 8),
                     significance_level: float = 0.95) -> List[AveragesFromCWT]:
    """The averages section of the pycwt sample for several equal-length series in one batched call: the
    global wavelet spectrum (``power.mean(axis=1)``) and the scale-averaged power over the periods
    ``lo <= period < hi`` (``dj dt / C_delta * sum |W|^2 / s``), both reduced on the device, with
    ``significance(var, ..., sigma_test=1, dof=n0 - scales)`` and ``sigma_test=2`` over the band's scales.
    ``var = y.var()`` and ``alpha = ar1(y)`` per series (``ar1`` raises ``Warning`` when it cannot bound the
    estimate).  Series are transformed as given, as pycwt.cwt does; the module constants DT, DJ, S0 and J drive
    the transform, as in ``run_cwt_batch``."""
    if not cwt_data_list:
        return []
    mother = wavelet._as_mother(cwt_data_list[0].mother_wavelet)
    ys = [np.asarray(d.y_values, dtype=float) for d in cwt_data_list]
    if len({y.size for y in ys}) != 1:
        raise ValueError("run_cwt_averages takes series of equal length")
    n0 = ys[0].size
    _, scales, freqs, _ = wavelet._resolve_s0_J(n0, DT, DJ, S0, J, mother)
    period = 1 / freqs
    sel = np.nonzero((period >= period_band[0]) & (period < period_band[1]))[0]
    if sel.size == 0:
        raise ValueError(f"no scale has a period in [{period_band[0]}, {period_band[1]})")
    if mother.cdelta == -1:
        raise ValueError(f"C_delta is not defined for {mother.name} with these parameters")
    alphas = [wavelet.ar1(y)[0] for y in ys]
    kind, param = wavelet._mother_code(mother)
    glbl, scale_avg = _shim.cwt_averages(np.stack(ys), DT, DJ, S0, int(J), kind, param,
                                         band=(int(sel[0]), int(sel[-1])), band_factor=DJ * DT / mother.cdelta,
                                         f64=True)
    out = []
    for b, (y, alpha) in enumerate(zip(ys, alphas)):
        var = y.var()
        glbl_signif, _ = wavelet.significance(var, DT, scales, 1, alpha, significance_level=significance_level,
                                              dof=n0 - scales, wavelet=mother)
        avg_signif, _ = wavelet.significance(var, DT, scales, 2, alpha, significance_level=significance_level,
                                             dof=[scales[sel[0]], scales[sel[-1]]], wavelet=mother)
        out.append(AveragesFromCWT(period.copy(), glbl[b], glbl_signif, scale_avg[b], float(avg_signif)))
    return out
