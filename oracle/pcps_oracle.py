"""TEST INFRASTRUCTURE ONLY (oracle) -- NumPy float64 restatement of the Scilab FFT acquisition.

PARITY UNPINNED beyond the restatement itself: Scilab/Octave are not installed here, no recording
or expected output ships with the reference (SURVEY.md §8c), and Scilab's fft is FFTW (not
vendored).  What *is* pinned: the code generators (C/A against the reference C generator
OSG/correlator/correlator.c:63-91 and IS-GPS-200 PRN 1 = 1100100000; tests/test_codes.py) and the
algebra below, which follows the reference line by line:

  SCI/GLONASS/L1/acquisition.sci:49-191   (SCI = trunk/GNSS_SOFTWARE_RECEIVERS/POSTPROCESSING_SCILAB_RECEIVERS)
  SCI/GPS/L1/acquisition.sci              (same algorithm; code table per PRN, '>' at :157)
  SCI/GLONASS/L1/include/makeStTable.sci:41-67, generateSTcode.sci:35-42
  SCI/GPS/L1/include/makeCaTable.sci:43-72,  generateCAcode.sci:42-87
  SCI/*/postProcessing.sce:76-102         (int8 I,Q -> I + i*Q)

It deliberately uses the reference's formulation (Tcoh*16000-point FFTs of the replicated code, one
wipe-off + FFT per bin), not the folded / spectrum-shift formulation of the CUDA path.

Non-coherent mode (n_noncoh >= 2, BASELINE config 4) is NOT in the Scilab code (which keeps the
better of two blocks); it is defined here as the sum over K consecutive Tcoh-ms blocks of
abs(ifft(...))^2 with the same per-block wipe-off, no data-bit handling.

Second-peak window (extension).  acquisition.sci:151-168 searches the second peak over the code phases at circular
distance >= chip = round(fs/codeFreqBasis) from the peak P (1-based), written as three index ranges.  At 31997 of the
32000 (system, P) positions that is exactly second_peak_window(); at GPS P = 17 and GLONASS P = 32 and 15969 the
reference's range leaves 1..N and Scilab stops with an error (exclusion_range restates the ranges as written).  This
library defines those three positions by the circular rule the reference follows everywhere else:
acquisition(..., undefined="circular").  The default, undefined="raise", raises as the reference does.  The per-row
seconds of acquisition()'s "row_second" (the reference computes the second peak of the winning row only) use the
circular rule at every position, as the CUDA path does for every row.
"""
from __future__ import annotations

import os
import sys
from dataclasses import dataclass, field

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
from gnss_sdr_ru_b200.codes import ca_code, st_code  # noqa: E402  (generators are pinned separately)


@dataclass
class AcqSettings:
    system: str = "gps"  # "gps" | "glonass"
    samplingFreq: float = 16.0e6
    IF: float = 2.42e6
    L1_IF_step: float = 0.0
    codeFreqBasis: float = 1.023e6
    codeLength: int = 1023
    acqSearchBand: float = 14.0  # kHz
    acqCohIntegration: int = 4  # ms
    acqThreshold: float = 3.0
    svList: list = field(default_factory=lambda: list(range(1, 33)))  # acqSatelliteList / acqFCHList
    n_noncoh: int = 0

    @staticmethod
    def gps(**kw):
        return AcqSettings(**kw)

    @staticmethod
    def glonass(**kw):
        d = dict(system="glonass", IF=1.0e6, L1_IF_step=0.5625e6, codeFreqBasis=0.511e6, codeLength=511,
                 acqSearchBand=12.0, acqCohIntegration=5, svList=list(range(-7, 7)))
        d.update(kw)
        return AcqSettings(**d)


def samples_per_code(s: AcqSettings) -> int:
    return int(round(s.samplingFreq / (s.codeFreqBasis / s.codeLength)))


def num_bins(s: AcqSettings) -> int:
    # Scilab round(): half away from zero
    return int(np.floor(s.acqSearchBand * 2 * s.acqCohIntegration + 0.5)) + 1


def sampled_code(s: AcqSettings, sv: int) -> np.ndarray:
    """makeCaTable / makeStTable: idx = ceil(ts*(1:N)/tc), last index forced to codeLength."""
    n = samples_per_code(s)
    ts = 1.0 / s.samplingFreq
    tc = 1.0 / s.codeFreqBasis
    idx = np.ceil((ts * np.arange(1, n + 1)) / tc).astype(np.int64)
    idx[-1] = s.codeLength
    chips = ca_code(sv) if s.system == "gps" else st_code()
    return chips[idx - 1].astype(np.float64)


def bin_freq(s: AcqSettings, sv: int, k1: int) -> float:
    """frqBins(k), k 1-based (acquisition.sci:105-108)."""
    base = s.IF + (sv * s.L1_IF_step if s.system == "glonass" else 0.0)
    return base - (s.acqSearchBand / 2) * 1000 + (1000 / (2 * s.acqCohIntegration)) * (k1 - 1)


def to_complex(iq_int8: np.ndarray) -> np.ndarray:
    x = np.asarray(iq_int8, dtype=np.int8).astype(np.float64)
    return x[0::2] + 1j * x[1::2]


def samples_needed(s: AcqSettings) -> int:
    n = samples_per_code(s)
    return (2 if s.n_noncoh <= 1 else s.n_noncoh) * s.acqCohIntegration * n


def acquisition_rows(longSignal: np.ndarray, s: AcqSettings, sv: int, bins=None):
    """results(frqBinIndex,:) for one sv, reduced to per-row (max, first argmax 0-based, block)."""
    rows, full, _ = _rows(longSignal, s, sv, bins)
    return rows, full


def _rows(longSignal, s, sv, bins=None):
    """acquisition_rows plus, per row, the maximum of every block (stock mode: the two the '>' compares)."""
    n = samples_per_code(s)
    T = s.acqCohIntegration
    L = T * n
    ts = 1.0 / s.samplingFreq
    phasePoints = np.arange(L) * 2 * np.pi * ts
    code = np.tile(sampled_code(s, sv), T)
    codeFreqDom = np.conj(np.fft.fft(code))
    nb = num_bins(s)
    bins = range(1, nb + 1) if bins is None else bins
    K = 2 if s.n_noncoh <= 1 else s.n_noncoh
    blocks = [longSignal[k * L:(k + 1) * L] for k in range(K)]
    rows = {}
    full = {}
    block_max = {}
    for k1 in bins:
        f = bin_freq(s, sv, k1)
        sigCarr = np.exp(1j * f * phasePoints)
        res = []
        for blk in blocks:
            fd = np.fft.fft(sigCarr * blk)
            res.append(np.abs(np.fft.ifft(fd * codeFreqDom)) ** 2)
        if s.n_noncoh <= 1:
            blk_idx = 0 if res[0].max() > res[1].max() else 1  # strict '>' (:130)
            row = res[blk_idx][:n]
        else:
            blk_idx = 0
            row = np.sum(res, axis=0)[:n]
        rows[k1] = (float(row.max()), int(np.argmax(row)), blk_idx)
        full[k1] = row
        block_max[k1] = tuple(float(r[:n].max()) for r in res)
    return rows, full, block_max


def exclusion_range(s: AcqSettings, codePhase1: int) -> np.ndarray:
    """1-based code-phase indices searched for the second peak (acquisition.sci:151-168)."""
    n = samples_per_code(s)
    chip = int(np.floor(s.samplingFreq / s.codeFreqBasis + 0.5))
    e1 = codePhase1 - chip
    e2 = codePhase1 + chip
    wrap_hi = (e2 >= n) if s.system == "glonass" else (e2 > n)
    if e1 < 2:
        rng = np.arange(e2, n + e1 + 1)
    elif wrap_hi:
        rng = np.arange(e2 - n, e1 + 1)
    else:
        rng = np.concatenate([np.arange(1, e1 + 1), np.arange(e2, n + 1)])
    return rng


def second_peak_window(s: AcqSettings, codePhase1: int) -> np.ndarray:
    """1-based code-phase indices at circular distance >= chip from the 1-based peak codePhase1: the window of
    exclusion_range wherever that range lies inside 1..N, and this library's definition where it does not."""
    n = samples_per_code(s)
    chip = int(np.floor(s.samplingFreq / s.codeFreqBasis + 0.5))
    d = np.abs(np.arange(1, n + 1) - codePhase1)
    return np.flatnonzero(np.minimum(d, n - d) >= chip) + 1


def row_seconds(s: AcqSettings, rows: dict, full: dict) -> dict:
    """Per row: the largest value inside second_peak_window around that row's own argmax (what the CUDA path stores
    as a row's `second`)."""
    return {k1: float(full[k1][second_peak_window(s, rows[k1][1] + 1) - 1].max()) for k1 in rows}


def acquisition_job(job):
    """(int8 I,Q record, settings) -> acquisition(): a picklable entry point so that tests can run one code entry per
    process (BASELINE config 4 needs about two minutes per PRN in this formulation)."""
    rec, s = job
    return acquisition(to_complex(rec), s)


def acquisition(longSignal: np.ndarray, s: AcqSettings, undefined: str = "raise"):
    """acqResults = acquisition(longSignal, settings).  Returns a list of dicts (one per sv) with
    the reference's fields plus the raw peak data: "rows" {bin: (peak, argmax, block)}, "row_second" {bin: second
    peak of that row} and "row_block_max" {bin: maximum of each block}.
    undefined: what a peak at one of the three positions whose exclusion range leaves 1..N gives -- "raise" (the
    reference stops there) or "circular" (second_peak_window, this library's definition)."""
    if undefined not in ("raise", "circular"):
        raise ValueError(undefined)
    n = samples_per_code(s)
    out = []
    for sv in s.svList:
        rows, full, block_max = _rows(longSignal, s, sv)
        nb = num_bins(s)
        rowmax = np.array([rows[k][0] for k in range(1, nb + 1)])
        peak = rowmax.max()
        frequencyBinIndex = int(np.argmax(rowmax)) + 1  # first row attaining the max (:145)
        colmax = np.max(np.stack([full[k] for k in range(1, nb + 1)]), axis=0)
        codePhase = int(np.argmax(colmax)) + 1  # first column attaining it (:148)
        rng = exclusion_range(s, codePhase)
        if rng.min() < 1 or rng.max() > n:
            if undefined == "raise":
                raise IndexError(f"Scilab would raise: exclusion range of peak {codePhase} leaves 1..{n} (acquisition.sci:151-168)")
            rng = second_peak_window(s, codePhase)
        second = float(full[frequencyBinIndex][rng - 1].max())
        metric = peak / second
        r = dict(sv=sv, peakMetric=metric, bin=frequencyBinIndex, codePhaseRaw=codePhase, peak=float(peak),
                 second=second, carrFreq=0.0, codePhase=0, freqChannel=0, rows=rows,
                 row_second=row_seconds(s, rows, full), row_block_max=block_max)
        if metric > s.acqThreshold:
            r["codePhase"] = codePhase
            r["carrFreq"] = bin_freq(s, sv, frequencyBinIndex)
            r["freqChannel"] = sv
        out.append(r)
    return out
