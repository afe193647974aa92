"""TEST INFRASTRUCTURE ONLY (oracle) -- NumPy float64 restatement of the Scilab receivers' tracking.

PARITY: the loop closure -- discriminators, FLL-assisted PLL and DLL filters, carrier / code NCO updates, block
sizes and the code-phase remainder -- is PINNED against the reference's own saved run
SCI/GLONASS/L1/trackingResults.dat (1500 ms of a real GLONASS signal, Scilab `save` of trackResults / settings /
acqResults / channel, postProcessing.sce:143): fed with the recorded correlator outputs, LoopFilters / block_size
below reproduce the recorded carrFreq, codeFreq, dllDiscr, dllDiscrFilt and absoluteSample series bit for bit, pllDiscr
to one ulp of atan() and pllDiscrFilt to 1e-13 (tests/test_softtrack_refrun.py; that run predates two lines of today's tracking.sci, whose
earlier forms survive as comments at :366 and :379 and are selectable here).  The correlator sums themselves are
UNPINNED: the recording that run read (FFF005.DAT) is not in the repository and there is no Scilab here.
Follows, line by line,

  SCI/GLONASS/L1/tracking.sci:100-425        (SCI = trunk/GNSS_SOFTWARE_RECEIVERS/POSTPROCESSING_SCILAB_RECEIVERS)
  SCI/GLONASS/L1/include/calcLoopCoef.sci:38-43, calcFLLPLLLoopCoef.sci:36-38
  SCI/GLONASS/L1/include/preRun.sci:66-81    (channel list from acqResults, strongest first)
  SCI/GLONASS/L1/initSettings.sci:41-107

for GLONASS L1OF, and the same algorithm with the C/A code and the GPS code-aiding term
(tracking.sci:366, the commented GPS formula) when settings.system == "gps".

One code period per iteration, variable block size ceil((L-rem)/step), float carrier/code NCOs,
FLL-assisted PLL + DLL (tracking.sci:226-400).  Elementwise expressions keep the reference's operation
order; the only intentional freedom is the summation order inside sum().
"""
from __future__ import annotations

import os
import sys
from dataclasses import dataclass, field

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
from gnss_sdr_ru_b200.codes import ca_code, st_code  # noqa: E402


@dataclass
class TrackSettings:
    system: str = "glonass"
    samplingFreq: float = 16e6
    IF: float = 1e6
    L1_IF_step: float = 0.5625e6
    GLONASS_zero_channel: float = 1602e6
    codeFreqBasis: float = 0.511e6
    codeLength: int = 511
    skipNumberOfSamples: int = 0  # skipNumberOfBytes / dataTypeSizeInBytes (complex samples)
    msToProcess: int = 1000
    numberOfChannels: int = 8
    dllDampingRatio: float = 0.7
    dllNoiseBandwidth: float = 0.5
    dllCorrelatorSpacing: float = 0.05
    pllNoiseBandwidth: float = 25.0
    fllNoiseBandwidth: float = 250.0
    codeAiding: bool = True         # tracking.sci:367-369 (False: the earlier form kept as a comment at :366)
    absSampleRemCorr: bool = True   # tracking.sci:384-385 (False: the earlier form kept as a comment at :379)

    @staticmethod
    def gps(**kw):
        d = dict(system="gps", IF=2.42e6, L1_IF_step=0.0, codeFreqBasis=1.023e6, codeLength=1023,
                 dllNoiseBandwidth=0.1, dllCorrelatorSpacing=0.2)
        d.update(kw)
        return TrackSettings(**d)


def calc_loop_coef(LBW, zeta, k):
    Wn = LBW * 8 * zeta / (4 * zeta ** 2 + 1)
    return k / (Wn * Wn), 2.0 * zeta / Wn


def calc_fll_pll_coef(pllbw, fllbw, T):
    k1 = T * ((pllbw / 0.53) ** 2) + 1.414 * (pllbw / 0.53)
    k2 = 1.414 * (pllbw / 0.53)
    k3 = T * (fllbw / 0.25)
    return k1, k2, k3


def pre_run(acq, settings: TrackSettings):
    """preRun.sci:66-81: channels = detected signals sorted by peakMetric (descending)."""
    order = np.argsort(-np.asarray(acq["peakMetric"]), kind="stable")
    n = min(settings.numberOfChannels, int(np.sum(np.asarray(acq["carrFreq"]) != 0)))
    chans = []
    for ii in range(n):
        i = int(order[ii])
        chans.append(dict(SVN=i + 1, FCH=int(acq["freqChannel"][i]), acquiredFreq=float(acq["carrFreq"][i]),
                          codePhase=int(acq["codePhase"][i])))
    return chans


FIELDS = ("I_E", "I_P", "I_L", "Q_E", "Q_P", "Q_L", "carrFreq", "codeFreq", "dllDiscr", "dllDiscrFilt", "pllDiscr",
          "pllDiscrFilt", "absoluteSample")


def block_size(s: TrackSettings, remCodePhase: float, codeFreq: float):
    """tracking.sci:232-236, 262-263: samples of this code period and the remainder carried into the next one"""
    codePhaseStep = codeFreq / s.samplingFreq
    blksize = int(np.ceil((s.codeLength - remCodePhase) / codePhaseStep))
    last = remCodePhase + float(blksize - 1) * codePhaseStep  # tcode(blksize) of remCodePhase : step : ((blksize-1)*step+rem)
    return blksize, codePhaseStep, (last + codePhaseStep) - s.codeLength


class LoopFilters:
    """tracking.sci:320-372: what turns the six correlator sums of a code period into the next carrier / code frequency"""

    def __init__(self, s: TrackSettings, channel: dict):
        self.s = s
        self.fch = channel["FCH"]
        self.tau1code, self.tau2code = calc_loop_coef(s.dllNoiseBandwidth, s.dllDampingRatio, 1.0)
        self.k1, self.k2, self.k3 = calc_fll_pll_coef(s.pllNoiseBandwidth, s.fllNoiseBandwidth, 0.001)
        self.carrFreqBasis = channel["acquiredFreq"]
        self.oldCodeNco = self.oldCodeError = self.oldCarrNco = self.oldCarrError = 0.0
        self.I1 = self.I2 = self.Q1 = self.Q2 = 0.001

    def update(self, I_E, Q_E, I_P, Q_P, I_L, Q_L):
        """returns carrFreq, codeFreq, codeError, codeNco, carrError, carrNco"""
        s = self.s
        PDIcode = 0.001
        self.I2, self.Q2 = self.I1, self.Q1
        self.I1, self.Q1 = I_P, Q_P
        cross = self.I1 * self.Q2 - self.I2 * self.Q1
        dot = abs(self.I1 * self.I2 + self.Q1 * self.Q2)
        freqError = np.arctan2(cross, dot) / np.pi
        carrError = np.arctan(Q_P / I_P) / (2.0 * np.pi)
        carrNco = self.oldCarrNco + self.k1 * carrError - self.k2 * self.oldCarrError - self.k3 * freqError
        self.oldCarrNco = carrNco
        self.oldCarrError = carrError
        carrFreq = self.carrFreqBasis + carrNco
        sE = np.sqrt(I_E * I_E + Q_E * Q_E)
        sL = np.sqrt(I_L * I_L + Q_L * Q_L)
        codeError = (sE - sL) / (sE + sL)
        codeNco = self.oldCodeNco + (self.tau2code / self.tau1code) * (codeError - self.oldCodeError) + codeError * (PDIcode / self.tau1code)
        self.oldCodeNco = codeNco
        self.oldCodeError = codeError
        if not s.codeAiding:
            codeFreq = s.codeFreqBasis - codeNco
        elif s.system == "glonass":
            codeFreq = s.codeFreqBasis - codeNco + (carrFreq - (s.IF + s.L1_IF_step * self.fch)) / (
                (s.GLONASS_zero_channel + self.fch * s.L1_IF_step) / s.codeFreqBasis)
        else:
            codeFreq = s.codeFreqBasis - codeNco + ((carrFreq - s.IF) / 1540)
        return carrFreq, codeFreq, codeError, codeNco, carrError, carrNco


def replay(rec: dict, channel: dict, s: TrackSettings):
    """The loop closure alone, driven by RECORDED correlator outputs rec["I_E"] ... rec["Q_L"] (a saved run of the
    reference): returns the series the reference would have stored next to them."""
    lf = LoopFilters(s, channel)
    pos = s.skipNumberOfSamples + (channel["codePhase"] - 1)
    currentSample = 2 * pos
    codeFreq = s.codeFreqBasis
    remCodePhase = 0.0
    names = ("carrFreq", "codeFreq", "dllDiscr", "dllDiscrFilt", "pllDiscr", "pllDiscrFilt", "absoluteSample", "blksize")
    out = {f: [] for f in names}
    for k in range(len(rec["I_P"])):
        blksize, _, remCodePhase = block_size(s, remCodePhase, codeFreq)
        currentSample += 2 * blksize
        carrFreq, codeFreq, codeError, codeNco, carrError, carrNco = lf.update(
            float(rec["I_E"][k]), float(rec["Q_E"][k]), float(rec["I_P"][k]), float(rec["Q_P"][k]), float(rec["I_L"][k]), float(rec["Q_L"][k]))
        absoluteSample = currentSample / 2 - (remCodePhase * (s.samplingFreq / 1000) / s.codeLength if s.absSampleRemCorr else 0.0)
        for f, v in zip(names, (carrFreq, codeFreq, codeError, codeNco, carrError, carrNco, absoluteSample, blksize)):
            out[f].append(v)
    return {f: np.array(v) for f, v in out.items()}


def _chips(caCode: np.ndarray, t: np.ndarray, what: str) -> np.ndarray:
    """caCode(ceil(tcode)+1) (1-based) as a 0-based lookup; an index outside the padded code raises, as in Scilab."""
    idx = np.ceil(t).astype(np.int64)
    if idx.size and (idx.min() < 0 or idx.max() > caCode.size - 1):
        raise IndexError(f"{what} code index {int(idx.min())}..{int(idx.max())} outside 0..{caCode.size - 1} "
                         "(Scilab: invalid index)")
    return caCode[idx]


def tracking(iq_int8: np.ndarray, channel: dict, s: TrackSettings, left_pad: float | None = None):
    """One channel of tracking.sci.  iq_int8: interleaved I,Q record (the whole file).  Returns a dict of
    arrays of length msToProcess (shorter if the record ends).  A code index outside the padded code raises
    IndexError, where Scilab stops with an invalid index (a correlator spacing of a chip or more in period 1).
    left_pad replaces the value of caCode($) at the front of the padded code (mutation checks; None: the reference)."""
    x = np.asarray(iq_int8, dtype=np.int8)
    sig_all = x[0::2].astype(np.float64) + 1j * x[1::2].astype(np.float64)
    fs = s.samplingFreq
    L = s.codeLength
    code = (ca_code(channel["FCH"]) if s.system == "gps" else st_code()).astype(np.float64)
    caCode = np.concatenate([code[-1:] if left_pad is None else [float(left_pad)], code, code[:1]])
    earlyLateSpc = s.dllCorrelatorSpacing
    lf = LoopFilters(s, channel)
    pos = s.skipNumberOfSamples + (channel["codePhase"] - 1)
    currentSample = 2 * pos  # bytes (dataAdaptCoeff = 2, 1 byte per value)
    codeFreq = s.codeFreqBasis
    remCodePhase = 0.0
    carrFreq = channel["acquiredFreq"]
    remCarrPhase = 0.0
    out = {f: [] for f in FIELDS}
    for _ in range(s.msToProcess):
        codePhaseStep = codeFreq / fs
        blksize = int(np.ceil((L - remCodePhase) / codePhaseStep))
        if pos + blksize > sig_all.size:
            break
        rawSignal = sig_all[pos:pos + blksize]
        pos += blksize
        currentSample += 2 * blksize
        j = np.arange(blksize, dtype=np.float64)
        tE = (remCodePhase - earlyLateSpc) + j * codePhaseStep
        tL = (remCodePhase + earlyLateSpc) + j * codePhaseStep
        tP = remCodePhase + j * codePhaseStep
        earlyCode = _chips(caCode, tE, "early")   # Scilab: caCode(ceil(tcode)+1), 1-based
        lateCode = _chips(caCode, tL, "late")
        promptCode = _chips(caCode, tP, "prompt")
        remCodePhase = (tP[blksize - 1] + codePhaseStep) - L
        time = np.arange(blksize + 1, dtype=np.float64) / fs
        trigarg = ((carrFreq * 2.0 * np.pi) * time) + remCarrPhase
        last = trigarg[blksize]
        remCarrPhase = last - np.fix(last / (2 * np.pi)) * (2 * np.pi)
        carrsig = np.exp(1j * trigarg[:blksize])
        mixed = carrsig * rawSignal
        qBB = mixed.real
        iBB = mixed.imag
        I_E = float(np.sum(earlyCode * iBB))
        Q_E = float(np.sum(earlyCode * qBB))
        I_P = float(np.sum(promptCode * iBB))
        Q_P = float(np.sum(promptCode * qBB))
        I_L = float(np.sum(lateCode * iBB))
        Q_L = float(np.sum(lateCode * qBB))
        carrFreq, codeFreq, codeError, codeNco, carrError, carrNco = lf.update(I_E, Q_E, I_P, Q_P, I_L, Q_L)
        absoluteSample = currentSample / 2 - (remCodePhase * (fs / 1000) / L if s.absSampleRemCorr else 0.0)
        for f, v in zip(FIELDS, (I_E, I_P, I_L, Q_E, Q_P, Q_L, carrFreq, codeFreq, codeError, codeNco, carrError, carrNco,
                                 absoluteSample)):
            out[f].append(v)
    return {f: np.array(v) for f, v in out.items()}
