import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box)")


@pytest.fixture(scope="session")
def oracle_lib():
    from oracle import oracle_api

    oracle_api.build()
    return oracle_api


@pytest.fixture(scope="session")
def track_record():
    """~1.75 s GPS record, three satellites in Doppler bins +1/-1/+1 (seed 2002-like)."""
    from gnss_sdr_ru_b200.synth import Sat, make_record

    nblk = 3400
    sats = [
        Sat(prn=27, doppler_hz=1200, cn0_dbhz=50, code_phase_chips=1000.3, data_seed=5),
        Sat(prn=9, doppler_hz=-900, cn0_dbhz=47, code_phase_chips=980.0, data_seed=6),
        Sat(prn=32, doppler_hz=1000, cn0_dbhz=49, code_phase_chips=1010.0, data_seed=7),
    ]
    # generated in every session: a file shared between runs could come from another version of synth.py
    return make_record(sats, 8192 * nblk, seed=2002), nblk
