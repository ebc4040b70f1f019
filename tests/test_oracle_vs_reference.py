"""Pins the C restatement against the reference's own object code (oracle/_ref: the unmodified reference sources
compiled against stubs).  Where oracle/_ref is built the reference answers live; everywhere else its side comes from
tests/golden/recorded_cases.npz (tests/golden/reference_cases.py says what each case computes)."""
import pytest

from tests.golden import reference_cases as rc

pytestmark = pytest.mark.reference


def _check(name):
    rc.assert_same(rc.compute(name, ref=False), rc.reference(name))


@pytest.mark.parametrize("maxdrift,hbw,thr", rc.PIPELINE_PARAMS)
def test_pipeline_bit_exact_on_synthetic(maxdrift, hbw, thr):
    """FDR geometry and window, spectrogram, normalized average, candidates, blobs, every sync_and_demodulate call
    and every decoder record on four windows from -8 to -28.5 dB"""
    _check("pipeline_md%d_hbw%d_thr%d" % (maxdrift, hbw, thr))


def test_two_signals_and_noise_only():
    _check("two_signals_and_noise")


def test_sync_and_demodulate_function_direct():
    """arbitrary arguments, both drift models, lags that run off both ends of the buffer"""
    _check("sync_and_demodulate_direct")


def test_slm_exhaustive():
    _check("slm_exhaustive")


def test_code_tables_and_decoder():
    _check("code_tables_and_decoder")


def test_sliding_window_against_reference_block():
    want = rc.reference("sliding_window")
    assert int(want["count"][0]) == 4
    _check("sliding_window")
