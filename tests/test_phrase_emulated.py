"""The phrase kernels (bm25_phrase.cuh) on the CPU SIMT emulator (tests/emu): the functions of tests/test_phrase_gpu.py run
unchanged against the oracle with libsb200_emu.so underneath, the way test_bm25_emulated.py runs the other BM25 kernels."""
import ctypes as C
import os
import subprocess

import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
EMU = os.path.join(HERE, "emu")


@pytest.fixture(scope="module")
def emulated():
    subprocess.check_call(["make", "-C", EMU], stdout=subprocess.DEVNULL)
    from stract_b200 import _lib
    L = _lib.declare(C.CDLL(os.path.join(EMU, "libsb200_emu.so")))
    assert b"emulation" in L.sb200_version()
    saved = _lib._LIB
    _lib._LIB = L
    import test_phrase_gpu as T
    T.RANDOM_DOCS, T.RANDOM_LEN, T.QUERIES_PER_LEN = 300, 200, (2, 1, 1)
    try:
        yield T
    finally:
        _lib._LIB = saved


def test_reference_scenarios(emulated):
    emulated.test_reference_scenarios_on_device()


def test_random_phrases(emulated):
    emulated.test_random_phrases_bit_exact()


def test_ties_searcher_term_info_store(emulated):
    emulated.test_ties_order_by_doc()
    emulated.test_searcher_over_three_segments_matches_one_big_segment()
    emulated.test_term_info_store_positions_ranges_on_device()


def test_errors_and_corrupt_positions(emulated):
    emulated.test_errors()
