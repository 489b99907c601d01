"""Differential test: the oracle restatement vs the UNMODIFIED reference, through the reference's answers to
the same seeded cases (tests/ref_answers.py, recorded by tests/golden/make_golden.py)."""
import pytest

import ref_answers as ra


@pytest.fixture(scope="module")
def answers():
    return ra.load()


def test_datagen_identical(oracle, answers):
    for case, got, want in zip(ra.DATAGEN_CASES, ra.datagen_records(oracle), answers["datagen"]):
        assert got == want, case


def test_compress_and_decode_identical(oracle, answers):
    got = ra.compress_records(oracle, oracle)
    assert len(got) == len(answers["compress"])
    for trial, (g, w) in enumerate(zip(got, answers["compress"])):
        assert g == w, (trial, g, w)


def test_noisy_source_identical(oracle, answers):
    """tests/fuzzer.c:588-622 idea: corrupted blocks must give the same verdict, return value and
    bytes as the reference decoder (x86-64 build)."""
    got = ra.noisy_records(oracle, oracle)
    assert len(got) == len(answers["noisy"])
    for trial, (g, w) in enumerate(zip(got, answers["noisy"])):
        assert g == w, (trial, g, w)
    assert sum(r >= 0 for rets, _ in got for r in rets) > 100
