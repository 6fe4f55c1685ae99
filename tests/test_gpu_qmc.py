"""GPU tests of the device QMC sequence generator (SURVEY.md section 8f row N3) against the
reference's sampling module (oracle/_ref, or its answers recorded under tests/golden): known-answer parity, fp64 bit
for bit."""
import hashlib
import json
import os

import numpy as np
import pytest

from conftest import ROOT

pytestmark = pytest.mark.gpu

KINDS = ["halton", "hammersley", "halton_zaremba", "hammersley_zaremba", "base2", "sobol", "larcher_pillichshammer"]
SCRAMBLES = ["none", "braaten_weller", "faure", "reverse", "custom"]


def bits64(a):
    return np.ascontiguousarray(a, np.float64).view(np.uint64)


def first_primes(n):
    p, k = [], 2
    while len(p) < n:
        if all(k % q for q in p if q * q <= k):
            p.append(k)
        k += 1
    return p


def seeded_tables(n_primes):
    """Permutation tables of the first n_primes primes back to back, from a fixed seed: the stand-in for the
    reference's ScrambleRandomized tables (host-RNG specific) where the reference is not built."""
    rs = np.random.RandomState(4)
    return np.concatenate([rs.permutation(p) for p in first_primes(n_primes)]).astype(np.uint32)


@pytest.mark.parametrize("kind", ["halton", "hammersley"])
@pytest.mark.parametrize("scramble", SCRAMBLES)
def test_halton_hammersley_all_scrambles(cuda_trace, ref_answers, kind, scramble):
    k, s = KINDS.index(kind), SCRAMBLES.index(scramble)
    perm, n_primes, tag = None, 0, scramble
    if scramble == "custom":  # the reference's ScrambleRandomized table is host-RNG specific: upload it
        ref = ref_answers.ref
        perm, n_primes = (ref.qmc_tables(4, 128) if ref is not None else seeded_tables(128)), 128
        tag = "custom_reference_table" if ref is not None else "custom_seeded_table"
    # dimensions 0..39 cross the 16-prime Braaten-Weller limit, 120..135 the 128-prime limit
    for n0, cnt, d0, dn in ((0, 300, 0, 40), (100000, 64, 120, 16), (4294967000, 40, 0, 3), (7, 50, 990, 10)):
        got = cuda_trace.qmc_sequence(kind, n0, cnt, d0, dn, num_smp=1024, scramble=scramble, perm=perm, perm_primes=n_primes)
        ref_answers.check("qmc/%s/%s/%d+%d/dim%d+%d" % (kind, tag, n0, cnt, d0, dn), bits64(got),
                          lambda r: bits64(r.qmc_sequence(k, s, n0, cnt, d0, dn, num_smp=1024)),
                          reference_free=(tag == "custom_seeded_table"))


@pytest.mark.parametrize("kind", ["halton_zaremba", "hammersley_zaremba"])
def test_zaremba(cuda_trace, ref_answers, kind):
    k = KINDS.index(kind)
    for n0, cnt, d0, dn in ((0, 500, 0, 20), (123456789, 100, 3, 5), (4294967200, 50, 0, 4)):
        got = cuda_trace.qmc_sequence(kind, n0, cnt, d0, dn, num_smp=777)
        ref_answers.check("qmc/%s/none/%d+%d/dim%d+%d" % (kind, n0, cnt, d0, dn), bits64(got),
                          lambda r: bits64(r.qmc_sequence(k, 0, n0, cnt, d0, dn, num_smp=777)))


@pytest.mark.parametrize("kind", ["base2", "sobol", "larcher_pillichshammer"])
@pytest.mark.parametrize("scramble_bits", [0, 0xDEADBEEF, 0xFFFFFFFF])
def test_base2_families(cuda_trace, ref_answers, kind, scramble_bits):
    k = KINDS.index(kind)
    for n0, cnt in ((0, 4096), (0xFFFFF000, 4000), (0x80000000 - 100, 200)):
        got = cuda_trace.qmc_sequence(kind, n0, cnt, bits=scramble_bits)
        ref_answers.check("qmc/%s/bits%08x/%d+%d" % (kind, scramble_bits, n0, cnt), bits64(got),
                          lambda r: bits64(r.qmc_sequence(k, 0, n0, cnt, bits=scramble_bits)))


def test_faure_and_prime_tables_generated_here_match_reference(cuda_trace, ref_answers):
    # the device path regenerates primes (sieve) and Faure permutations itself; a wrong table would show
    # up above, this pins them directly through the generated sequences of every table dimension
    got = cuda_trace.qmc_sequence("halton", 1, 200, 0, 128, scramble="faure")
    ref_answers.check("qmc/halton/faure/1+200/dim0+128", bits64(got), lambda r: bits64(r.qmc_sequence(0, 2, 1, 200, 0, 128)))
    if ref_answers.ref is not None:
        assert [ref_answers.ref.qmc_prime(i) for i in (0, 1, 15, 127, 999)] == [2, 3, 53, 719, 7919]


def test_braaten_weller_asset_matches_reference(ref_answers):
    asset = np.fromfile(os.path.join(ROOT, "assets", "sampling", "braaten_weller_16.u32"), np.uint32)
    assert len(asset) == 381
    at = 0
    for p in first_primes(16):  # one permutation of 0..p-1 per prime
        assert sorted(asset[at:at + p].tolist()) == list(range(p))
        at += p
    ref_answers.check("qmc/tables/braaten_weller/16", asset, lambda r: r.qmc_tables(1, 16))


def test_cranley_patterson_including_the_reference_quirk(cuda_trace, ref_answers):
    x = np.array([0.0, 0.25, 0.999, 1.0, 1.0000001, 1.5, 0.7], np.float64)
    for e in (0.0, 0.3, 0.9999):
        ref_answers.check("qmc/cranley_patterson/%r" % e, bits64(cuda_trace.qmc_cranley_patterson(x, e)),
                          lambda r: bits64(r.cranley_patterson(x, e)))
    # the reference tests x (not x + e) against 1: 0.7 + 0.9 is NOT wrapped
    assert cuda_trace.qmc_cranley_patterson(np.array([0.7]), 0.9)[0] > 1.0


def test_argument_errors(cuda_trace):
    from conftest import pkg
    capi = pkg("capi")
    with pytest.raises(capi.CudaTraceError):
        cuda_trace.qmc_sequence("halton", 0, 4, 999, 2)           # dimension beyond the prime table
    with pytest.raises(capi.CudaTraceError):
        cuda_trace.qmc_sequence("hammersley", 0, 4, num_smp=0)
    with pytest.raises(capi.CudaTraceError):
        cuda_trace.qmc_sequence("halton", 0, 4, scramble="custom")  # no table supplied
    bad = np.full(5, 9, np.uint32)
    with pytest.raises(capi.CudaTraceError):
        cuda_trace.qmc_sequence("halton", 0, 4, scramble="custom", perm=bad, perm_primes=2)
