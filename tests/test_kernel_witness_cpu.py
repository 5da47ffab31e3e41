"""parse_kernel (tests/kernel_witness.py) on the demangled names the profiler reports for the library's kernels: a slip here would
make the kernel-variant matrices assert the wrong kernel, so it is checked without a GPU."""
import pytest

from kernel_witness import Registry, parse_kernel


@pytest.mark.parametrize("name,want", [
    ("void rx4096_kernel<true, false, (int)257, true>(Fast4096Params, const float2 *, long)", ("rx4096_kernel", (True, False, 257, True))),
    ("void rx4096_kernel<false, true, (int)4369, false>(Fast4096Params, float2*)", ("rx4096_kernel", (False, True, 0x1111, False))),
    ("void rx_t4_fast_kernel<(int)32, true, false>(T4Params, T4FastExtra, PlanDev<float>, DevConst<float>, const float2 *, long, long)",
     ("rx_t4_fast_kernel", (32, True, False))),
    ("void rx_t4_fast_kernel<(int)13, false, true>(T4Params, T4FastExtra, PlanDev<float>, DevConst<float>)", ("rx_t4_fast_kernel", (13, False, True))),
    ("void t4_post_kernel<false, true, false>(T4Params, T4FastExtra, PlanDev<float>, DevConst<float>, long, const float2 *, T4Stats)",
     ("t4_post_kernel", (False, True, False))),
    ("void t4_sym_kernel<(int)13>(T4Params, T4FastExtra, const float2 *, long, long, int, const int *, const double *)", ("t4_sym_kernel", (13,))),
    ("void rx_t3_kernel<(int)32, true>(T3Params, T4FastExtra, DevConst<float>, float, float, const float2 *)", ("rx_t3_kernel", (32, True))),
    ("void rx_chain_kernel<float>(LinkDev<float>, PlanDev<float>, const cx<float> *)", ("rx_chain_kernel", ("float",))),
    ("void tx_chain_kernel<double>(LinkDev<double>, const unsigned int *, long, cx<double> *)", ("tx_chain_kernel", ("double",))),
    ("rx_t4_kernel(T4Params, PlanDev<float>, DevConst<float>, const float2 *, long)", ("rx_t4_kernel", ())),
    ("void t4_ifo_kernel(T4FastExtra, const float2 *, long, long, int, int, const int *, const double *, int *)", ("t4_ifo_kernel", ())),
    ("void tx1024_kernel(Tx1024Params, DevConst<float>, const unsigned int *, long, float2 *, double *)", ("tx1024_kernel", ())),
    ("void ns::inner::k<(unsigned int)7u, (long)-3l>(int)", ("k", (7, -3))),
])
def test_parse_kernel_names(name, want):
    assert parse_kernel(name) == want


@pytest.mark.parametrize("name", ["Memset (Device)", "Memcpy HtoD (Pageable -> Device)", "Memcpy DtoD (Device -> Device)", "", "void"])
def test_parse_kernel_skips_activity_that_is_not_a_kernel(name):
    assert parse_kernel(name) is None


def test_registry_records_cases_and_missing_profiler():
    r = Registry()
    assert r.available is None
    assert r.record([("t4_sym_kernel", (32,)), ("t4_post_kernel", (True, False, False))], "a")
    assert r.record([("t4_sym_kernel", (32,))], "b")
    assert r.available is True and r.seen[("t4_sym_kernel", (32,))] == {"a", "b"}
    assert not r.record(None, "c")
    assert r.available is False and "c" not in set().union(*r.seen.values())
