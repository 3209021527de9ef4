"""Building a handle or a plan and destroying it again gives back all the device memory the build
took: the staging arrays of the HLL constructors, the temporaries and the arrays of SELL-P plans,
and the slice plans SpMM builds for itself."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

KNOB_DEFAULTS = {"sell": -1, "sell_panels": 0, "sell_max_row": 4096, "sell_chunk": 256, "sell_panel_mb": 64}


@pytest.fixture(scope="module")
def torch():
    import torch
    assert torch.cuda.is_available()
    return torch


def test_builds_return_their_device_memory(sp, torch):
    A = sp.gen_ragged(5000, 700)               # row lengths spread over 0..700
    E = sp.csr_from_arrays("empty", 1000, 64, np.zeros(1001, np.int32), [], [])  # 32 hacks, all empty
    # 3.5M columns of uniform random gathers, 16 MB panels: 1, 4 and 7 column panels for 1, 2 and 4
    # right-hand sides, so SpMM builds plans of its own
    U = sp.gen_uniform_random(3_500_000, 2)
    XY = [(torch.ones((U.N, k), dtype=torch.float64, device="cuda"),
           torch.empty((U.M, k), dtype=torch.float64, device="cuda")) for k in (2, 4)]
    resident = {"ragged": sp.CsrDevice.from_host(A), "empty": sp.CsrDevice.from_host(E)}

    def hll(make):                             # the handle and, from it, a SELL-P plan
        h = make()
        assert h.sell_info(build=True)["state"] == 1
        h.close()

    def sell(check):
        h = sp.CsrDevice.from_host(A)
        info = h.sell_info(build=True)
        assert info["state"] == 1 and check(info), info
        h.close()

    def spmm():
        h = sp.CsrDevice.from_host(U)
        assert h.sell_info(build=True)["panels"] == 1
        for X, Y in XY:
            h.spmm(X, Y)
            l0 = sp.counters()["launches"]
            h.spmm(X, Y)
            assert sp.counters()["launches"] - l0 > 1  # more panels than the SpMV plan: a plan of its own
        h.close()

    cases = []
    for name, M in (("ragged", A), ("empty", E)):
        for col_major in (False, True):
            H = sp.csr_to_hll(M, col_major)
            cases.append((f"hll {name} col_major={col_major}", {}, lambda H=H: hll(lambda: sp.HllDevice.from_host(H))))
        cases.append((f"hll {name} from csr", {}, lambda c=resident[name]: hll(c.to_hll)))
    cases += [
        # most rows of A fall in one length bin: the knob forces virtual rows, as it forces panels below
        ("sell virtual rows", {"sell": 1}, lambda: sell(lambda i: i["chunk"] == 256 and i["split_rows"] > 0)),
        ("sell panels", {"sell_panels": 2, "sell_max_row": 100},
         lambda: sell(lambda i: i["panels"] == 2 and i["chunk"] == 0 and i["long_rows"] > 0)),
        ("spmm plans", {"sell": 1, "sell_chunk": 0, "sell_panel_mb": 16}, spmm),
    ]
    try:
        for name, knobs, run in cases:
            for k, v in {**KNOB_DEFAULTS, **knobs}.items():
                sp.set_knob(k, v)
            run()                              # first use of every kernel involved (lazy module loading)
            torch.cuda.synchronize()
            free0 = torch.cuda.mem_get_info()[0]
            for _ in range(20):
                run()
            torch.cuda.synchronize()
            assert abs(torch.cuda.mem_get_info()[0] - free0) <= 2 << 20, name
    finally:
        for k, v in KNOB_DEFAULTS.items():
            sp.set_knob(k, v)
        for c in resident.values():
            c.close()
