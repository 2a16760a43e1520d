"""Which solve-kernel specialisation a solve launches (enqueue_solve's selection rule), read from the kernel names
torch.profiler records.  Batch sizes are multiples of the SM count, so that choose_pb settles on the intended lanes
per CTA (PB); the expected PB is part of each row.  The hard-first queue order (queue_order_kernel) runs exactly when
the option is on and the batch does not fit the grid's lanes at once."""
import numpy as np
import pytest

from mpc_ros_b200 import capi
from oracle.oracle_py import YAML_DEFAULT, CFG_DEFAULT
from tests.problems import mild

pytestmark = pytest.mark.gpu


def _k(spt, cpb, warm, rate, nc=4):
    b = lambda x: "true" if x else "false"
    return "nmpc_solve_kernel<%d, %d, %s, %s, %d>" % (spt, cpb, b(warm), b(rate), nc)


def _dual(warm, rate):
    return "nmpc_solve_kernel_dual<%s, 4, %s>" % ("true" if warm else "false", "true" if rate else "false")


# (id, weights, N, batch in units of the SM count, options, warm, PB, expected kernel)
ROWS = [
    ("yaml-full-cold", YAML_DEFAULT, 20, 40, {}, False, 32, _dual(False, False)),
    ("yaml-full-warm", YAML_DEFAULT, 20, 40, {}, True, 32, _dual(True, False)),
    ("yaml-full-unordered", YAML_DEFAULT, 20, 40, {"hard_first": 0}, False, 32, _dual(False, False)),
    ("yaml-full-single-cold", YAML_DEFAULT, 20, 40, {"dual_groups": 0}, False, 32, _k(2, 32, False, False)),
    ("yaml-full-single-warm", YAML_DEFAULT, 20, 40, {"dual_groups": 0}, True, 32, _k(2, 32, True, False)),
    ("cfg-full-cold", CFG_DEFAULT, 20, 36, {}, False, 28, _dual(False, True)),
    ("cfg-full-warm", CFG_DEFAULT, 20, 36, {}, True, 28, _dual(True, True)),
    ("cfg-full-single-cold", CFG_DEFAULT, 20, 36, {"dual_groups": 0}, False, 28, _k(2, 28, False, True)),
    ("cfg-full-single-warm", CFG_DEFAULT, 20, 36, {"dual_groups": 0}, True, 28, _k(2, 28, True, True)),
    ("cfg-small-cold", CFG_DEFAULT, 20, 10, {}, False, 10, _k(2, 0, False, True)),
    ("cfg-small-warm", CFG_DEFAULT, 20, 10, {}, True, 10, _k(2, 0, True, True)),
]
for _pb in (16, 8, 4, 1):
    ROWS += [
        ("narrow%d-cold" % _pb, YAML_DEFAULT, 20, _pb, {}, False, _pb, _k(1, _pb, False, False)),
        ("narrow%d-warm" % _pb, YAML_DEFAULT, 20, _pb, {}, True, _pb, _k(1, _pb, True, False)),
        ("narrow%d-two-stage" % _pb, YAML_DEFAULT, 20, _pb, {"narrow_one_stage": 0}, False, _pb, _k(2, _pb, False, False)),
    ]
ROWS += [
    # only the 32-lane warm kernel is specialised: a warm two-stage solve in narrower CTAs runs the generic one
    ("narrow16-two-stage-warm", YAML_DEFAULT, 20, 16, {"narrow_one_stage": 0}, True, 16, _k(2, 0, True, False)),
    # 64 + 30 * 16 threads exceed the one-stage kernel's bound at 16 lanes: two stages per stage thread
    ("N30-pb16", YAML_DEFAULT, 30, 16, {}, False, 16, _k(2, 16, False, False)),
    # the dual-group kernel starts at N = 11
    ("N10-full", YAML_DEFAULT, 10, 40, {}, False, 32, _k(2, 32, False, False)),
    ("N100-cold", YAML_DEFAULT, 100, 12, {}, False, 6, _k(2, 6, False, False)),
    ("N100-warm", YAML_DEFAULT, 100, 12, {}, True, 6, _k(2, 0, True, False)),
    ("nc6-cold", YAML_DEFAULT, 20, 4, {"poly_coeffs": 6}, False, 4, _k(2, 0, False, False, 8)),
    ("nc6-rate-warm", CFG_DEFAULT, 20, 4, {"poly_coeffs": 6}, True, 4, _k(2, 0, True, True, 8)),
    ("pb7", YAML_DEFAULT, 20, 14, {"problems_per_cta": 7}, False, 7, _k(2, 0, False, False)),
]


@pytest.fixture(scope="module")
def torch_dev():
    torch = pytest.importorskip("torch")
    torch.cuda.init()
    return torch


def _kernels(fn):
    """names of the kernels fn launches (the part after 'nmpc::' / before the argument list)"""
    from torch.profiler import profile, ProfilerActivity
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        fn()
    names = [e.name for e in prof.events()]
    return [n.split("(")[0].split("::")[-1] for n in names if "nmpc_solve_kernel" in n or "queue_order_kernel" in n]


@pytest.mark.parametrize("row", ROWS, ids=[r[0] for r in ROWS])
def test_solve_kernel_choice(torch_dev, row):
    _, weights, N, per_sm, opts, warm, pb, expect = row
    sms = torch_dev.cuda.get_device_properties(0).multi_processor_count
    B = per_sm * sms
    prm = capi.params_from_map(dict(weights, STEPS=N), capi.yaml_default_params())
    prm.max_iter = 3
    sv = capi.Solver(prm, B, 0)
    for k, v in opts.items():
        sv.set_option(k, v)
    state, c4 = mild(5, B)
    coeffs = np.zeros((sv.nc, B)); coeffs[:4] = c4
    ws = capi.lib().mpc_b200_warm_size(N)
    u0 = np.zeros((2, B)); pred = np.zeros((3 * N, B)); rec = np.zeros((ws, B))
    warm_in = None
    if warm:
        sv.solve_raw(B, state, coeffs, u0, pred, warm_out=rec)
        warm_in = rec
    got = _kernels(lambda: sv.solve_raw(B, state, coeffs, u0, pred, warm_in=warm_in))
    sv.close()
    solves = [n for n in got if n.startswith("nmpc_solve_kernel")]
    assert solves == [expect], got
    grid = min((B + pb - 1) // pb, sms)
    ordered = opts.get("hard_first", 1) != 0 and B > grid * pb
    assert got.count("queue_order_kernel") == (1 if ordered else 0), got
