"""Lane-major offsets of coded block-rows (DESIGN.md §3): a coded block-row with n = 4a + 2b + c stored planes keeps
its 64 n bytes of 16-bit offsets as a chunks of 256 B (8 B per lane), then a 128-B chunk (4 B per lane) if b, then a
64-B chunk (2 B per lane) if c.  The block reader decodes the masks of the structured beam with compile-time registers
and every other mask on a generic path.  Every case here is compared bit for bit with the numpy reference or with the
all-raw layout (SAA_VALUE_CODE=0), through the host and the device set-up paths."""
import numpy as np
import pytest
import scipy.sparse as sp

import saa_b200  # noqa: F401
from saa_b200 import plan as splan
from util import bits_equal
from test_gpu_format_conformance import check_plan, device_plan, host_plan, references
from test_gpu_value_coding import coded_model

pytestmark = pytest.mark.gpu

SPECIALISED = (0x1FF, 0x0EE)                          # the coded masks of the structured beam
# every n = 1 .. 9 (so every split 4a + 2b + c), the specialised masks and masks of the generic path for the same n
STEP_MASKS = (0x010, 0x001, 0x011, 0x180, 0x111, 0x007, 0x0F0, 0x11F, 0x0EE, 0x03F, 0x1F5, 0x07F, 0x1FE, 0x0FF, 0x1FF)


def _bits(x):
    return np.asarray(x, dtype=np.float64).view(np.int64)


def _from_bits(b):
    return np.asarray(b, dtype=np.int64).view(np.float64)


def _plane_value(A, B, lane, symmetric):
    """a plane whose 32 lanes span a few ulps: coded unless a case below says otherwise"""
    if A == B:
        return _from_bits(_bits(2.0e3 + 100.0 * A) + lane)
    if symmetric:
        A, B = min(A, B), max(A, B)
    return _from_bits(_bits(-3.0e2 - 10.0 * (3 * A + B)) + (lane % 7))


def _problem(slices, n_last=32, symmetric=False, seed=5):
    """one 3x3 block per node (its own); slice s stores the planes of masks[s] in every lane, with plane values from
    overrides[s] = {plane: 32 bit patterns} where given"""
    nn = 32 * (len(slices) - 1) + n_last
    rows, cols, data = [], [], []
    for e in range(nn):
        s, l = divmod(e, 32)
        mask, over = slices[s]
        for A in range(3):
            for B in range(3):
                p = 3 * A + B
                if not (mask >> p) & 1:
                    continue
                v = _from_bits(over[p][l]) if p in over else _plane_value(A, B, l, symmetric)
                rows.append(3 * e + A), cols.append(3 * e + B), data.append(v)
    n = 3 * nn
    K = sp.csr_matrix((np.array(data), (np.array(rows), np.array(cols))), shape=(n, n))
    K.sort_indices()
    assert K.nnz == len(data)                          # stored zeros are kept
    rng = np.random.default_rng(seed)
    return dict(K=K, F=rng.standard_normal(n), lM=1.0 + rng.random(n), dirichlet=np.array([4, 100], dtype=np.int64),
                dt=1e-3, alpha=0.3, d0=1e-3 * rng.standard_normal(n), dn=1e-3 * rng.standard_normal(n), tn0=0.5,
                rows=np.repeat(np.arange(n), np.diff(K.indptr)), cols=K.indices.astype(np.int64), vals=K.data,
                n_nodes=nn, family="lane_major_offsets")


def step_problem():
    """STEP_MASKS, one slice each, all coded; then the coding boundary on plane (0,1): span 65535 (coded, 0x1FF and
    0x0EE) and 65536 (raw); +0.0 with subnormals and -0.0 with negative subnormals in a stored plane (coded); and a
    last slice of 28 nodes whose padding lanes hold +0.0 (raw)"""
    lane = np.arange(32)
    lo = _bits(1.0e3)
    span = lambda w: {1: lo + (lane * w) // 31}
    slices = [(m, {}) for m in STEP_MASKS]
    slices += [(0x1FF, span(65535)), (0x0EE, span(65535)), (0x1FF, span(65536)), (0x07F, span(65536)),
               (0x0EE, {1: np.where(lane % 3 == 0, 0, lane)}),
               (0x03F, {1: np.where(lane % 3 == 0, _bits(-0.0), _bits(-0.0) + lane)}),
               (0x111, {4: np.where(lane % 2 == 0, 0, 3 * lane)}),
               (0x1F5, {})]
    return _problem(slices, n_last=28)


def _counters(pl):
    return dict(value_planes=pl.value_planes, coded_planes=pl.coded_planes, streamed_matrix_bytes=pl.streamed_matrix_bytes)


@pytest.mark.parametrize("variant", [0, 1, 2, 3, 4, 5])
def test_every_split_and_mask_equals_reference(monkeypatch, variant):
    prob = step_problem()
    model = coded_model(prob["K"])
    raw_planes = 9 + 7 + 7                            # the 65536 spans and the padded last slice
    assert model["coded_planes"] == model["value_planes"] - raw_planes
    refs = references(prob)
    monkeypatch.setenv("SAA_KVARIANT", str(variant))
    monkeypatch.setenv("SAA_STEP_HOST_PIPELINE", "5")
    for setup in (host_plan, device_plan):
        pl = setup(prob)
        assert _counters(pl) == model, setup.__name__
        check_plan(pl, prob, refs, variant, (variant, setup.__name__))


def test_cg_diag_reads_lane_major_offsets(monkeypatch):
    """block-Jacobi CG on a block-diagonal SPD matrix: the diagonal blocks come from saa_load_block_lane, one lane at a
    time, for coded masks with n = 3, 5, 7, 9 (h and t, q0 and t, q0, h and t, q0, q1 and t)"""
    masks = (0x111, 0x11B, 0x155, 0x1B1, 0x15F, 0x1F5, 0x1BB, 0x1FF)
    prob = _problem([(m, {}) for m in masks], symmetric=True)
    K = prob["K"]
    assert abs(K - K.T).max() == 0.0
    for setup in (host_plan, device_plan):
        monkeypatch.setenv("SAA_VALUE_CODE", "0")
        raw = setup(prob)
        monkeypatch.delenv("SAA_VALUE_CODE")
        coded = setup(prob)
        assert raw.coded_planes == 0 and coded.coded_planes == coded.value_planes == sum(bin(m).count("1") for m in masks)
        res = [pl.solve_static(rtol=1e-12) for pl in (raw, coded)]
        assert res[0].converged and res[0].iterations == res[1].iterations
        assert bits_equal(res[0].x.cpu().numpy(), res[1].x.cpu().numpy())
        x = np.asarray(res[1].x.cpu().numpy())
        free = np.setdiff1d(np.arange(K.shape[0]), prob["dirichlet"])
        r = (K @ x - prob["F"])[free]
        assert np.abs(r).max() <= 1e-8 * np.abs(prob["F"]).max()
