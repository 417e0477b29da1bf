"""
CPU tests: the RPC restatements (oracle/rpc_oracle.py, oracle/rpc_oracle.c) against known answers of
the compiled reference C (golden vectors; and oracle/_ref/disp_to_h.so itself when it was built).
"""
import numpy as np
import pytest

import util
from oracle import rpc_ctypes, rpc_oracle

R = util.load_rpc_golden()
RA, RB = util.rpc_from_array(R["rpc_a"]), util.rpc_from_array(R["rpc_b"])


def test_projection_bit_exact():
    lla = R["lonlatalt"]
    for rpc, key in ((RA, "ref_proj_a"), (RB, "ref_proj_b")):
        col, row = rpc.projection(lla[:, 0], lla[:, 1], lla[:, 2])
        assert np.array_equal(np.stack((col, row), axis=1), R[key])
    port = rpc_ctypes.load_port()
    for rpc, key in ((RA, "ref_proj_a"), (RB, "ref_proj_b")):       # the C port against the compiled reference's output
        assert np.array_equal(rpc_ctypes.port_project(port, rpc, lla), R[key]), key


def test_localization_bit_exact():
    cra = R["colrowalt"]
    port = rpc_ctypes.load_port()
    assert np.array_equal(rpc_ctypes.port_localize(port, RA, cra, delta=1.0), R["ref_loc_a_delta1"])
    assert np.array_equal(rpc_ctypes.port_localize(port, RA, cra, delta=0.1), R["ref_loc_a_delta01"])
    lon, lat = RA.localization(cra[:, 0], cra[:, 1], cra[:, 2], delta=1.0)
    assert np.array_equal(np.stack((lon, lat), axis=1), R["ref_loc_a_delta1"])
    # localisation inverts projection
    col, row = RA.projection(lon, lat, cra[:, 2])
    assert np.abs(col - cra[:, 0]).max() < 1e-5 and np.abs(row - cra[:, 1]).max() < 1e-5


def test_triangulation_bit_exact():
    port = rpc_ctypes.load_port()
    out, err = rpc_ctypes.triangulate(port, RA, RB, R["kp_a"], R["kp_b"], delta=0.1)
    assert np.array_equal(out, R["ref_tri_lonlatalt"])
    assert np.array_equal(err, R["ref_tri_err"])


def test_against_compiled_reference_if_present():
    ref = rpc_ctypes.load_ref()
    if ref is None:
        pytest.skip("oracle/_ref/disp_to_h.so not built (no reference tree)")
    rng = np.random.default_rng(9)
    n = 300
    lla = np.stack([RA.lon_offset + rng.uniform(-.03, .03, n), RA.lat_offset + rng.uniform(-.03, .03, n),
                    RA.alt_offset + rng.uniform(-500, 500, n)], axis=1)
    port = rpc_ctypes.load_port()
    assert np.array_equal(rpc_ctypes.ref_project(ref, RB, lla), rpc_ctypes.port_project(port, RB, lla))
    pa, pb = rpc_ctypes.port_project(port, RA, lla), rpc_ctypes.port_project(port, RB, lla)
    o_ref, e_ref = rpc_ctypes.triangulate(ref, RA, RB, pa, pb, ref=True)
    o_port, e_port = rpc_ctypes.triangulate(port, RA, RB, pa, pb)
    assert np.array_equal(o_ref, o_port) and np.array_equal(e_ref, e_port)
    assert np.abs(o_ref[:, 2] - lla[:, 2]).max() < 0.01      # float32 keypoints -> mm-level height noise


def test_rpc_file_round_trip(tmp_path):
    f = tmp_path / "a.rpc"
    RA.write_to_file(str(f))
    r2 = rpc_oracle.RPCModel.from_file(str(f))
    assert np.allclose(util.rpc_from_array(R["rpc_a"]).col_num, r2.col_num)
    assert abs(r2.lat_offset - RA.lat_offset) < 1e-11
