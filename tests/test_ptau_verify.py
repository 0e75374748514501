"""`powersoftau verify` on the GPU (csrc/ptau_verify.cu).

The device report, records and claims must equal the host hook's byte for byte at powers <= 4 with the same seed; every
tampered file of the CPU tests must give its message at power 10, on a chain built on the device; and a power-22
ceremony built in the library (contribute, contribute, beacon, prepare) must verify, with one tampered point past the
first 2^22-point MSM chunk of section 2 and one on the top level of section 12 caught.
"""
import pytest

from nzcp_circom_b200 import api, groth16
from oracle import formats
from oracle.bn254 import G1, g1_from_bytes_mont, g1_to_bytes_mont
from test_ptau_verify_cpu import VSEED, _Log, chain, get_chain, raw, tampered

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("power,prepared", [(1, True), (2, False), (3, True), (4, True), (4, False)])
def test_device_equals_host(lib, power, prepared):
    buf = get_chain(power, prepared)[0]
    assert raw(buf, VSEED, device=0) == raw(buf, VSEED)
    assert api.ptau_verify(buf, seed=VSEED)["ok"]


def test_device_equals_host_on_tampered(lib):
    buf = get_chain(2, True)[0]
    for name, bad, _ in tampered(buf, 2):
        assert raw(bad, VSEED, device=0) == raw(bad, VSEED), name


def test_power10_tampered(lib):
    buf, hashes = chain(10, True, host=False)
    timings, log = {}, _Log()
    res = api.ptau_verify(buf, timings=timings)
    assert res["ok"], res["message"]
    assert [c["response_hash"] for c in res["contributions"]] == hashes
    assert sorted(timings) == sorted(api.PTAU_VERIFY_TIMINGS + ("pairings",)) and all(t >= 0 for t in timings.values())
    assert groth16.powersOfTau.verify(buf, log)
    assert ("info", "Powers of Tau Ok!") in log.lines and not any(lvl == "warn" for lvl, _ in log.lines)
    for name, bad, msg in tampered(buf, 10):
        res = api.ptau_verify(bad, seed=VSEED)
        assert not res["ok"] and res["message"] == msg, (name, res["message"])


def _double_point(buf, sid, idx):
    """The file with G1 point idx of section sid doubled (in place in a copy)."""
    _, secs = formats.read_container(buf, b"ptau")
    off = secs[sid][0][0] + 64 * idx
    out = bytearray(buf)
    out[off:off + 64] = g1_to_bytes_mont(G1.mul(g1_from_bytes_mont(bytes(out[off:off + 64])), 2))
    return bytes(out)


def test_power22_ceremony(lib):
    """Section 2 has 2^23 - 1 points and section 12 2^24 - 1: both MSMs cross the 2^22-base chunk."""
    buf, hashes = chain(22, True, host=False)
    res = api.ptau_verify(buf)
    assert res["ok"], res["message"]
    assert res["prepared"] and [c["response_hash"] for c in res["contributions"]] == hashes
    bad2 = _double_point(buf, 2, (1 << 22) + 12345)
    res = api.ptau_verify(bad2)
    assert not res["ok"] and res["message"] == "tauG1 section. Powers do not match"
    del bad2
    top = (1 << 23) - 1                      # level 23 (power + 1) of section 12 starts at point 2^23 - 1
    bad12 = _double_point(buf, 12, top + (1 << 22) + 777)
    res = api.ptau_verify(bad12)
    assert not res["ok"] and res["message"] == "Phase2 caclutation does not match with powers of tau"
    groth16.terminate()
