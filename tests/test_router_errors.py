"""Revert payloads of the two routers (no GPU): SelectorUnknown(bytes4) of RiscZeroVerifierRouter and RouteNotFound(bytes4) of
SP1VerifierGateway are the keccak-256 selector of the signature, then the record's bytes4 left-aligned in a 32-byte word."""
import pytest


def test_keccak_known_answers():
    from stylus_zkvm_verifiers_b200 import errors as E
    assert E.keccak256(b"").hex() == "c5d2460186f7233c927e7db2dcc703c0e500b653ca82273b7bfad8045d85a470"
    assert E.keccak256(b"transfer(address,uint256)")[:4].hex() == "a9059cbb"


@pytest.mark.parametrize("name, sig", [("SelectorUnknown", "SelectorUnknown(bytes4)"), ("RouteNotFound", "RouteNotFound(bytes4)")])
def test_router_error_payloads(name, sig):
    from stylus_zkvm_verifiers_b200 import errors as E
    cls = getattr(E, name)
    e = cls(b"\x9f\x39\x69\x6c")
    assert isinstance(e, E.VerifierError) and e.signature == sig and e.selector == b"\x9f\x39\x69\x6c"
    p = e.payload
    assert len(p) == 36 and p == e.abi_encode()
    assert p[:4] == E.keccak256(sig.encode())[:4]
    assert p[4:8] == b"\x9f\x39\x69\x6c" and p[8:] == bytes(28)
    assert cls(bytearray(b"\x00\x00\x00\x01")).payload[4:] == b"\x00\x00\x00\x01" + bytes(28)
