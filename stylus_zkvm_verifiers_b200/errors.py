"""Revert payloads of the reference, rebuilt from the per-proof status byte (SURVEY.md section 8f-1).

The reference's `verify` / `verify_proof` return `Err(Vec<u8>)` holding an ABI-encoded Solidity custom
error (/root/reference/contracts/src/common/errors.rs:3-26, risc0/errors.rs:8-32, sp1/errors.rs:8-32).
`abi_encode()` of a custom error is keccak256(signature)[:4] followed by the arguments, each padded to
32 bytes (bytes4 is left-aligned).  Keccak-256 is implemented here because hashlib's sha3_256 uses a
different padding.
"""

_RC = [0x0000000000000001, 0x0000000000008082, 0x800000000000808A, 0x8000000080008000, 0x000000000000808B, 0x0000000080000001,
       0x8000000080008081, 0x8000000000008009, 0x000000000000008A, 0x0000000000000088, 0x0000000080008009, 0x000000008000000A,
       0x000000008000808B, 0x800000000000008B, 0x8000000000008089, 0x8000000000008003, 0x8000000000008002, 0x8000000000000080,
       0x000000000000800A, 0x800000008000000A, 0x8000000080008081, 0x8000000000008080, 0x0000000080000001, 0x8000000080008008]
_ROT = [[0, 36, 3, 41, 18], [1, 44, 10, 45, 2], [62, 6, 43, 15, 61], [28, 55, 25, 21, 56], [27, 20, 39, 8, 14]]
_M = (1 << 64) - 1


def _rol(x, n):
    return ((x << n) | (x >> (64 - n))) & _M if n else x


def keccak256(data: bytes) -> bytes:
    rate = 136
    msg = bytearray(data) + b"\x01" + bytes((-len(data) - 2) % rate) + b"\x80" if (len(data) + 1) % rate else bytearray(data) + b"\x81"
    a = [[0] * 5 for _ in range(5)]
    for off in range(0, len(msg), rate):
        for i in range(rate // 8):
            a[i % 5][i // 5] ^= int.from_bytes(msg[off + 8 * i:off + 8 * i + 8], "little")
        for rnd in range(24):
            c = [a[x][0] ^ a[x][1] ^ a[x][2] ^ a[x][3] ^ a[x][4] for x in range(5)]
            d = [c[(x - 1) % 5] ^ _rol(c[(x + 1) % 5], 1) for x in range(5)]
            a = [[a[x][y] ^ d[x] for y in range(5)] for x in range(5)]
            b = [[0] * 5 for _ in range(5)]
            for x in range(5):
                for y in range(5):
                    b[y][(2 * x + 3 * y) % 5] = _rol(a[x][y], _ROT[x][y])
            a = [[b[x][y] ^ ((~b[(x + 1) % 5][y]) & b[(x + 2) % 5][y]) for y in range(5)] for x in range(5)]
            a[0][0] ^= _RC[rnd]
    out = b"".join(a[i % 5][i // 5].to_bytes(8, "little") for i in range(4))
    return out


def _sel(sig):
    return keccak256(sig.encode())[:4]


class VerifierError(Exception):
    """Base class; `payload` is the byte string the reference would return in `Err(..)`."""
    signature = ""

    def __init__(self, *args4):
        self.args4 = args4
        self.payload = _sel(self.signature) + b"".join(a + bytes(28) for a in args4)
        super().__init__(self.signature)

    def abi_encode(self):
        return self.payload


class VerificationFailed(VerifierError):
    signature = "VerificationFailed()"          # common/errors.rs:4


class InvalidInitialization(VerifierError):
    signature = "InvalidInitialization()"       # common/errors.rs:5


class AlreadyInitialized(VerifierError):
    signature = "AlreadyInitialized()"          # common/errors.rs:6


class InvalidProofData(VerifierError):
    signature = "InvalidProofData()"            # common/errors.rs:7


class SelectorMismatch(VerifierError):
    signature = "SelectorMismatch(bytes4,bytes4)"       # risc0/errors.rs:9

    def __init__(self, received, expected):
        super().__init__(bytes(received), bytes(expected))
        self.received, self.expected = bytes(received), bytes(expected)


class WrongVerifierSelector(VerifierError):
    signature = "WrongVerifierSelector(bytes4,bytes4)"  # sp1/errors.rs:9

    def __init__(self, received, expected):
        super().__init__(bytes(received), bytes(expected))
        self.received, self.expected = bytes(received), bytes(expected)


class SelectorUnknown(VerifierError):
    signature = "SelectorUnknown(bytes4)"               # RiscZeroVerifierRouter: no verifier registered under the seal's selector

    def __init__(self, selector):
        super().__init__(bytes(selector))
        self.selector = bytes(selector)


class RouteNotFound(VerifierError):
    signature = "RouteNotFound(bytes4)"                 # SP1VerifierGateway: no route for the proof's selector

    def __init__(self, selector):
        super().__init__(bytes(selector))
        self.selector = bytes(selector)
