"""Differential pinning of the oracle restatement against the reference's upstream C engine, CPU only:
seeded samples of arbitrary byte strings as INPUT of Encode (identical bytes and return codes for every
capacity class) and as COMPRESSED STREAMS of Decode (identical accept/reject decision and length for
well-formed and malformed input alike), compared with that engine's recorded results
(tests/golden/ref_engine.npz)."""
from tests import inputs


def test_encode_port_equals_reference(port, ref):
    ref.check("fuzz_encode", *inputs.fuzz_encode_rows(port, port))


def test_decode_port_equals_reference_on_arbitrary_streams(port, ref):
    ref.check("fuzz_decode", *inputs.fuzz_decode_rows(port, port))     # offset-0 content is unspecified
