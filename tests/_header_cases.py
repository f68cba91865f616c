"""The header shapes of tests/test_headers.py and how a text-layer process_headers (xm.py:36-46, 120-174) answers them.
Plain Python: tests/golden/make_header_golden.py uses it without pytest or the library."""
import io

REC = "r1\t0\tchr1\t1\t42\t5M\t*\t0\t0\tACGTA\tFFFFF\tAS:i:10\n"
H1 = "@HD\tVN:1.0\tSO:unsorted\n@SQ\tSN:chr1\tLN:1000\n@PG\tID:bowtie2\tPN:bowtie2\tVN:2.2.6\tCL:\"bowtie2-align-s --local\"\n"
H2 = "@HD\tVN:1.0\n@SQ\tSN:1\tLN:500\n"
NAMES = ("primary_specific", "secondary_specific", "primary_multi", "secondary_multi", "unassigned", "unresolved")
ENABLED = {"all": 0x3F, "primary_specific_only": 0x01, "primary_bins": 0x15}

CASES = {
    "plain": (H1 + REC, H2 + REC),
    "crlf": ((H1 + REC).replace("\n", "\r\n"), H2 + REC),
    "lone_cr_in_header": (H1.replace("\n", "\r") + REC, H2 + REC),
    "no_header": (REC, H2 + REC),
    "empty": ("", H2 + REC),
    "header_only": (H1, H2 + REC),
    "blank_line_after_header": (H1 + "\n" + REC, H2 + REC),
    "pg_without_id": (H1, "@HD\tVN:1.0\n@PG\tPN:bowtie2\n" + REC),
    "pg_id_after_unicode_space": (H1 + REC, "@HD\tVN:1.0\n@PG\tPN:x ID:abc VN:1\n" + REC),
    "pg_not_last": (H1 + "@CO\tsomething\n" + REC, H2 + REC),
    "non_ascii_header": (H1 + REC, "@CO\tnaïve café\n" + REC),
    "secondary_header_only": (H1 + REC, H2),
}


def key(name, enabled):
    return "%s|0x%02x" % (name, enabled)


def text_layer(module, text1, text2, enabled):
    """(exception class name or None, six header strings, remaining text of both inputs) from a text-layer implementation"""
    f1, f2 = io.StringIO(text1, newline=None), io.StringIO(text2, newline=None)
    outs = {n: (io.StringIO() if (enabled >> b) & 1 or b == 0 else None) for b, n in enumerate(NAMES)}
    try:
        module.process_headers(f1, f2, **outs)
    except Exception as e:                                       # noqa: BLE001 -- the class is what is compared
        return type(e).__name__, None, None
    return None, [outs[n].getvalue() if outs[n] else None for n in NAMES], [f1.read(), f2.read()]
