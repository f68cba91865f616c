"""Header processing inside the library (csrc/xm_headers.h: xm_process_headers_fds / _mem) against the reference's
get_sam_header / add_pg_tag / process_headers (xm.py:36-46, 120-174): same six header texts, same errors, and the byte
offset of the first record.  The text layer's answers are stored in tests/golden/headers.json
(tests/golden/make_header_golden.py); the package's Python text path must still give them too."""
import json
import os

import pytest

from tests._header_cases import CASES, ENABLED, H1, H2, NAMES, REC, key, text_layer
from xenomapper_b200 import _lib
from xenomapper_b200 import xenomapper as xm

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "headers.json")


def expected(name, enabled):
    """the stored answer of the text layer; the package's Python text path (StringIO inputs never take the native
    route) must give the same"""
    with open(GOLDEN, encoding="utf-8") as f:
        a = json.load(f)["answers"][key(name, enabled)]
    want = a["error"], a["headers"], a["rest"]
    assert text_layer(xm, *CASES[name], enabled) == want, "the Python text layer no longer gives the stored answer"
    return want


@pytest.mark.parametrize("enabled", list(ENABLED.values()), ids=list(ENABLED))
@pytest.mark.parametrize("name", list(CASES))
def test_native_headers_match_the_text_layer(tmp_path, name, enabled):
    t1, t2 = CASES[name]
    err, texts, rest = expected(name, enabled)
    b1, b2 = t1.encode(), t2.encode()
    for route in ("mem", "fds"):
        if route == "mem":
            rc, bad, offs, got, status = _lib.process_headers(b1, b2, "1.0.2")
        else:
            for k, b in enumerate((b1, b2)):
                open(tmp_path / ("h%d.sam" % k), "wb").write(b)
            fds = [os.open(tmp_path / ("h%d.sam" % k), os.O_RDONLY) for k in range(2)]
            rc, bad, offs, got, status = _lib.process_headers(fds[0], fds[1], "1.0.2")
            [os.close(f) for f in fds]
        first_error = None
        if rc == _lib.XM_ERR_INDEX:
            first_error = "IndexError"
        elif rc == _lib.XM_ERR_UNICODE:
            first_error = "UnicodeDecodeError"
        else:
            assert rc == 0
            for b in range(6):
                if ((enabled >> b) & 1 or b == 0) and status[b] == _lib.XM_ERR_INDEX:
                    first_error = "IndexError"
                    break
        assert first_error == err, (route, rc, status)
        if err is None:
            for b in range(6):
                if texts[b] is not None:
                    assert got[b].decode() == texts[b], (route, NAMES[b])
            # the first record starts where the text layer left its file: compare what is left, newline-normalised
            for k, (raw, left) in enumerate(zip((b1, b2), rest)):
                assert raw[offs[k]:].decode().replace("\r\n", "\n").replace("\r", "\n") == left


def test_invalid_utf8_in_the_header_is_a_decode_error():
    rc, bad, *_ = _lib.process_headers(b"@HD\tVN:1.0\n@CO\t\xff\xfe\n" + REC.encode(), (H2 + REC).encode(), "1.0.2")
    assert rc == _lib.XM_ERR_UNICODE and bad == 0


def test_header_longer_than_the_first_read(tmp_path):
    """xm_process_headers_fds reads 64 KiB first and widens until the header ends"""
    big = "".join("@SQ\tSN:contig%06d\tLN:%d\n" % (k, 1000 + k) for k in range(9000))          # ~260 KB
    open(tmp_path / "a.sam", "w").write(big + REC)
    open(tmp_path / "b.sam", "w").write(H2 + REC)
    fa, fb = os.open(tmp_path / "a.sam", os.O_RDONLY), os.open(tmp_path / "b.sam", os.O_RDONLY)
    rc, bad, offs, got, status = _lib.process_headers(fa, fb, "1.0.2")
    os.close(fa); os.close(fb)
    assert rc == 0 and offs == [len(big), len(H2)]
    assert got[0].decode() == big + "@PG\tID:Xenomapper\tPN:Xenomapper\tVN:1.0.2\n@CO\tspecies specific reads\n"


def test_process_headers_on_real_files_takes_the_native_route(tmp_path):
    """the module-level process_headers: real files at their start go through the library, are left at their first
    record, and main_* then hands descriptors + byte offsets over without consulting tell() cookies"""
    open(tmp_path / "p.sam", "w").write(H1 + REC)
    open(tmp_path / "s.sam", "w").write(H2 + REC)
    out = open(tmp_path / "o.sam", "w+")
    with open(tmp_path / "p.sam") as f1, open(tmp_path / "s.sam") as f2:
        xm.process_headers(f1, f2, primary_specific=out)
        assert xm._RECORD_OFFSET[f1] == len(H1) and xm._RECORD_OFFSET[f2] == len(H2)
        assert f1.readline() == REC and f2.readline() == REC
    out.seek(0)
    assert out.read() == H1 + "@PG\tID:Xenomapper\tPN:Xenomapper\tPP:bowtie2\tVN:1.0.2\n@CO\tspecies specific reads\n"
