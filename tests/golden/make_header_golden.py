#!/usr/bin/env python3
"""Write tests/golden/headers.json: what the SAM text layer's process_headers (xm.py:36-46, 120-174) gives for every header
case of tests/test_headers.py -- the exception class, the six header texts and the text left in both inputs.

    python tests/golden/make_header_golden.py [REFERENCE_SOURCE_TREE]

Given the source tree of the unmodified reference, the answers come from the reference itself; without it, from the
package's Python mirror of the same functions (xenomapper_b200/xenomapper.py, whose header bytes tests/test_host_shim.py
checks against the reference's goldens).  The file records which of the two produced it.
"""
import json
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)

from tests._header_cases import CASES, ENABLED, key, text_layer  # noqa: E402


def main():
    if len(sys.argv) > 1:
        sys.path.insert(0, sys.argv[1])
        from xenomapper import xenomapper as module
        source = "the unmodified reference, version %s" % module.__version__
    else:
        from xenomapper_b200 import xenomapper as module
        source = "xenomapper_b200/xenomapper.py, the package's mirror of the reference's text layer (version %s)" % module.__version__
    answers = {}
    for name, (t1, t2) in CASES.items():
        for enabled in ENABLED.values():
            err, texts, rest = text_layer(module, t1, t2, enabled)
            answers[key(name, enabled)] = dict(error=err, headers=texts, rest=rest)
    with open(os.path.join(HERE, "headers.json"), "w") as f:
        json.dump(dict(source=source, answers=answers), f, indent=0, sort_keys=True, ensure_ascii=False)
        f.write("\n")
    print("wrote %d answers from %s" % (len(answers), source))


if __name__ == "__main__":
    main()
