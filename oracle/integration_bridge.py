"""TEST INFRASTRUCTURE ONLY — type-checks the bridge shown in INTEGRATION.md against the reference's own headers.

Run by oracle/Makefile (target ref) where the reference sources are, next to the build of the reference binary:
    python3 integration_bridge.py <reference src dir> <result file>
The result file holds digest() of what was checked and the compiler's exit code on its first line, then
the compiler's diagnostics; tests/test_abi.py holds the current INTEGRATION.md to it.
"""
import hashlib
import os
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def bridge_source():
    """INTEGRATION.md's first ```cpp block inside namespace chromap, after the reference headers it uses and include/chromap_b200.h."""
    md = open(os.path.join(ROOT, "INTEGRATION.md")).read()
    a = md.index("```cpp") + 6
    code = md[a:md.index("```", a)].replace('#include "chromap_b200.h"', "")
    return ("#include <cstdint>\n#include <string>\n#include <vector>\n#include \"mapping_parameters.h\"\n#include \"sequence_batch.h\"\n"
            "#include \"bed_mapping.h\"\n#include \"utils.h\"\n#include \"chromap_b200.h\"\nnamespace chromap {\n" + code + "\n}\nint main() { return 0; }\n")


def digest():
    """sha256 of what the check depends on in this repository: the translation unit and include/chromap_b200.h."""
    return hashlib.sha256((bridge_source() + open(os.path.join(ROOT, "include", "chromap_b200.h")).read()).encode()).hexdigest()


def main(ref_src, out):
    src = bridge_source()
    with tempfile.TemporaryDirectory() as d:
        p = os.path.join(d, "bridge.cc")
        with open(p, "w") as f:
            f.write(src)
        r = subprocess.run(["/usr/bin/g++", "-std=c++11", "-fsyntax-only", "-I" + ref_src, "-I" + os.path.join(ROOT, "include"), p],
                           capture_output=True, text=True)
    with open(out, "w") as f:
        f.write("%s %d\n%s" % (digest(), r.returncode, r.stderr[:2000]))


if __name__ == "__main__":
    main(sys.argv[1], sys.argv[2])
