"""Compare the SASS instruction streams of the kernels in two builds of one object file:

    python tools/compare_sass.py OLD/score_tc.o NEW/score_tc.o
    python tools/compare_sass.py OLD/select.o NEW/select.o

Kernels are matched by name with the anonymous-namespace hash removed and an added ``bool = false`` template argument
dropped; instruction offsets and encodings are ignored.  Prints ``identical`` / ``DIFFERENT`` per kernel of the old
build and lists the kernels only the new build has.
"""
import re
import subprocess
import sys

FUNCTION = re.compile(r"Function : (\S+)")
# "        /*0040*/                   UTMALDG.2D [UR8], [UR4] ;   /* 0x...*/" -> "UTMALDG.2D [UR8], [UR4]"
INSTRUCTION = re.compile(r"\s*/\*[0-9a-f]{4,}\*/\s+(.*?)\s*;")


def kernels(obj):
    """{kernel name: [instruction text, ...]} of one object file."""
    out = subprocess.run(["cuobjdump", "-sass", obj], capture_output=True, text=True, check=True).stdout
    result, name = {}, None
    for line in out.splitlines():
        m = FUNCTION.search(line)
        if m:
            name = m.group(1)
            result[name] = []
            continue
        m = INSTRUCTION.match(line)
        if name is not None and m:
            result[name].append(m.group(1))
    return result


def normalised(name):
    name = re.sub(r"_GLOBAL__N__[0-9a-f]+_\d+_\w+?_cu_[0-9a-f]+", "", name)
    return name.replace("ELb0EEE", "EEE")


def main():
    old = {normalised(k): v for k, v in kernels(sys.argv[1]).items()}
    new = {normalised(k): v for k, v in kernels(sys.argv[2]).items()}
    different = 0
    for name in sorted(old):
        if name not in new:
            print("MISSING", name)
            different += 1
            continue
        same = old[name] == new[name]
        different += 0 if same else 1
        print("identical" if same else "DIFFERENT", len(old[name]), len(new[name]), name)
    print("new only:", sorted(k for k in new if k not in old))
    sys.exit(1 if different else 0)


if __name__ == "__main__":
    main()
