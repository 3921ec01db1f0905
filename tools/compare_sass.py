"""Compare the SASS instruction streams of the kernels in two builds of one object file:

    python tools/compare_sass.py OLD/score_tc.o NEW/score_tc.o
    python tools/compare_sass.py OLD/select.o NEW/select.o

Kernels are matched by their demangled name without the anonymous namespace, the parameter list and an added
``bool = false`` template argument, so a kernel that gained a compile-time flag (and the parameters only its ``true``
instantiation reads) is compared with its old self; instruction offsets and encodings are ignored.  Prints
``identical`` / ``DIFFERENT`` per kernel of the old build and lists the kernels only the new build has.
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


def normalised(names):
    """{mangled name: key}: ``void xmve::<unnamed>::k<1, (bool)0>(...)`` -> ``xmve::k<1>``."""
    out = subprocess.run(["cu++filt"], input="\n".join(names), capture_output=True, text=True, check=True).stdout
    keys = {}
    for name, dem in zip(names, out.splitlines()):
        key = dem.replace("<unnamed>::", "").replace("(anonymous namespace)::", "")
        key = key.replace("(bool)0", "false").replace("(bool)1", "true")
        key = re.sub(r"\(\w+\)(-?\d+)", r"\1", key)                # (int)1 -> 1
        key = re.sub(r"^void ", "", key)
        key = re.sub(r"\(.*\)$", "", key)
        key = key.replace(", false>", ">").replace("<false>", "")
        keys[name] = key
    assert len(set(keys.values())) == len(keys), "two kernels share a key"
    return keys


def main():
    old, new = kernels(sys.argv[1]), kernels(sys.argv[2])
    key_old, key_new = normalised(list(old)), normalised(list(new))
    old = {key_old[k]: v for k, v in old.items()}
    new = {key_new[k]: v for k, v in new.items()}
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
