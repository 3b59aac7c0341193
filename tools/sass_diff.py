"""Compare the kernels of two builds of the CUDA library instruction by instruction.

    python tools/sass_diff.py OLD.so NEW.so

Runs `cuobjdump -sass` on both libraries, keeps each kernel's instructions without their addresses and encodings,
and matches kernels by (mangled) name, whichever translation unit holds them.  Prints one line per kernel -- same,
DIFFERENT (with the first differing instruction), or present in only one library -- then a total, and exits 1 on
any difference.  A change that only moves or restructures host code must leave every kernel the same.
Needs no GPU."""
import os
import re
import subprocess
import sys

CUOBJDUMP = os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "bin", "cuobjdump")
FUNC = re.compile(r"^\s*Function : (\S+)")
INSTR = re.compile(r"^\s*/\*[0-9a-f]{4,}\*/\s+(.*?)\s*;")     # "/*0040*/  IMAD R1, ... ;  /* 0x... */"


def kernels(lib):
    """{kernel name: [instruction text, ...]} of every kernel in `lib`."""
    out = subprocess.run([CUOBJDUMP, "-sass", lib], capture_output=True, text=True, check=True).stdout
    found, name = {}, None
    for line in out.splitlines():
        m = FUNC.match(line)
        if m:
            name = m.group(1)
            if name in found:
                raise SystemExit(f"{lib}: kernel {name} appears twice")
            found[name] = []
            continue
        m = INSTR.match(line)
        if m and name is not None:
            found[name].append(re.sub(r"\s+", " ", m.group(1)))
    return found


def main(argv):
    if len(argv) != 3:
        raise SystemExit(__doc__)
    old, new = kernels(argv[1]), kernels(argv[2])
    differing = 0
    for name in sorted(set(old) | set(new)):
        if name not in new:
            print(f"ONLY OLD   {name}")
        elif name not in old:
            print(f"ONLY NEW   {name}")
        elif old[name] == new[name]:
            print(f"same       {name} ({len(old[name])} instructions)")
            continue
        else:
            a, b = old[name], new[name]
            i = next((k for k, (x, y) in enumerate(zip(a, b)) if x != y), min(len(a), len(b)))
            print(f"DIFFERENT  {name} ({len(a)} -> {len(b)} instructions; first at #{i}: "
                  f"{a[i] if i < len(a) else '<end>'!r} -> {b[i] if i < len(b) else '<end>'!r})")
        differing += 1
    print(f"{len(set(old) | set(new))} kernels, {differing} differing")
    return 1 if differing else 0


if __name__ == "__main__":
    sys.exit(main(sys.argv))
