"""Compare the SASS of two builds of csrc, function by function.

    git archive <commit> | tar -x -C /tmp/old && make -C /tmp/old/residual-td3-robot-navigation_b200/csrc -j8
    make -C residual-td3-robot-navigation_b200/csrc -j8
    python tools/sass_diff.py /tmp/old/residual-td3-robot-navigation_b200/csrc/build residual-td3-robot-navigation_b200/csrc/build

Each directory holds the per-source objects the Makefile writes (csrc/build/*.o).  Addresses and encoding words are dropped, so two
functions compare equal when they have the same instructions in the same order.  The hash in the names of anonymous namespaces
depends on where a tree was compiled and is dropped too.  Prints, per object, the functions only one side has and the functions
whose instructions differ; the exit status is 1 if a function present on both sides differs."""
import glob
import os
import re
import subprocess
import sys

CUOBJDUMP = os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "bin", "cuobjdump")


def functions(obj):
    """{mangled name: [instruction lines]} of one object file."""
    out = subprocess.run([CUOBJDUMP, "-sass", obj], check=True, capture_output=True, text=True).stdout
    funcs, name = {}, None
    for line in out.splitlines():
        line = re.sub(r"_GLOBAL__N__[0-9a-f]+_", "_GLOBAL__N__", line)
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            name = m.group(1)
            funcs[name] = []
        elif name is not None:
            line = re.sub(r"/\*.*?\*/", "", line).strip()      # /*0040*/ addresses and /* 0x... */ encoding words
            if line:
                funcs[name].append(line)
    return funcs


def main(old_dir, new_dir):
    names = sorted({os.path.basename(p) for d in (old_dir, new_dir) for p in glob.glob(os.path.join(d, "*.o"))})
    changed = 0
    for obj in names:
        old = functions(os.path.join(old_dir, obj)) if os.path.isfile(os.path.join(old_dir, obj)) else {}
        new = functions(os.path.join(new_dir, obj)) if os.path.isfile(os.path.join(new_dir, obj)) else {}
        differ = sorted(f for f in old.keys() & new.keys() if old[f] != new[f])
        changed += len(differ)
        print("%-24s %3d -> %3d functions, %d identical, %d differ" % (obj, len(old), len(new), len(old.keys() & new.keys()) - len(differ),
                                                                      len(differ)))
        for tag, fs in (("only old", sorted(old.keys() - new.keys())), ("only new", sorted(new.keys() - old.keys())), ("differs", differ)):
            for f in fs:
                print("    %-9s %s" % (tag, f))
    return 1 if changed else 0


if __name__ == "__main__":
    if len(sys.argv) != 3:
        sys.exit(__doc__)
    sys.exit(main(sys.argv[1], sys.argv[2]))
