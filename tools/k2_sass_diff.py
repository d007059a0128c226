"""Compare the SASS of kernel 2's top-2 instantiations between two builds of csrc/k2_sim.cu (no GPU needed).

    python tools/k2_sass_diff.py OLD.o NEW.o

Each object's `cuobjdump -sass` is cut into functions; the k2_sim_top2_kernel instantiations are keyed by their template
arguments (TF32, MC, PAIR) and compared instruction by instruction after stripping addresses, encodings and symbol names.
Exit status 0 = every instantiation identical.  For changes that share kernel 2's main loop with another epilogue.
"""
import re
import subprocess
import sys

CUOBJDUMP = "/usr/local/cuda/bin/cuobjdump"


def top2_functions(obj):
    out = subprocess.run([CUOBJDUMP, "-sass", obj], capture_output=True, text=True, check=True).stdout
    funcs, key = {}, None
    for line in out.splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            t = re.search(r"k2_sim_top2_kernelILb(\d)ELi(\d)ELb(\d)E", m.group(1))
            key = tuple(int(x) for x in t.groups()) if t else None
            if key:
                funcs[key] = []
            continue
        if key is None:
            continue
        ins = re.sub(r"/\*[0-9a-f]{4,}\*/", "", line)        # address
        ins = re.sub(r"/\* 0x[0-9a-f]+ \*/", "", ins)        # encoding
        ins = re.sub(r"_ZN\w+", "<sym>", ins)                # symbol names (the anonymous namespace hash differs per build)
        ins = ins.strip()
        if ins and not ins.startswith("..."):
            funcs[key].append(ins)
    return funcs


def main(old, new):
    a, b = top2_functions(old), top2_functions(new)
    ok = True
    for key in sorted(set(a) | set(b)):
        name = "TF32=%d MC=%d PAIR=%d" % key
        if key not in a or key not in b:
            print(f"{name}: missing in {'old' if key not in a else 'new'}")
            ok = False
            continue
        same = a[key] == b[key]
        ok &= same
        print(f"{name}: {len(a[key])} / {len(b[key])} instructions, {'identical' if same else 'DIFFERENT'}")
    print(f"{len(a)} instantiations compared: {'identical' if ok and len(a) == 8 else 'not identical'}")
    return 0 if ok and len(a) == 8 else 1


if __name__ == "__main__":
    sys.exit(main(*sys.argv[1:3]))
