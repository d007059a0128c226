"""Compare the SASS of kernel 2's top-2 instantiations between two builds of csrc/k2_sim.cu (no GPU needed).

    python tools/k2_sass_diff.py OLD.o NEW.o
    python tools/k2_sass_diff.py --topk OLD.o NEW.o       (the same builds, top-KP instantiations)
    python tools/k2_sass_diff.py --spair OLD.o NEW.o      (two builds of csrc/spair_batch.cu)

Each object's `cuobjdump -sass` is cut into functions; the k2_sim_top2_kernel instantiations are keyed by their template
arguments (TF32, MC, PAIR) and compared instruction by instruction after stripping addresses, encodings and symbol names.
Exit status 0 = every instantiation identical.  For changes that share kernel 2's main loop with another epilogue.

--topk compares the row top-KP instantiations (k2_sim_topk_kernel) instead, keyed by (TF32, MC, PAIR, KP).

--spair compares the fp32 instantiations of the SPair batch kernels instead: spair_stream_kernel keyed by (KT, MMA, TERMS)
and spair_batch_kernel by KT.  Builds that template them on the map's element type as well carry a leading `f` in the
float instantiations' mangled names; only those are matched (the bf16 / fp16 ones have no counterpart in an fp32-only
build).  For changes that add element types without touching the fp32 code.
"""
import re
import subprocess
import sys

CUOBJDUMP = "/usr/local/cuda/bin/cuobjdump"


def k2_key(name):
    t = re.search(r"k2_sim_top2_kernelILb(\d)ELi(\d)ELb(\d)E", name)
    return tuple(int(x) for x in t.groups()) if t else None


def k2_topk_key(name):
    t = re.search(r"k2_sim_topk_kernelILb(\d)ELi(\d)ELb(\d)ELi(\d+)E", name)
    return ("topk",) + tuple(int(x) for x in t.groups()) if t else None


def spair_key(name):
    t = re.search(r"spair_stream_kernelIf?Li(\d+)ELb(\d)ELi(\d)EE", name)
    if t:
        return ("stream",) + tuple(int(x) for x in t.groups())
    t = re.search(r"spair_batch_kernelIf?Li(\d+)EE", name)
    return ("batch", int(t.group(1))) if t else None


def top2_functions(obj, key_of=k2_key):
    out = subprocess.run([CUOBJDUMP, "-sass", obj], capture_output=True, text=True, check=True).stdout
    funcs, key = {}, None
    for line in out.splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            key = key_of(m.group(1))
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


def key_name(key):
    if key[0] == "stream":
        return "spair_stream_kernel KT=%d MMA=%d TERMS=%d" % key[1:]
    if key[0] == "topk":
        return "TF32=%d MC=%d PAIR=%d KP=%d" % key[1:]
    if key[0] == "batch":
        return "spair_batch_kernel KT=%d" % key[1:]
    return "TF32=%d MC=%d PAIR=%d" % key


def main(old, new, spair=False, topk=False):
    key_of = spair_key if spair else (k2_topk_key if topk else k2_key)
    a, b = top2_functions(old, key_of), top2_functions(new, key_of)
    want = 24 if spair else (16 if topk else 8)  # spair: 6 key-point tiles x (3 streaming forms + the first form); topk: KP 8 and 16
    ok = True
    for key in sorted(set(a) | set(b)):
        name = key_name(key)
        if key not in a or key not in b:
            print(f"{name}: missing in {'old' if key not in a else 'new'}")
            ok = False
            continue
        same = a[key] == b[key]
        ok &= same
        print(f"{name}: {len(a[key])} / {len(b[key])} instructions, {'identical' if same else 'DIFFERENT'}")
    print(f"{len(a)} instantiations compared: {'identical' if ok and len(a) == want else 'not identical'}")
    return 0 if ok and len(a) == want else 1


if __name__ == "__main__":
    args = [x for x in sys.argv[1:] if x not in ("--spair", "--topk")]
    sys.exit(main(*args[:2], spair="--spair" in sys.argv[1:], topk="--topk" in sys.argv[1:]))
