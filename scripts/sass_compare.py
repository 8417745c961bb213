"""Compare the SASS of two builds of one object file, kernel by kernel, with addresses and symbol names stripped.

    python scripts/sass_compare.py OLD.o NEW.o

Kernels are matched by demangled name with a trailing `false` template argument dropped, so that the default
instantiation of a kernel that gained a `bool` template flag is compared with its old self.  Exit status 1 if a kernel
differs or disappeared.  Needs only the CUDA toolkit (cuobjdump), no GPU.
"""
import re
import subprocess
import sys
from pathlib import Path

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
from neural_speech_decoding_b200.build import find_nvcc  # noqa: E402

CUOBJ = str(Path(find_nvcc()).resolve().parent / "cuobjdump")

def funcs(obj):
    out = subprocess.run([CUOBJ, "-sass", obj], capture_output=True, text=True).stdout
    res, name, body = {}, None, []
    for line in out.splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            if name: res[name] = body
            name, body = m.group(1), []
            continue
        if name is None: continue
        m = re.match(r"\s*/\*[0-9a-f]{4,}\*/\s*(.*?)\s*;?\s*/\*", line)
        if m:
            ins = m.group(1)
            ins = re.sub(r"_Z\w+", "<sym>", ins)
            ins = re.sub(r"(BRA|CALL\.REL\.NOINC|BSSY(\.RECONVERGENT)?\s+B\d+,|SSY|PBK|PCNT)\s+0x[0-9a-f]+", r"\1 <addr>", ins)
            body.append(ins)
    if name: res[name] = body
    return res

def demangle(names):
    out = subprocess.run(["c++filt"], input="\n".join(names), capture_output=True, text=True).stdout.splitlines()
    return dict(zip(names, out))

a, b = funcs(sys.argv[1]), funcs(sys.argv[2])
da, db = demangle(list(a)), demangle(list(b))
def key(d):
    # "void na::tc::decoder_infer_x3_kernel<0, false>(...)" -> "decoder_infer_x3_kernel<0>"
    d = d.split("(")[0].replace("void ", "")
    d = re.sub(r"(, false)+>", ">", d)
    return d
ka = {key(da[n]): n for n in a}
kb = {key(db[n]): n for n in b}
bad = 0
for k in sorted(ka):
    if k not in kb:
        print("MISSING in new:", k); bad += 1; continue
    x, y = a[ka[k]], b[kb[k]]
    if x != y:
        bad += 1
        import difflib
        d = list(difflib.unified_diff(x, y, lineterm="", n=1))
        print(f"DIFF {k}: {len(x)} vs {len(y)} instructions, {sum(1 for l in d if l[:1] in '+-')} changed lines")
        print("\n".join(d[:40]))
    else:
        print(f"same {k} ({len(x)} instructions)")
print("new-only:", sorted(set(kb) - set(ka)))
sys.exit(1 if bad else 0)
