"""Compare the policy kernels of two builds instruction by instruction (cuobjdump -sass) and by ptxas -v (registers, stack,
spills): one line per kernel of the OLD build, matched to the NEW build's instantiation with the multi-policy flag false.

    python tools/policy_sass_compare.py OLD_OBJ_DIR NEW_OBJ_DIR OLD_PTXAS_LOG NEW_PTXAS_LOG file.o ...

The object directories are com_marl_b200/lib/obj of `python -m com_marl_b200.build --force -v`, whose output is the ptxas
log.  "identical modulo param offsets (+32 bytes)": every differing instruction only reads a kernel parameter 32 bytes
further on (cm_policy_io grew by 32 bytes in ABI 6).
"""
import re, subprocess, sys
OLD, NEW = sys.argv[1], sys.argv[2]   # lib/obj dirs
def sass(obj):
    out = subprocess.run(["/usr/local/cuda/bin/cuobjdump", "-sass", obj], capture_output=True, text=True).stdout
    funcs, cur = {}, None
    for line in out.splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m: cur = m.group(1); funcs[cur] = []; continue
        m = re.match(r"\s*/\*[0-9a-f]{4,}\*/\s+(.*?);", line)
        if cur and m: funcs[cur].append(m.group(1).strip())
    return funcs
def norm(ins): return [re.sub(r"c\[0x0\]\[0x[0-9a-f]+\]", "c[0x0][P]", i) for i in ins]
def same_mod_shift(a, b, shift=0x20):
    """every differing instruction differs only in hex constants that grew by `shift` (kernel parameters behind cm_policy_io)"""
    if len(a) != len(b): return False
    for x, y in zip(norm(a), norm(b)):
        if x == y: continue
        hx, hy = re.findall(r"0x[0-9a-f]+", x), re.findall(r"0x[0-9a-f]+", y)
        if re.sub(r"0x[0-9a-f]+", "H", x) != re.sub(r"0x[0-9a-f]+", "H", y) or len(hx) != len(hy): return False
        if any(int(v, 16) - int(u, 16) not in (0, shift) for u, v in zip(hx, hy)): return False
    return True
def ptxas(log):
    res, cur = {}, None
    for line in open(log):
        m = re.search(r"Compiling entry function '(\S+)'", line) or re.search(r"Function properties for (\S+)", line)
        if m: cur = m.group(1)
        m = re.search(r"(\d+) bytes stack frame, (\d+) bytes spill stores, (\d+) bytes spill loads", line)
        if m and cur: res.setdefault(cur, {})["spill"] = m.groups()
        m = re.search(r"Used (\d+) registers", line)
        if m and cur: res.setdefault(cur, {})["regs"] = m.group(1)
    return res
def canon(name):
    name = re.sub(r"ELb0EEEvNSt11conditionalIXT1_ENS_14AttnMmaSetArgsENS_11AttnMmaArgsEE4typeE", "EEEvNS_11AttnMmaArgsE", name)
    name = re.sub(r"ELb0EEEv", "EEEv", name)
    return re.sub(r"ILb0EEEv(NS_10PolicyArgsE)", r"E\1", name)   # the new bool template argument, false = the existing kernel
po, pn = ptxas(sys.argv[3]), ptxas(sys.argv[4])
for obj in sys.argv[5:]:
    fo, fn = sass(f"{OLD}/{obj}"), sass(f"{NEW}/{obj}")
    mapped = {}
    for k in fn:
        mapped.setdefault(canon(k), k)
    for k in sorted(fo):
        if not k.startswith("_ZN2cm") or "prepare" in k: continue
        kn = mapped.get(k, k if k in fn else None)
        if kn is None: print(obj, k, "MISSING"); continue
        a, b = fo[k], fn[kn]
        st = "identical" if a == b else ("identical modulo param offsets" if norm(a) == norm(b) else ("identical modulo param offsets (+32 bytes)" if same_mod_shift(a, b) else f"DIFFERENT ({len(a)} -> {len(b)} instructions)"))
        same = "ptxas-same" if po.get(k) == pn.get(kn) else f"ptxas {po.get(k)} -> {pn.get(kn)}"
        print(obj, kn, len(b), st, same)
    new_only = [k for k in fn if k.startswith("_ZN2cm") and canon(k) not in fo and k not in fo]
    if new_only: print(obj, "new only:", new_only)
