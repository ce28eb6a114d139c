"""Code footprint of one kernel of the library, on the CPU (no GPU, no profiler): what the instruction cache has to hold.
    python tools/sass_footprint.py [--lib LIB | --src ROOT] [--kernel SYMBOL] [--func NAME]
--lib: a built libwrsn_b200.so; registers and stack then come from `cuobjdump -res-usage` (ptxas' spill counts need a
build).  Otherwise the library is compiled into a temporary directory from ROOT (default: this repository) with
__graft_entry__.NVCC_FLAGS plus -Xptxas -v, and ptxas' own report is printed.
Prints, for the kernel (default: g32::k_env<MODE_STEP>, one warp per environment): the size of its body and of every
out-of-line device function from the cubin's FUNC symbols, the opcode counts of the function(s) whose name starts with
NAME (default: reward_loop) that matter for the hot loop — shuffles, their divergent-warp fallback (WARPSYNC /
ENDCOLLECTIVE / BSSY), local-memory traffic — and registers, stack and spills."""
import argparse, collections, os, re, subprocess, sys, tempfile

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
from sass_hotspots import disasm, extract_cubin, short_name  # noqa: E402

WATCH = ["SHFL", "WARPSYNC", "ENDCOLLECTIVE", "BRA.DIV", "BSSY", "LDL", "STL", "LDS", "STS", "LD", "ST", "CALL", "IMAD"]


def build(root, tmp):
    sys.path.insert(0, os.path.dirname(HERE))
    from __graft_entry__ import NVCC_FLAGS
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    lib = os.path.join(tmp, "libwrsn_b200.so")
    cmd = [nvcc] + NVCC_FLAGS + ["-Xptxas", "-v", "-I", os.path.join(root, "include"), "-o", lib,
                                 os.path.join(root, "multi_agent_rl_wrsn_b200", "csrc", "wrsn_kernels.cu")]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode:
        sys.exit(r.stdout + r.stderr)
    return lib, r.stdout + r.stderr


def func_sizes(cubin, kern):
    """FUNC symbols of the kernel: the device functions inside its section ("$kernel$function") and what is left of
    the kernel symbol, which spans the whole section, for its own body."""
    out = subprocess.run(["readelf", "-sW", cubin], capture_output=True, text=True).stdout
    sizes, section = {}, 0
    for ln in out.splitlines():
        f = ln.split()
        if len(f) < 8 or f[3] != "FUNC":
            continue
        name = f[-1]
        if name == kern:
            section = int(f[2], 0)
        elif name.startswith("$" + kern + "$"):
            sizes[short_name(name)] = int(f[2], 0)
    if section:
        sizes["(kernel body)"] = section - sum(sizes.values())
    return sizes


def opcode(text):
    t = text.split()
    if t and t[0].startswith("@"):
        t = t[1:]
    return t[0] if t else ""


def ptxas_report(log, kern, func):
    """ptxas -v lines of the kernel and of the device functions named `func*` compiled with it (the functions' lines
    follow their kernel's "Compiling entry function" line)."""
    lines, entry, keep = [], None, False
    for ln in log.splitlines():
        m = re.search(r"Compiling entry function '([^']+)'", ln)
        if m:
            entry, keep = m.group(1), False
            continue
        m = re.search(r"Function properties for (\S+)", ln)
        if m:
            name = m.group(1)
            short = "kernel" if name == kern else short_name("$" + name)
            keep = entry == kern and (name == kern or short.startswith(func))
            if keep:
                lines.append(short + ":")
            continue
        if keep and ("stack frame" in ln or "Used" in ln):
            lines.append("    " + ln.split(":", 1)[-1].strip() if "Used" in ln else "    " + ln.strip())
    return lines


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--lib", help="built libwrsn_b200.so (default: build one)")
    ap.add_argument("--src", default=os.path.dirname(HERE), help="repository root to build from (without --lib)")
    ap.add_argument("--kernel", default="_ZN3g325k_envILi4EEEv7KParams", help="mangled kernel symbol")
    ap.add_argument("--func", default="reward_loop", help="device function(s) to count opcodes in (name prefix)")
    a = ap.parse_args()
    tmp = tempfile.mkdtemp(prefix="sass_footprint_")
    log = None
    lib = a.lib
    if lib is None:
        lib, log = build(os.path.abspath(a.src), tmp)
    cubin = extract_cubin(lib, tmp)

    sizes = func_sizes(cubin, a.kernel)
    if not sizes:
        sys.exit("no FUNC symbol %s in %s" % (a.kernel, lib))
    total = sum(sizes.values())
    print("## %s: %d bytes of SASS (%d instructions), %d out of line in %d functions\n"
          % (a.kernel, total, total // 16, total - sizes.get("(kernel body)", 0), len(sizes) - 1))
    print("| function | bytes | instructions |\n|---|---|---|")
    for name, n in sorted(sizes.items(), key=lambda kv: -kv[1]):
        print("| `%s` | %d | %d |" % (name, n, n // 16))

    ins = disasm(cubin, a.kernel)
    per = collections.defaultdict(collections.Counter)
    for _, fn, _, text in ins:
        if fn.startswith(a.func):
            per[fn][opcode(text)] += 1
    print("\n## opcodes of %s*\n" % a.func)
    print("| function | instructions | " + " | ".join(WATCH) + " |\n|---|---|" + "---|" * len(WATCH))
    for fn, cnt in sorted(per.items()):
        base = collections.Counter()
        for op, n in cnt.items():
            base[op.split(".")[0] if not op.startswith("BRA.DIV") else "BRA.DIV"] += n
        print("| `%s` | %d | " % (fn, sum(cnt.values())) + " | ".join(str(base[w]) for w in WATCH) + " |")

    print("\n## registers, stack, spills\n")
    if log is not None:
        for ln in ptxas_report(log, a.kernel, a.func):
            print(ln)
    else:
        out = subprocess.run(["cuobjdump", "-res-usage", cubin], capture_output=True, text=True).stdout.splitlines()
        for k, ln in enumerate(out):
            m = re.match(r"\s*Function ([^:]+):", ln)
            if m and (m.group(1) == a.kernel or short_name("$" + m.group(1)).startswith(a.func)) and k + 1 < len(out):
                print("%s: %s" % ("kernel" if m.group(1) == a.kernel else short_name("$" + m.group(1)), out[k + 1].strip()))
        print("(spill counts: run without --lib)")


if __name__ == "__main__":
    main()
