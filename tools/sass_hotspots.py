"""Executed warp instructions per device function and per source line, from an ncu capture and the library it profiled.
    python tools/sass_hotspots.py <report.ncu-rep> <lib.so> <mangled kernel substring> [top]
Joins `ncu --page source --csv` (per-SASS-instruction counters, in address order) with `nvdisasm --print-line-info` of the
cubin (function labels + //## File "...", line N markers, same instruction order)."""
import csv, io, os, re, subprocess, sys, tempfile, collections


def extract_cubin(lib, tmp):
    """The sm_100a cubin embedded in a fat binary (`lib`), extracted into directory `tmp`."""
    subprocess.run(["cuobjdump", "-xelf", "all", os.path.abspath(lib)], cwd=tmp, check=True, stdout=subprocess.DEVNULL)
    return [os.path.join(tmp, f) for f in os.listdir(tmp) if f.endswith(".cubin")][0]


def short_name(lab):
    """Readable name of a device-function label or symbol of this project, e.g. `reward_loop` or `nodes_batch<0>`."""
    mm = re.search(r"\$_ZN\d+_INTERNAL_[0-9a-f]+_\d+_\w+?_cu_[0-9a-f]+\d*(?:4gany|3g32)(\d+)(\w+)", lab)
    name = lab
    if mm:
        n = int(mm.group(1)); name = mm.group(2)[:n]
        t = re.match(r"I((?:L[ib]\d+E)+)E", mm.group(2)[n:])          # template arguments, e.g. ILi4ELb1EE -> <4,1>
        if t:
            name += "<" + ",".join(re.findall(r"L[ib](\d+)E", t.group(1))) + ">"
    elif "$__internal" in lab or "$__cuda" in lab:
        name = lab.split("$")[-1]
    return name


def disasm(cubin, kern):
    """Instruction list of the kernel sections whose name contains `kern`: (offset, function, (file, line), text)."""
    dis = subprocess.run(["nvdisasm", "--print-line-info", "-c", cubin], capture_output=True, text=True).stdout.splitlines()
    ins, on, func, fl = [], False, "(kernel)", ("?", 0)
    for ln in dis:
        if ln.startswith("//---") and ".text." in ln:
            on = kern in ln
            func = "(kernel)"
            continue
        if not on:
            continue
        m = re.match(r"\s*//## File \"([^\"]+)\", line (\d+)", ln)
        if m:
            fl = (os.path.basename(m.group(1)), int(m.group(2))); continue
        m = re.match(r"^(\$\S+):", ln)
        if m:
            func = short_name(m.group(1)); continue
        m = re.match(r"\s+/\*([0-9a-f]{4,})\*/\s+(\S.*?);", ln)
        if m:
            ins.append((int(m.group(1), 16), func, fl, m.group(2)))
    return ins


def main():
    rep, lib, kern = sys.argv[1], sys.argv[2], sys.argv[3]
    top = int(sys.argv[4]) if len(sys.argv) > 4 else 40
    ins = disasm(extract_cubin(lib, tempfile.mkdtemp()), kern)
    out = subprocess.run(["ncu", "-i", rep, "--page", "source", "--csv"], capture_output=True, text=True).stdout
    rows = list(csv.reader(io.StringIO(out)))
    h = next(i for i, r in enumerate(rows) if r and r[0] == "Address")
    col = {c: i for i, c in enumerate(rows[h])}
    data = rows[h + 1:]
    base = int(data[0][col["Address"]], 16)
    byoff = {int(r[col["Address"]], 16) - base: r for r in data if r and r[0].startswith("0x")}
    tot = 0; f_acc = collections.Counter(); l_acc = collections.Counter(); f_samp = collections.Counter(); l_samp = collections.Counter()
    for off, fn, fl, txt in ins:
        r = byoff.get(off)
        if r is None:
            continue
        n = int(r[col["Instructions Executed"]]); s = int(r[col["# Samples"]])
        tot += n; f_acc[fn] += n; l_acc[fl] += n; f_samp[fn] += s; l_samp[fl] += s
    ts = sum(f_samp.values()) or 1
    print("total executed warp instructions: %d   (%d SASS instructions matched of %d)" % (tot, len(byoff), len(ins)))
    print("\n| function | executed warp instr | share | stall samples share |\n|---|---|---|---|")
    for fn, n in f_acc.most_common(25):
        print("| `%s` | %d | %.1f %% | %.1f %% |" % (fn, n, 100.0 * n / tot, 100.0 * f_samp[fn] / ts))
    print("\n| file:line | executed warp instr | share | samples share |\n|---|---|---|---|")
    for fl, n in l_acc.most_common(top):
        print("| %s:%d | %d | %.1f %% | %.1f %% |" % (fl[0], fl[1], n, 100.0 * n / tot, 100.0 * l_samp[fl] / ts))


if __name__ == "__main__":
    main()
