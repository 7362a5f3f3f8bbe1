"""SASS bytes per device function of one kernel object (instruction-cache footprint study): python tools/code_size.py inst_15_3.o
--hot: only the functions one IPM iteration of the original problem (RS = false) runs, with their sum"""
import subprocess, sys, re
HOT_PHASES = ("ph_derivs", "ph_trial", "ph_dir", "ph_accept")
HOT_OTHER = ("riccati_factor", "riccati_forward", "update_mu", "check_accept", "filter_add",
             "warp_sum", "seg_sum", "warp_max", "warp_min", "n_tan", "n_log", "n_pow", "n_sincos")
args = [a for a in sys.argv[1:] if a != "--hot"]; hot = "--hot" in sys.argv[1:]
obj = args[0]
out = subprocess.run(["cuobjdump", "-elf", obj], capture_output=True, text=True).stdout
rows = []; on = False
for line in out.splitlines():
    if line.startswith(".section .symtab"): on = True; continue
    if on and line.startswith(".section"): break
    a = line.split()
    if on and len(a) >= 7 and a[3] in ("0x2", "0x12", "0x22") and "$" in a[-1]:
        rows.append((int(a[2], 16), int(a[1], 16), a[-1].split("$")[-1]))
    elif on and len(a) >= 7 and a[3] == "0x12":
        rows.append((int(a[2], 16), int(a[1], 16), a[-1]))
rows.sort(reverse=True); tot = 0; phases = 0
for sz, off, n in rows:
    name = subprocess.run(["c++filt", n], capture_output=True, text=True).stdout.strip()
    name = re.sub(r"nmpc::LayT<(\d+), (\d+), (\w+), (\d+)>", r"L", name); name = re.sub(r"\(.*", "", name)
    if hot:
        base = re.match(r"(?:\S+\s+)?([\w:]+)", name).group(1).split("::")[-1]
        if base in HOT_PHASES:
            if not name.endswith("true>"):      # the restoration (RS = true) instantiations are not per-iteration code
                phases += sz
            else: continue
        elif base not in HOT_OTHER: continue
    print(f"{sz / 1024:8.1f} KB  {name[:90]}"); tot += sz
if hot:
    print(f"{phases / 1024:8.1f} KB  ph_derivs + ph_trial + ph_dir + ph_accept (RS = false)")
    print(f"{tot / 1024:8.1f} KB  per-iteration total")
else:
    print(f"{tot / 1024:8.1f} KB total")
