"""Regenerates profiles/r3_sass_summary.txt: per-kernel counts of the SASS mnemonics that show which hardware path a kernel
uses (TMA bulk copies, mbarriers, cp.async, cluster barriers, match, atomics, IEEE-division fast paths), from the shipped
libmvr_b200.so.   python scripts/sass_summary.py [> profiles/r3_sass_summary.txt]"""
import os, re, subprocess

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "mvtn_b200", "libmvr_b200.so")
KERNELS = ("mesh_shade_kernelILb0ELi4ELi4ELb0", "mesh_scatter_kernelILi4ELb0ELi256", "mesh_scatter_kernelILi8ELb0ELi128",
           "mesh_backward_kernel_stripILi3ELb0ELb0", "mesh_backward_kernel_stripILi2ELb0ELb1", "points_tile_kernelILi4E",
           "points_bin_kernel_fused", "points_backward_kernelILi4ELb0ELb0", "images_regularize_kernelILb1", "images_regularize_backward_rows_kernelILb1",
           "mesh_soft_blend_kernel", "mesh_soft_backward_kernel", "mesh_backward_finish_kernel", "look_at_forward_one_cta_kernel", "geom_pack_faces_kernelIt")
COLS = (("UBLKCP", r"^UBLKCP"), ("SYNCS", r"^SYNCS"), ("LDGSTS", r"^LDGSTS"), ("UCGABAR", r"^UCGABAR"), ("MATCH", r"^MATCH"),
        ("RED/ATOMG", r"^(RED|ATOMG)"), ("ATOMS", r"^ATOMS"), ("MUFU.RCP", r"^MUFU\.RCP"), ("LDG.256", r"^LDG\.E\.(\w+\.)*256"), ("FCHK", r"^FCHK"), ("ACQBULK", r"^ACQBULK"), ("PREEXIT", r"^PREEXIT"))

sass = subprocess.run(["cuobjdump", "-sass", LIB], capture_output=True, text=True, check=True).stdout
funcs, cur = {}, None
for line in sass.splitlines():
    m = re.search(r"Function : (\S+)", line)
    if m:
        cur = m.group(1); funcs[cur] = []
        continue
    m = re.match(r"\s*/\*[0-9a-f]{4,6}\*/\s+(?:@!?U?P\d+\s+)?([A-Z][A-Z0-9_.]*)", line)
    if m and cur:
        funcs[cur].append(m.group(1))

print("SASS mnemonic counts of the shipped libmvr_b200.so (cuobjdump -sass mvtn_b200/libmvr_b200.so; full listings: profiles/sass_*.txt;")
print("regenerate: python scripts/sass_summary.py)")
print("UBLKCP / SYNCS = 1-D TMA bulk copy + mbarrier (scatter kernel: face records; point tile kernel: point lists);")
print("LDGSTS = cp.async (strip backward); UCGABAR = thread-block-cluster barrier (clustered point binning, counters read through distributed")
print("shared memory); MATCH = __match_any_sync (warp-aggregated atomics); ATOMS = shared-memory atomics; RED/ATOMG = global atomics;")
print("FCHK = range check of an IEEE division's fast path; ACQBULK / PREEXIT = griddepcontrol.wait / .launch_dependents (programmatic dependent launch)")
for want in KERNELS:
    for name, ops in funcs.items():
        if want in name:
            counts = "  ".join(f"{label} {sum(1 for o in ops if re.match(rx, o))}" for label, rx in COLS)
            print(f"{name:<72s} instr {len(ops):5d}  {counts}")
