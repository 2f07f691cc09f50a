"""tools/deflate_phases.py for the 32 phase slots of deflate_split_roles.cu.txt (it also reads a library with 16 slots).
  cp tools/experiments/deflate_split_roles.cu.txt zipc_b200/csrc/deflate.cu
  make -C zipc_b200/csrc BUILD=build_timing OUT=../libzipc_b200_timing.so EXTRA=-DZB_DEFLATE_TIMING
  ZIPC_B200_LIB=$PWD/zipc_b200/libzipc_b200_timing.so python tools/experiments/deflate_phases_split_roles.py [level] [members]"""
import ctypes as C
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
from zipc_b200 import _lib, synth
from zipc_b200 import zipc_deflate as zd

level = sys.argv[1] if len(sys.argv) > 1 else "default"
count = int(sys.argv[2]) if len(sys.argv) > 2 else 3000
# Thread 0 (the parse warp, or warp 0 of level best's back end) accounts its whole timeline in slots 0-10, 15 and 21; the first
# front thread its own in 11-14 and 22; the closer's first thread (levels fast and default) its own in 16-20.  fin_* are closes
# run by all warps (the member's last block; every block at level best), C:fin_* mid-member closes by the closer.
names = ["P:help_walks", "wait_for_front", "parse0", "deep", "parse1", "tokens", "fin_sort", "fin_huff", "fin_hdr", "fin_pack", "other",
         "F:stage", "F:hash+partition", "F:insert", "F:shallow", "jump_codes",
         "C:fin_sort", "C:fin_huff", "C:fin_hdr", "C:fin_pack", "C:idle", "P:wait_buffer_free", "F:wait_empty"]
NSLOT = 32
ctx = zd.Context(0)
L = ctx.L
sizes = synth.member_sizes(count, seed=3)
datas = [synth.text_v1(1000 + i, int(n)) for i, n in enumerate(sizes)]
ctx.deflate_batch(datas, level, 2)
out = (C.c_ulonglong * NSLOT)()
L.zipc_b200_debug_deflate_phases.argtypes = [C.c_void_p, C.c_int]
L.zipc_b200_debug_deflate_phases(out, 1)
dbg = (C.c_ulonglong * 16)()
L.zipc_b200_debug_deflate_counters.argtypes = [C.c_void_p, C.c_int]
L.zipc_b200_debug_deflate_counters(dbg, 1)
t0 = time.perf_counter()
res = ctx.deflate_batch(datas, level, 2)
dt = time.perf_counter() - t0
L.zipc_b200_debug_deflate_phases(out, 0)
tot = sum(out[:11]) + out[15] + out[21]
U = sum(d.size for d in datas)
print(f"level {level}: {count} members, {U/1e6:.0f} MB, ratio {sum(r[1].size for r in res)/U:.4f}, call {dt*1e3:.1f} ms; cycles per input byte per SM-CTA: {tot/U:.2f}")
for n, v in zip(names, out):
    if v:
        print(f"  {n:18s} {100*v/tot:5.1f} %   {v/U:6.2f} clk/byte")
front = sum(out[11:15]) + out[22]
closer = sum(out[16:21])
print(f"  per role, clk/byte: thread 0 {tot/U:.2f}, front {front/U:.2f}" + (f", closer {closer/U:.2f} (idle {out[20]/U:.2f})" if closer else ""))
L.zipc_b200_debug_deflate_counters(dbg, 0)
tiles = sum(-(-d.size // 2048) for d in datas)
print("  deep (warp 0, per tile): passes %.2f, loop iterations %.1f, cycles: resume %.0f, walk loop %.0f, waiting for the other back warps %.0f"
      % (dbg[8] / tiles, dbg[9] / tiles, dbg[5] / tiles, dbg[6] / tiles, dbg[7] / tiles))
