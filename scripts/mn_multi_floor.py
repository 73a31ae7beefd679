"""Algorithmic bytes and operations of the weight-gradient side of the Envelope update's backward pass at the bench shape, from shapes only:
   python scripts/mn_multi_floor.py [kernel_us] [hbm_TBps] [tflops]
dW_k = G_k^T H_{k-1} + db_k = colsum(G_k) for the three 256 x 256 hidden layers and the 24-wide output layer over M = 65,536 pair rows,
f16x2 planes (4 bytes per element, three MMAs per product).  With a measured kernel time it prints the share of each floor."""
import sys

M = 1024 * 64          # batch x |W| pair rows
HID, OUT, LD_OUT = 256, 24, 64
PLANE_BYTES = 4         # f16x2: two fp16 planes per element
NPROD = 3

hbm = float(sys.argv[2]) if len(sys.argv) > 2 else 6.48     # TB/s, measured stream bandwidth of a B200 (DESIGN 4.6)
peak = float(sys.argv[3]) if len(sys.argv) > 3 else 1687.0  # TFLOP/s, measured dense fp16 MMA rate of a B200 (DESIGN 4.6)

# (g_cols, ldg, h_cols) per product; rows_per_split / S as the kernel plans them (148 / n_tiles splits, multiples of 32 rows)
jobs = [(HID, HID, HID)] * 3 + [(OUT, LD_OUT, HID)]
reads = writes = flops = 0
for gc, ldg, hc in jobs:
    n_tiles = (gc + 127) // 128
    S = 148 // n_tiles
    rps = ((M + S - 1) // S + 31) // 32 * 32
    S = (M + rps - 1) // rps
    reads += M * (ldg + hc) * PLANE_BYTES           # G and H planes, each read once
    writes += S * gc * hc * 4 + S * gc * 4          # fp32 partials (real rows only) + column-sum partials
    flops += 2 * NPROD * M * (n_tiles * 128) * hc   # MMAs as issued: 128-row tiles of G^T
t_read = reads / (hbm * 1e12) * 1e6
t_all = (reads + writes) / (hbm * 1e12) * 1e6
t_mma = flops / (peak * 1e12) * 1e6
print(f"operand reads   {reads / 1e6:8.1f} MB   floor {t_read:6.1f} us at {hbm} TB/s")
print(f"partial writes  {writes / 1e6:8.1f} MB   (reads + writes: floor {t_all:6.1f} us)")
print(f"MMAs            {flops / 1e9:8.1f} GFLOP floor {t_mma:6.1f} us at {peak} TFLOP/s")
if len(sys.argv) > 1:
    t = float(sys.argv[1])
    print(f"kernel {t:.1f} us: {t_read / t:.2f} of the read floor, {t_all / t:.2f} of the read + write floor, {t_mma / t:.2f} of the MMA floor")
