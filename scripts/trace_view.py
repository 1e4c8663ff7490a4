"""prints the time line recorded by scripts/actor_prof.py (TACTOR_TRACE=file.npy): item 1 of CTA 0"""
import sys
import numpy as np
w = np.load(sys.argv[1])
nph = 2                              # generator phases of actor_pipe_kernel
gen = w[:16 * 48 * 4].reshape(16, 48, 4).astype(np.int64)
iss = w[4096:4096 + 91 * 4].reshape(91, 4).astype(np.int64)
epi = w[4608:4608 + 4 * 7 * 2].reshape(4, 7, 2).astype(np.int64)
t0 = iss[0, 0]
rows = []
for ph in range(nph):
    wp = 4 * ph                      # row group 0 of each phase
    uu0 = (ph + nph - (91 % nph)) % nph
    for v in range(48):
        uu = uu0 + v * nph
        if uu >= 91:
            break
        s, x, m, st = gen[wp, uu // nph] - t0
        rows.append((uu, wp, s, x, m, st))
rows.sort()
print("chunk g c | warp start Xbuild mix sttm-wait | a_full issued period | sttm->a_full")
prev = 0
for uu, wp, s, x, m, st in rows:
    print(uu, uu // 13, uu % 13, "| w", wp, s, x - s, m - x, st - m, "|", iss[uu, 0] - t0, iss[uu, 2] - t0, iss[uu, 2] - t0 - prev, "|", iss[uu, 0] - t0 - st)
    prev = iss[uu, 2] - t0
for ew in range(4):
    print("epilogue warp", ew, [(int(epi[ew, g, 0] - t0), int(epi[ew, g, 1] - epi[ew, g, 0])) for g in range(7)])
