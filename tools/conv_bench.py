"""Per-layer tcgen05 convolution micro-benchmark (drs_bench_conv) over DRS_EXP_MODE timing experiments.

    python tools/conv_bench.py [--modes -1,2,3,7,8,9,10,12] [--pixels 757500] [--bf16]

Prints us per launch and TFLOP/s for the layer shapes of dilated_grsl_rate8 (k, rate, Ci, Co)."""
import ctypes as C, os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import drs_b200
from drs_b200 import lib as L

LAYERS = [("conv2", 5, 1, 64, 64), ("conv3", 4, 2, 64, 128), ("conv4", 4, 2, 128, 128), ("conv5", 3, 3, 128, 192),
          ("conv6", 3, 3, 192, 192), ("conv7", 3, 4, 192, 256), ("conv8", 3, 4, 256, 256)]


DENSE = [("d2", 5, 1, 32, 32), ("d3", 4, 2, 64, 64), ("d4", 4, 2, 128, 64), ("d5", 3, 3, 192, 128), ("d6", 3, 3, 320, 128),
         ("g6", 3, 3, 128, 320), ("g5", 3, 3, 128, 192), ("g4", 4, 2, 64, 128), ("g3", 4, 2, 64, 64), ("g2", 5, 1, 32, 32)]


def word(spec):
    """'-1' production default; otherwise tokens m<mode> k<K blocks per stage> i1 (instrumented)
    p1 / p2 (force single 128-pixel units / pairs of units per filter slice), e.g. k2 or k2m10i1 or p1."""
    import re
    if re.fullmatch(r"-?\d+", spec):
        return int(spec)
    w = 0
    for key, val in re.findall(r"([mkip])(\d+)", spec):
        val = int(val)
        w |= val if key == "m" else (val << 12 if key == "k" else ((val & 1) << 16 if key == "i" else (val & 3) << 20))
    return w


def main():
    args = sys.argv[1:]
    modes = [-1]
    crop, pixels, prec, reps = 25, 757500, "f16", 5
    only = None
    while args:
        a = args.pop(0)
        if a == "--modes":
            modes = [word(v) for v in args.pop(0).split(",")]
        elif a == "--pixels":
            pixels = int(args.pop(0))
        elif a == "--crop":
            crop = int(args.pop(0))
        elif a == "--bf16":
            prec = "bf16"
        elif a == "--reps":
            reps = int(args.pop(0))
        elif a == "--dense":
            LAYERS[:] = DENSE
        elif a == "--layers":
            only = args.pop(0).split(",")
    B = max(1, pixels // (crop * crop))
    s = drs_b200.Session("dilated_grsl_rate8", 5, 6, precision=prec, seed=1)
    lib = L.load()
    print("B=%d crop=%d pixels=%d %s reps=%d" % (B, crop, B * crop * crop, prec, reps))
    for name, k, rate, ci, co in LAYERS:
        if only and name not in only:
            continue
        row = []
        for m in modes:
            ms = C.c_float()
            ins = (C.c_uint32 * 10)()
            L.check(lib.drs_bench_conv(s._h, B, crop, k, rate, ci, co, L.PREC[prec], m, reps, C.byref(ms), ins))
            fl = 2.0 * B * crop * crop * k * k * ci * co
            tag = "prod" if m < 0 else "m%d%s" % (m & 0xff, "k%d" % ((m >> 12) & 0xf) if (m >> 12) & 0xf else "")
            txt = "%s %.0fus %.0fTF" % (tag, ms.value * 1e3, fl / ms.value / 1e9)
            if m >= 0 and (m >> 16) & 1:
                v = list(ins)
                st = max(v[2], 1)
                txt += (" [cyc/stage: producer %.0f = wait %.0f + expect_tx %.0f + tma %.0f + rest; mma %.0f = wait %.0f + mma %.0f "
                        "+ commit %.0f + rest (accumulator wait %.0f); %d stages, %.2f GHz]" %
                        (v[0] / st, v[1] / st, v[3] / st, v[4] / st, v[5] / st, v[6] / st, v[7] / st, v[8] / st, v[9] / st, v[2],
                         v[5] / (ms.value * 1e6)))
            row.append(txt)
        print("%s k%d r%d %dx%d: %s" % (name, k, rate, ci, co, " | ".join(row)), flush=True)
    s.close()


if __name__ == "__main__":
    main()
