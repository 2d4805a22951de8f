"""Band decode (mcgra_decode_band) at n = 65 536 on one GPU: CUDA-event time of one row band of the GraphMI result, the
bytes it writes over that time, and its share of the measured copy peak.

The kernel is a pure write stream of (b1 - b0) * n * 4 bytes (the 4 MB embedding it reads stays in L2), far beyond the
126 MB L2.  In the same call it times, for comparison:
  * a device-to-device copy of the same size (cudaMemcpyAsync: reads and writes the bytes, counted twice) and a fill
    (write only): the copy and write ceilings of this card;
  * the same band with mcgra_gram_accumulate variant 4 after a zero fill (what the MC-GRA ensemble uses at world > 1).
The copy peak of `MEASURED_PEAKS.json: hbm_gbs` is used when the file is present.

    python tools/decode_band_bench.py [--n 65536] [--rows 8192] [--reps 20] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else "unknown"


def timed(fn, reps):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps


def main():
    p = argparse.ArgumentParser()
    p.add_argument("--n", type=int, default=65536)
    p.add_argument("--rows", type=int, default=8192)
    p.add_argument("--reps", type=int, default=20)
    p.add_argument("--out", default=None)
    a = p.parse_args()
    from mcgra_b200 import _native as N
    n, rows = a.n, a.rows
    b0, b1 = n // 4, n // 4 + rows
    st = N.stream_ptr()
    g = torch.Generator(device="cuda").manual_seed(3)
    z = torch.randn(n, 16, device="cuda", generator=g)
    zn = torch.empty_like(z)
    N.call("mcgra_row_normalize", N.ptr(z), n, 16, 2.0, N.ptr(zn), st)
    out = torch.empty(rows, n, device="cuda")
    src = torch.empty(rows, n, device="cuda")
    nbytes = rows * n * 4

    def band():
        N.call("mcgra_decode_band", N.ptr(zn), n, b0, b1, N.ptr(out), n, st)

    def gram4():
        out.zero_()
        N.call("mcgra_gram_accumulate", N.ptr(zn), 16, n, 4, None, out.data_ptr() - b0 * n * 4, n, b0, b1, st)

    res = {}
    for _ in range(2):            # alternate, twice: the spread of the same measurement
        for name, fn in (("decode_band", band), ("copy_d2d", lambda: out.copy_(src)), ("fill", lambda: out.fill_(1.0)),
                         ("zero_fill_plus_gram_accumulate_v4", gram4)):
            res.setdefault(name, []).append(timed(fn, a.reps))
    band()
    torch.cuda.synchronize()
    peaks = {}
    pk = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(pk):
        peaks = json.load(open(pk))
    copy_gbs = [2 * nbytes / (ms * 1e-3) / 1e9 for ms in res["copy_d2d"]]
    ref = float(peaks["hbm_gbs"]) if "hbm_gbs" in peaks else max(copy_gbs)
    ms = min(res["decode_band"])
    report = dict(card=card(), n=n, band=[b0, b1], bytes_written=nbytes, ms=res,
                  decode_band_gbs=nbytes / (ms * 1e-3) / 1e9,
                  copy_peak_gbs=ref, copy_peak_source="MEASURED_PEAKS.json hbm_gbs" if "hbm_gbs" in peaks
                  else "copy_d2d of this run",
                  copy_d2d_gbs=copy_gbs, fill_gbs=[nbytes / (t * 1e-3) / 1e9 for t in res["fill"]],
                  fraction_of_copy_peak=nbytes / (ms * 1e-3) / 1e9 / ref)
    print(json.dumps(report))
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(report, f, indent=1)


if __name__ == "__main__":
    main()
