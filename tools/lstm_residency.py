"""Co-residency of the persistent LSTM recurrence (csrc/lstm_persistent.cu) on this device, for every shape the shape rules
admit: how many forward CTAs and backward 4-CTA clusters fit at once at the shared memory each launch uses, and whether
icd_lstm_seq_supported admits the shape.  Queries the occupancy calculator only; launches no kernel.

    python tools/lstm_residency.py [--out FILE.json]
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    import icd_b200  # noqa: F401
    from icd_b200._lib import check, lib
    assert torch.cuda.is_available(), "needs a GPU"
    torch.cuda.init()
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                          capture_output=True, text=True).stdout.strip()
    rows = []
    for B in (1, 128, 256, 384, 512):                     # 1 .. 4 row tiles: the shared memory depends on nothing else but H
        for H in range(16, 4 * 148 + 1, 16):
            if not lib().icd_lstm_seq_shape_ok(B, 1, H):
                continue
            f, b = ctypes.c_int(0), ctypes.c_int(0)
            check(lib().icd_lstm_seq_residency(B, H, ctypes.byref(f), ctypes.byref(b)), "icd_lstm_seq_residency")
            rows.append(dict(B=B, H=H, fwd_ctas=H // 4, fwd_fit=f.value, bwd_clusters=H // 16, bwd_fit=b.value,
                             admitted=bool(lib().icd_lstm_seq_supported(B, 1, H))))
    largest = {B: max([r["H"] for r in rows if r["B"] == B and r["admitted"]], default=0) for B in (1, 128, 256, 384, 512)}
    res = dict(card=card, sms=torch.cuda.get_device_properties(0).multi_processor_count, largest_admitted_H=largest,
               rows=rows)
    for r in rows:
        print("B=%3d H=%3d  fwd %3d CTAs / %3d fit   bwd %2d clusters / %2d fit   %s"
              % (r["B"], r["H"], r["fwd_ctas"], r["fwd_fit"], r["bwd_clusters"], r["bwd_fit"],
                 "admitted" if r["admitted"] else "REFUSED"))
    print("card:", card)
    print("largest admitted H:", largest)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            json.dump(res, fh, indent=1)


if __name__ == "__main__":
    main()
