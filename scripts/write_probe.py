"""Cost of the database write paths on S8 (2^17 items x 8 KiB, tcgen05 layout), one JSON line per case.

    python scripts/write_probe.py [--out FILE] [--old-sdk DIR]

Cases: looped update_item_raw over 1024 random full-size items; update_many_items with bodies of 1, 16, 1024 and 16384
random full-size items; one body rewriting all 2^17 items in index order beside uploading the same database (upload_slice
of every slice, which is what b200pir_db_upload does); load_raw_file of a 1 GiB raw file.  With --old-sdk DIR (a directory
holding another build's sdk_b200 package) the update_item_raw loop and load_raw_file also run on that build, alternating
with this one, each in a subprocess of its own.  The first line names the card and its power limit.  Timings are host clocks
around calls that synchronise the device before they return; the median of the repetitions is reported."""
import argparse
import json
import os
import struct
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
S8 = dict(n=2, nu_1=9, nu_2=8, p=256, q2_bits=22, t_gsw=8, t_conv=4, t_exp_left=8, t_exp_right=8, instances=1,
          db_item_size=8192, version=0)
ITEM = 8192
N_ITEMS = 1 << 17


def body_of(idxs, rng):
    import numpy as np
    data = rng.integers(0, 256, (len(idxs), ITEM), dtype=np.uint8)
    return b"".join(struct.pack(">II", 4 + ITEM, int(i)) + data[k].tobytes() for k, i in enumerate(idxs))


def median_time(fn, reps):
    fn()                                                    # warm-up: staging buffers, module load
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        ts.append(time.perf_counter() - t0)
    ts.sort()
    return ts[len(ts) // 2]


def child(case, sdk, raw_path):
    """one measurement in this process, on the sdk_b200 package found in `sdk`"""
    sys.path.insert(0, sdk)
    import numpy as np
    import sdk_b200.spiral as S
    G = S.Params(**S8)
    db = S.Database(G)
    rng = np.random.default_rng(1)
    if case == "update_item_raw_loop":
        idxs = rng.integers(0, N_ITEMS, 1024)
        data = rng.integers(0, 256, (1024, ITEM), dtype=np.uint8)
        def loop():
            for k, i in enumerate(idxs):
                db.update_item_raw(int(i), data[k])
        dt = median_time(loop, 5)
        out = {"case": case, "items": 1024, "seconds": dt, "items_per_s": 1024 / dt}
    elif case == "load_raw_file":
        dt = median_time(lambda: S.check(S.LIB.b200pir_db_load_raw_file(G._h, db._h, raw_path.encode())), 2)
        out = {"case": case, "bytes": os.path.getsize(raw_path), "seconds": dt}
    else:
        raise SystemExit("unknown case " + case)
    db.close()
    G.close()
    out["build"] = os.path.basename(os.path.normpath(sdk))
    print(json.dumps(out), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out")
    ap.add_argument("--old-sdk")
    ap.add_argument("--child", nargs=3, metavar=("CASE", "SDK", "RAW"))
    a = ap.parse_args()
    if a.child:
        return child(*a.child)
    lines = []

    def emit(d):
        print(json.dumps(d), flush=True)
        lines.append(d)

    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    emit({"case": "device", "nvidia_smi": smi[0] if smi else "unavailable"})
    sys.path.insert(0, ROOT)
    import numpy as np
    import sdk_b200.spiral as S
    G = S.Params(**S8)
    db = S.Database(G)
    rng = np.random.default_rng(2)
    for n in (1, 16, 1024, 16384):
        body = body_of(rng.integers(0, N_ITEMS, n), rng)
        dt = median_time(lambda: db.update_many_items(body), 7 if n < 16384 else 5)
        emit({"case": "update_many_items", "entries": n, "seconds": dt, "items_per_s": n / dt,
              "plaintext_MB_per_s": n * ITEM / dt / 1e6})
    body = body_of(np.arange(N_ITEMS), rng)
    dt = median_time(lambda: db.update_many_items(body), 3)
    emit({"case": "update_many_items_all_items", "entries": N_ITEMS, "seconds": dt, "plaintext_MB_per_s": N_ITEMS * ITEM / dt / 1e6})
    del body
    slices = S8["instances"] * S8["n"] ** 2
    words = rng.integers(0, 1 << 56, 512 * 256 * 2048, dtype=np.uint64)           # one slice, reused for each
    dt = median_time(lambda: [db.upload_slice(s, words) for s in range(slices)], 3)
    emit({"case": "db_upload", "slices": slices, "seconds": dt})
    del words
    db.close()
    G.close()
    with tempfile.TemporaryDirectory() as tmp:
        raw = os.path.join(tmp, "raw.bin")
        with open(raw, "wb") as f:
            for _ in range(N_ITEMS * ITEM // (64 << 20)):
                f.write(rng.integers(0, 256, 64 << 20, dtype=np.uint8).tobytes())
        builds = [ROOT] + ([os.path.abspath(a.old_sdk)] if a.old_sdk else [])
        for rep in range(2):
            for case in ("update_item_raw_loop", "load_raw_file"):
                for sdk in (builds if rep == 0 else builds[::-1]):
                    r = subprocess.run([sys.executable, os.path.abspath(__file__), "--child", case, sdk, raw],
                                       capture_output=True, text=True)
                    if r.returncode:
                        sys.stderr.write(r.stderr)
                        raise SystemExit("child %s on %s failed" % (case, sdk))
                    d = json.loads(r.stdout.strip().splitlines()[-1])
                    d["build"] = "this" if sdk == ROOT else "old"
                    d["rep"] = rep
                    emit(d)
    if a.out:
        with open(a.out, "w") as f:
            for d in lines:
                f.write(json.dumps(d) + "\n")


if __name__ == "__main__":
    main()
