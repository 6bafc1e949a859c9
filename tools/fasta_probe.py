"""FASTA text -> resident sequences on one GPU (import_fasta, DESIGN §4.7): device parse + pack against the copy of
the text, for a 3.1 Gbp genome (24 contigs, 60 columns) and a C2-shaped fg / bg pair (100 000 + 100 000 x 500 bp,
80 columns), both in pinned host buffers; the existing kmerlr_sequences_create on the flattened buffers and a numpy
stand-in for the host parse (NOT the Go reader, which cannot run here) beside them; a genome of about --e2e-gbp
(8 contigs of random length: 367 Mbp with the default seed) end to end to wiggle bytes through both paths.  Prints
one JSON object; the card's name and power limit are part of it.

    python tools/fasta_probe.py [--genome-gbp 3.1] [--reps 5] [--out result.json]
"""
import argparse
import ctypes as C
import hashlib
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import kmerlr_b200 as K  # noqa: E402

HBM_PEAK = 6533.5e9   # bytes/s, the HBM peak the project quotes (DESIGN §0)


def card():
    q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                       capture_output=True, text=True, timeout=30).stdout.strip()
    name, power = [x.strip() for x in q.split(",")]
    return name, power


def fasta_text(lens, width, rng, prefix=b"chr"):
    """a FASTA text of random bases (from a 4 MiB random pool) in a pinned host buffer; returns (tensor, array)"""
    pool = np.frombuffer(b"ACGTacgtN", dtype=np.uint8)[rng.integers(0, 9, 1 << 22)]
    heads = [b">%s%d\n" % (prefix, i + 1) for i in range(len(lens))]
    sizes = [len(h) + n + (n + width - 1) // width for h, n in zip(heads, lens)]
    pin = torch.empty(sum(sizes), dtype=torch.uint8).pin_memory()
    a = pin.numpy()
    p, q = 0, 0
    for h, n in zip(heads, lens):
        a[p:p + len(h)] = np.frombuffer(h, dtype=np.uint8)
        p += len(h)
        full, r = divmod(n, width)
        body = a[p:p + full * (width + 1)].reshape(full, width + 1)
        idx = (q + np.arange(full * width, dtype=np.int64)) & ((1 << 22) - 1)
        body[:, :width] = pool[idx].reshape(full, width)
        body[:, width] = 10
        p += full * (width + 1)
        q += full * width
        if r:
            a[p:p + r] = pool[(q + np.arange(r)) & ((1 << 22) - 1)]
            a[p + r] = 10
            p += r + 1
            q += r
    assert p == len(a)
    return pin, a


def numpy_parse(a):
    """numpy stand-in for the host parse of a clean text (no blanks inside lines): (flat bases, offsets)"""
    ends = np.flatnonzero(a == 10)
    starts = np.concatenate([[0], ends[:-1] + 1])
    hdr = a[starts] == ord(">")
    mark = np.zeros(len(a) + 1, dtype=np.int8)
    np.add.at(mark, starts[hdr], 1)
    np.add.at(mark, ends[hdr], -1)
    keep = (np.cumsum(mark[:-1], dtype=np.int8) == 0) & (a != 10) & (a != 13)
    seq = a[keep]
    kept = np.where(hdr, 0, ends - starts - (a[ends - 1] == 13))
    koff = np.concatenate([[0], np.cumsum(kept)])
    off = np.append(koff[np.flatnonzero(hdr)], koff[-1]).astype(np.int64)
    return seq, off


def traffic(T, L, bases):
    """bytes the kernels of the device parse read and write (DESIGN §4.7): the text three times (line count, line
    ends, pack), 8-byte per-line arrays (line ends 8 L; classify 16 L in, 24 L out; two scans 48 L; records 24 L;
    pack 24 L of line metadata), 6 bytes of packed output per 16 bases"""
    return 3 * T + 144 * L + bases * 6 // 16


def timed(f, reps):
    ts = []
    for _ in range(reps):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        r = f()
        torch.cuda.synchronize()
        ts.append(time.perf_counter() - t0)
        if hasattr(r, "free"):
            r.free()
    return float(np.median(ts)) * 1e3


def measure(label, pin, a, reps, texts=None):
    texts = texts or [a]
    T = len(a)
    L = int(np.count_nonzero(a == 10))
    dev = torch.empty(T, dtype=torch.uint8, device="cuda")
    copy_ms = timed(lambda: dev.copy_(pin, non_blocking=True), reps)
    del dev
    s = K.import_fasta(*texts)
    bases, n = s.total_bases, s.n
    s.free()
    K.api.profile(True)
    s = K.import_fasta(*texts)
    prof = K.api.profile_dump()
    K.api.profile(False)
    s.free()
    kernel_ms = sum(v[0] for v in prof.values())
    total_ms = timed(lambda: K.import_fasta(*texts), reps)
    device_ms = K.last_device_ms()
    byts = traffic(T, L, bases)
    # the existing path: kmerlr_sequences_create on the flattened buffers (pinned), and the numpy stand-in
    t0 = time.perf_counter()
    seq, off = numpy_parse(a)
    numpy_ms = (time.perf_counter() - t0) * 1e3
    pseq = torch.from_numpy(seq).pin_memory()
    create_ms = timed(lambda: K.Sequences((pseq.numpy(), off)), reps)
    return {
        "set": label, "text_bytes": T, "lines": L, "records": n, "bases": bases,
        "copy_ms": round(copy_ms, 3), "copy_GBps": round(T / copy_ms / 1e6, 1),
        "parse_pack_kernels_ms": round(kernel_ms, 3), "kernels": {k: round(v[0], 3) for k, v in prof.items()},
        "call_device_ms": round(device_ms, 3), "call_wall_ms": round(total_ms, 3),
        "parse_bytes": byts, "parse_GBps": round(byts / kernel_ms / 1e6, 1),
        "parse_fraction_of_hbm_peak": round(byts / (kernel_ms * 1e-3) / HBM_PEAK, 3),
        "parse_below_copy": kernel_ms < copy_ms,
        "existing_sequences_create_ms": round(create_ms, 3),
        "numpy_host_parse_stand_in_ms": round(numpy_ms, 1),
    }


def end_to_end(rng, gbp, tmp):
    """a genome text to wiggle bytes: text -> import_fasta -> regions -> resident scores -> save_wiggle, against
    host parse -> host slices -> kmerlr_score_windows -> save_wiggle"""
    lens = [int(x) for x in rng.integers(int(gbp * 1e9 / 8 * 0.5), int(gbp * 1e9 / 8 * 1.5), 8)]
    pin, a = fasta_text(lens, 60, rng)
    kc = K.NewKmerCounter(1, 6, revcomp=True)
    sample = a[:200_000]
    d = K.compile_test_data(None, kc, None, None, True, False, [bytes(sample[sample != 10][100:100_000])])
    ck, cc = d.Kmers()
    sel = np.sort(rng.choice(d.m, 40, replace=False))
    model = dict(counter=kc, class_k=ck[sel], class_code=cc[sel], features=[[i, i] for i in range(40)],
                 theta=rng.normal(size=41) * 0.1, summary="")
    g = K.genomicKmerLr([model])
    W, step = 200, 10
    # BED-like ranges: the middle 90 % of every contig
    reg = [(i, n // 20, n - n // 20) for i, n in enumerate(lens)]
    names = ["chr%d" % (i + 1) for i in range(len(lens))]
    wig = [(names[i], f) for i, f, _ in reg]
    slots = [K.api.lib().kmerlr_window_slots(t - f, W, step) for _, f, t in reg]
    out = {}
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    s = K.import_fasta(a)
    r = s.regions([x[0] for x in reg], [x[1] for x in reg], [x[2] for x in reg])
    h = C.c_uint64(0)
    K.api.check(K.api.lib().kmerlr_score_windows_resident(g._arr, 1, r.h, W, step, None, C.byref(h)))
    f1 = os.path.join(tmp, "text.wig")
    K.saveWindowPredictionsWiggle(f1, wig, slots, "probe", W, step, scores=h.value)
    out["text_path_ms"] = round((time.perf_counter() - t0) * 1e3, 1)
    K.api.check(K.api.lib().kmerlr_free(h.value))
    s.free(); r.free()
    t0 = time.perf_counter()
    seq, off = numpy_parse(a)
    parts = [seq[off[i] + f:off[i] + t] for i, f, t in reg]
    buf = np.concatenate(parts)
    boff = np.concatenate([[0], np.cumsum([len(p) for p in parts])]).astype(np.int64)
    preds = g.predict_window_genomic((buf, boff), W, step)
    f2 = os.path.join(tmp, "host.wig")
    K.saveWindowPredictionsWiggle(f2, wig, preds, "probe", W, step)
    out["existing_path_with_numpy_stand_in_ms"] = round((time.perf_counter() - t0) * 1e3, 1)
    digest = [hashlib.sha256(open(f, "rb").read()).hexdigest() for f in (f1, f2)]
    out.update(genome_bases=sum(lens), wiggle_bytes=os.path.getsize(f1), identical=digest[0] == digest[1])
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--genome-gbp", type=float, default=3.1)
    ap.add_argument("--e2e-gbp", type=float, default=0.384)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default="", help="also write the JSON object to this file")
    args = ap.parse_args()
    name, power = card()
    K.init(0)
    rng = np.random.default_rng(0)
    res = {"card": name, "power_limit": power, "hbm_peak_GBps": HBM_PEAK / 1e9}
    lens = [int(x) for x in rng.integers(int(args.genome_gbp * 1e9 / 24 * 0.4), int(args.genome_gbp * 1e9 / 24 * 1.6), 24)]
    lens = [int(x * args.genome_gbp * 1e9 / sum(lens)) for x in lens]
    pin, a = fasta_text(lens, 60, rng)
    res["genome"] = measure("genome %.1f Gbp, 24 contigs, 60 columns" % (sum(lens) / 1e9), pin, a, args.reps)
    del pin, a
    pf, af = fasta_text([500] * 100_000, 80, rng, b"fg")
    pb, ab = fasta_text([500] * 100_000, 80, rng, b"bg")
    both = torch.cat([pf, pb]).pin_memory()
    res["c2_pair"] = measure("C2 fg / bg 100 000 + 100 000 x 500 bp, 80 columns", both, both.numpy(), args.reps,
                             texts=[af, ab])
    with tempfile.TemporaryDirectory() as tmp:
        res["end_to_end_wiggle"] = end_to_end(rng, args.e2e_gbp, tmp)
    print(json.dumps(res, indent=1))
    if args.out:
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
