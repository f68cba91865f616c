"""Time the exact walk (k_scan + k_classify, chosen with XM_DEBUG_FORCE_GENERIC) on a resident synthetic pair.

    python scripts/time_exact_walk.py [--records N] [--steps K] [--warmup W] [--lib PATH ...]

Each --lib (default: the package's library) is timed in a process of its own through XM_LIB_PATH, in alternating
rounds, so that two builds can be compared in one visit.  Every round prints one JSON line: the mean and median of
res.ms_scan / res.ms_classify (CUDA events around each kernel) over the timed calls, the kernels that ran, the bin
lengths and the category counts (the same for every build of the same walk), the GPU's name and power limit.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def generate(ctx, R, threads, chunk=4_000_000):
    """records [0, R) of the single-end synthetic pair, generated on the host a chunk at a time and copied to the device"""
    from xenomapper_b200 import synth
    sp, ss = synth.generate(20000, seed=1, style=synth.STYLE_SE_BOWTIE2)
    cap_p, cap_s = R * (int(sp.nbytes / 20000 * 1.015) + 2) + (1 << 20), R * (int(ss.nbytes / 20000 * 1.015) + 2) + (1 << 20)
    d_p, d_s = ctx.dev_alloc(cap_p), ctx.dev_alloc(cap_s)
    len_p = len_s = 0
    for lo in range(0, R, chunk):
        n = min(chunk, R - lo)
        per = (n + threads - 1) // threads
        parts = [None] * threads

        def work(t):
            a = lo + t * per
            k = max(0, min(per, lo + n - a))
            if k:
                parts[t] = synth.generate(k, seed=1, style=synth.STYLE_SE_BOWTIE2, first=a)
        th = [threading.Thread(target=work, args=(t,)) for t in range(threads)]
        [t.start() for t in th]
        [t.join() for t in th]
        for part in parts:
            if part is None:
                continue
            p, s = part
            assert len_p + p.nbytes <= cap_p and len_s + s.nbytes <= cap_s
            ctx.h2d(d_p + len_p, p)
            ctx.h2d(d_s + len_s, s)
            len_p += p.nbytes
            len_s += s.nbytes
    return d_p, len_p, d_s, len_s


def child(args):
    import ctypes as C
    from xenomapper_b200 import _lib
    ctx = _lib.Context(0)
    d_p, len_p, d_s, len_s = generate(ctx, args.records, max(1, os.cpu_count() or 1))
    ctx.set_debug(_lib.DEBUG_FORCE_GENERIC)
    opts = ctx.opts(mode=_lib.MODE_SE, skip_repeated=True)
    res = _lib.Result()
    rc = ctx.lib.xm_classify_device(ctx.h, d_p, len_p, d_s, len_s, C.byref(opts), (C.c_void_p * 6)(), (C.c_uint64 * 6)(), C.byref(res))
    assert rc in (_lib.XM_OK, _lib.XM_ERR_ARG), ctx.error()
    out_len = [int(res.out_len[b]) for b in range(6)]
    d_out = [ctx.dev_alloc(n + 64) for n in out_len]
    ms_scan, ms_cls = [], []
    for k in range(args.warmup + args.steps):
        rc, r = ctx.classify_device(d_p, len_p, d_s, len_s, opts, d_out, [n + 64 for n in out_len])
        assert rc == _lib.XM_OK, ctx.error()
        if k >= args.warmup:
            ms_scan.append(float(r.ms_scan))
            ms_cls.append(float(r.ms_classify))
    gpu = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip()
    print(json.dumps(dict(lib=os.environ.get("XM_LIB_PATH", _lib.LIB_PATH), gpu=gpu, records=args.records, bytes_in=len_p + len_s,
                          steps=args.steps, kernels=ctx.walk_kernels(),
                          ms_scan_mean=statistics.mean(ms_scan), ms_scan_median=statistics.median(ms_scan),
                          ms_classify_mean=statistics.mean(ms_cls), ms_classify_median=statistics.median(ms_cls),
                          ms_classify_all=ms_cls, out_len=[int(r.out_len[b]) for b in range(6)], counts=list(r.counts)[:6])), flush=True)
    ctx.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--records", type=int, default=100_000_000)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--rounds", type=int, default=2)
    ap.add_argument("--lib", action="append", default=[])
    ap.add_argument("--child", action="store_true")
    args = ap.parse_args()
    if args.child:
        return child(args)
    libs = args.lib or [""]
    rows = {lib: [] for lib in libs}
    for _ in range(args.rounds):
        for lib in libs:
            env = dict(os.environ)
            if lib:
                env["XM_LIB_PATH"] = os.path.abspath(lib)
            r = subprocess.run([sys.executable, os.path.abspath(__file__), "--child", "--records", str(args.records),
                                "--steps", str(args.steps), "--warmup", str(args.warmup)], env=env, capture_output=True, text=True)
            if r.returncode:
                sys.stderr.write(r.stderr)
                raise SystemExit("round failed for %s" % (lib or "the package library"))
            line = r.stdout.strip().splitlines()[-1]
            print(line, flush=True)
            rows[lib].append(json.loads(line))
    summary = {lib or "package": dict(ms_classify_median=[x["ms_classify_median"] for x in v], ms_scan_median=[x["ms_scan_median"] for x in v])
               for lib, v in rows.items()}
    same = len({json.dumps([x["out_len"], x["counts"]]) for v in rows.values() for x in v}) == 1
    print(json.dumps(dict(summary=summary, same_outputs=same)))


if __name__ == "__main__":
    main()
