#!/usr/bin/env python
"""bench.py — headline benchmark of the bftkv signature-verify + quorum-tally hot path on B200.

Workload (BASELINE.json configs[1]): one batch of 65 536 RSA-2048 / SHA-256 PKCS#1 v1.5 signature
verifies over 16 keys (1 % corrupted, 0.1 % unknown signer; SURVEY §8d config 2), synthetic.
A "step" = one pass of the hot path over one such batch.  N GPUs = N independent shards
(weak scaling, no collective on the data path; torch.distributed is used only for the barrier and
the max-over-ranks time).

  value        verifies/s, inputs already resident in HBM (device API, CUDA events on the launch stream), K steps
  sustained    the same leg run for >= 2 s (value_sustained) with the clocks sampled over exactly that region
  e2e          verifies/s through the reference-facing operator bftq_signature_verify_batch (= crypto.Signature.Verify's
               batch form): OpenPGP packets + signed bytes in PAGE-LOCKED HOST blobs (bftq_host_alloc, what the shim's
               aggregator fills), H2D + K0 parse/digest + K1 + D2H inside the timed region; e2e.sustained = >= 2 s
  e2e_pageable the same call with the blobs in pageable memory (the library stages them itself)
  e2e_flat     the flat tuple call (bftq_rsa_verify_batch, pinned host buffers, digests precomputed)
  quorum_ops   BASELINE configs[2] device-resident (65 536 read ops x 16 replicas, K1 + K2) and, in `e2e`, this rank's
               shard of configs[4] (1 048 576 read ops x 31 replicas over 8 GPUs = 131 072 ops x 31 per GPU) through
               bftq_verify_read_batch from page-locked host buffers: quorum-certified ops/s end to end
  roofline     integer-ALU bound: 156 864 32x32->64 MACs per verify (SURVEY §8d) x verifies / kernel
               time, against the IMAD.WIDE rate measured live on the same GPU (bftq_measure_int_peak)
  cpu_baseline the libcrypto stand-in for the Go CPU path (SURVEY §8d(2): EVP_PKEY_verify, one pthread per core) and
               the plain-C port of the oracle beside it (rank 0, N=1)

`--impl reference` times the CPU stand-in of the reference path (libcrypto when built, else the oracle's C port; the Go
reference itself cannot be built here: no Go toolchain, un-vendored x/crypto) on all host threads.

`--dump-outputs DIR` writes what the `value` leg (or, with `--impl reference`, the CPU stand-in) returned in its last timed
step as DIR/status.npy: the per-signature status bytes as float32 (DIR/status_rank<r>.npy per rank when N > 1).  The
inputs are seeded, so two builds run with the same arguments can be compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

MACS_PER_VERIFY = 156864          # 19 Montgomery products x (2*64^2 + 64) word-MACs, SURVEY §8(d)
EXECUTED_MACS_PER_VERIFY = 2 * 8192 + 16 * (4096 + 2176)     # 2 general products + 16 squarings (544 a x a + 1024 n x q IMAD.WIDE per lane)
NCU_DRAM_BYTES_PER_LAUNCH = 19225600      # profiles/ncu_rsa_verify_r02c_unified.txt: 19.2256 MB read + 0 B written per 65536-item launch
BYTES_PER_VERIFY = 549            # n 256 + s 256 + digest 32 + key idx 4 + status 1, SURVEY §8(d)
ITEMS = 65536
NKEYS = 16
WORKLOAD = ("batch 65536 RSA-2048 PGP signature verifies (BASELINE configs[1]), 16 keys, e=65537, SHA-256, "
            "1% corrupted + 0.1% unknown signer")
# K1b (ed25519_fast.cuh): expected 21.4 + 26.0 non-zero signed digits (radix 2^12 for S / the base point, 2^10 for k / the key) x 7 field
# products (100 IMAD.WIDE each) per mixed addition + 126 word products of the Barrett reduction + kernel 2: 5 products per signature + 1/8 of
# an inversion (254 squarings x 55 + 11 x 100)
ED25519_MACS = int(47.4 * 700 + 126 + 500 + (254 * 55 + 11 * 100) / 8)        # = 35 689 executed 32x32->64 multiplies per verification


def host_cores():
    """Usable host cores: affinity mask capped by the cgroup CPU quota (containers on the GPU box
    are quota-limited well below the 128 hardware threads)."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            n = max(1, min(n, int(int(q) / int(per) + 0.5)))
    except Exception:
        pass
    return n


def cgroup_throttled():
    """(nr_throttled, throttled_usec) of this container's CPU controller (CFS quota), or None."""
    try:
        d = dict(l.split() for l in open("/sys/fs/cgroup/cpu.stat").read().strip().splitlines())
        return int(d.get("nr_throttled", 0)), int(d.get("throttled_usec", 0))
    except Exception:
        return None


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx, self.rows, self.proc = gpu_index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                          "-i", str(self.idx), "-lms", "100"], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")] + [time.perf_counter()])

    def mark(self):
        return time.perf_counter()

    def window(self, t0, t1):
        """Clocks of the samples taken between two mark()s."""
        rows = [r for r in self.rows if len(r) >= 9 and t0 <= r[-1] <= t1 and r[1].replace(".", "").isdigit()]
        sm = sorted(int(float(r[1])) for r in rows)
        pw = [float(r[3]) for r in rows if r[3].replace(".", "").isdigit()]
        return {"sm_mhz_median": sm[len(sm) // 2] if sm else None, "sm_mhz_min": sm[0] if sm else None, "samples": len(sm),
                "power_w_max": max(pw) if pw else None}

    def stop(self):
        if self.proc:
            self.proc.terminate()
        sm = sorted(int(float(r[1])) for r in self.rows if len(r) >= 9 and r[1].replace(".", "").isdigit())
        mx = [int(float(r[2])) for r in self.rows if len(r) >= 9 and r[2].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows if len(r) >= 9 for i in range(4) if r[4 + i].lower().startswith("active")})
        # the busiest samples are the ones under load: take the upper half
        under = sm[len(sm) // 2:] if sm else []
        return {"sm_mhz": under[len(under) // 2] if under else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


def dump_outputs(out_dir, arrays, rank, world):
    """Writes each array as out_dir/<name>.npy in float32 (exact for the byte-sized statuses dumped here)."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ("_rank%d" % rank if world > 1 else "") + ".npy"), np.asarray(a, np.float32))


def w_pool_clean(w):
    """The genuinely signed, known-key subset of a config-2 batch, as a pool for config 3."""
    import numpy as np
    keep = np.nonzero(w["expect"] == 0)[0]
    return {"keys": w["keys"], "key_idx": w["key_idx"][keep], "sig": w["sig"][keep], "digest": w["digest"][keep]}


def cpu_verify(w, threads, reps, kind):
    """kind 'libcrypto' (SURVEY §8d(2) stand-in) or 'port' (the oracle's plain-C restatement)."""
    from oracle import c_oracle
    ns, es = [k["n"] for k in w["keys"]], [k["e"] for k in w["keys"]]
    fn = c_oracle.libcrypto_rsa_verify_batch if kind == "libcrypto" else c_oracle.rsa_verify_batch
    fn(ns, es, w["key_idx"][:512], w["sig"][:512], w["digest"][:512], threads=threads)   # warm
    t0 = time.perf_counter()
    for _ in range(reps):
        st = fn(ns, es, w["key_idx"], w["sig"], w["digest"], threads=threads)
    dt = time.perf_counter() - t0
    return ITEMS * reps / dt, st


CPU_KIND_TEXT = {
    "libcrypto": "OpenSSL libcrypto EVP_PKEY_verify (RSA_PKCS1_PADDING, SHA-256 digest given), one pthread per usable core: the stand-in "
                 "SURVEY §8(d)(2) prescribes for crypto/pgp -> rsa.VerifyPKCS1v15 on boxes without Go",
    "port": "oracle/c plain-C port (u128 CIOS Montgomery) of crypto/pgp -> rsa.VerifyPKCS1v15",
}


def run_reference(args, rank, world):
    if rank != 0:
        return
    from bftkv_b200 import workload
    from oracle import c_oracle
    threads = host_cores()
    kind = "libcrypto" if c_oracle.libcrypto_available() else "port"
    w = workload.make_verify_batch(ITEMS, NKEYS)
    for _ in range(args.warmup):
        cpu_verify(w, threads, 1, kind)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        rate, st = cpu_verify(w, threads, 1, kind)
    dt = time.perf_counter() - t0
    assert (st == w["expect"]).all()
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"status": st}, rank, world)
    v = ITEMS * args.steps / dt
    port_rate, _ = cpu_verify(w, threads, 1, "port")
    print(json.dumps({
        "impl": "reference", "metric": "rsa2048_signature_verifies_per_sec", "value": v, "unit": "verifies/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u32/u64 integer", "data": "synthetic",
        "config": {"workload": WORKLOAD},
        "cpu_baseline": {"value": v, "unit": "verifies/s", "cores": threads, "kind": "port",
                         "sample": "the full 65536-item batch per step; " + CPU_KIND_TEXT[kind] +
                                   " (the Go reference is unbuildable here: no Go toolchain, un-vendored x/crypto)",
                         "implementation": kind, "plain_c_port_verifies_per_sec": port_rate},
        "e2e": {"value": v, "unit": "verifies/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


def run_gpu(args, rank, local_rank, world):
    import ctypes as C
    import numpy as np
    import torch
    import torch.distributed as dist
    from bftkv_b200 import Engine, workload
    from bftkv_b200 import _lib as L_
    from bftkv_b200.crypto_gpu import Keyring, _blob

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    # stdout carries exactly one JSON line: whatever libraries write to fd 1 meanwhile (NCCL's version banner under
    # NCCL_DEBUG=VERSION, for one) goes to stderr; the line itself is written to the saved descriptor at the end
    sys.stdout.flush()
    real_stdout = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    cores_rank = max(1, host_cores() // world)
    eng = Engine(local_rank)
    numa_node = eng.bind_thread()            # this rank's threads and page-locked buffers live on its GPU's NUMA node from here on
    w = workload.make_verify_batch(ITEMS, NKEYS, seed=0xBF7C0002 + rank, corrupt_seed=0xBF7C0003 + rank, threads=cores_rank)
    eng.register_rsa_keys([k["n"] for k in w["keys"]], [k["e"] for k in w["keys"]])
    int_peak = eng.measure_int_peak()
    vp = lambda a: C.c_void_p(a.ctypes.data)

    # ---- device-resident leg: COPIES distinct input sets (> L2) rotated between steps ----------
    copies = args.copies
    d_idx = [torch.from_numpy(w["key_idx"].astype(np.int32)).to(dev) for _ in range(copies)]
    d_sig = [torch.from_numpy(w["sig"]).to(dev) for _ in range(copies)]
    d_dig = [torch.from_numpy(w["digest"]).to(dev) for _ in range(copies)]
    d_st = [torch.empty(ITEMS, dtype=torch.uint8, device=dev) for _ in range(copies)]
    stream = torch.cuda.Stream(device=dev)
    # The timed launches alternate over NSTREAMS streams: the blocks of batch i+1 fill the partially occupied last
    # wave of batch i and the two batches run out of phase (one loads / compares while the other multiplies) —
    # what a server with several batches in flight gets anyway (tools/tail_experiment.py: +7.6 % over one stream).
    NSTREAMS = max(1, args.streams)
    streams = [stream] + [torch.cuda.Stream(device=dev) for _ in range(NSTREAMS - 1)]

    def step(i, st=None):
        c = i % copies
        eng.rsa_verify_batch_dev(d_idx[c], d_sig[c], d_dig[c], ITEMS, d_st[c], stream=(st or stream).cuda_stream)

    def barrier():
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def timed_launches(n):
        """n launches alternating over the streams, CUDA events around the whole region on the first stream."""
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record(stream)
        for st in streams[1:]:
            st.wait_event(ev0)
        for i in range(n):
            step(i, streams[i % NSTREAMS])
        for st in streams[1:]:
            stream.wait_stream(st)
        ev1.record(stream)
        stream.synchronize()
        return ev0.elapsed_time(ev1)

    # warm-up, serial on one stream, with per-launch events: the duration of one launch running alone
    evs = [torch.cuda.Event(enable_timing=True) for _ in range(args.warmup + 1)]
    evs[0].record(stream)
    for i in range(args.warmup):
        step(i)
        evs[i + 1].record(stream)
    stream.synchronize()
    serial_ms = sorted(evs[i].elapsed_time(evs[i + 1]) for i in range(1, args.warmup)) or [evs[0].elapsed_time(evs[1])]
    for i in range(NSTREAMS):
        step(i, streams[i])
    barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    launches0 = eng.stats()["launches"]
    barrier()
    dev_ms = timed_launches(args.steps)
    barrier()
    gpu_launches = eng.stats()["launches"] - launches0
    for c in range(min(copies, args.steps)):
        assert np.array_equal(d_st[c].cpu().numpy(), w["expect"]), "device-resident results differ from expectation"
    if args.dump_outputs:                    # the buffer the last timed step wrote, before the sustained leg reuses it
        dump_outputs(args.dump_outputs, {"status": d_st[(args.steps - 1) % copies].cpu().numpy()}, rank, world)
    # the same leg for >= SUSTAIN seconds: what the clocks do under a seconds-long integer load
    n_sus = max(args.steps, int(args.sustain * 1e3 / max(dev_ms / args.steps, 1e-3)) + 1)
    barrier()
    m0 = sampler.mark()
    sus_ms = timed_launches(n_sus)
    m1 = sampler.mark()
    barrier()
    assert np.array_equal(d_st[0].cpu().numpy(), w["expect"])

    # ---- end-to-end leg: pinned host buffers through the flat host C-ABI call ------------------------
    # NCALLERS concurrent callers (bftkv calls the crypto layer from one goroutine per peer,
    # transport/transport.go:110-127; the C ABI is re-entrant): while one call's kernel runs, the
    # other call's H2D copy is in flight.  Every step still copies its full inputs H2D and its
    # status bytes D2H inside the timed region.
    NCALLERS = max(1, min(args.callers, cores_rank))
    h_in = [(torch.from_numpy(w["key_idx"].astype(np.int32)).pin_memory(), torch.from_numpy(w["sig"]).pin_memory(),
             torch.from_numpy(w["digest"]).pin_memory(), torch.empty(ITEMS, dtype=torch.uint8).pin_memory()) for _ in range(NCALLERS)]

    def caller(c, n):
        eng.bind_thread()
        for _ in range(n):
            eng.rsa_verify_batch(h_in[c][0], h_in[c][1], h_in[c][2], out=h_in[c][3])

    def run_callers(fn, shares):
        """Runs fn(c, shares[c]) on one thread per caller; returns the seconds from the common start signal (given once
        every thread exists and waits — thread creation is not part of a step) to the last caller's return + device sync."""
        gun = threading.Event()

        def body(c):
            eng.bind_thread()
            gun.wait()
            fn(c, shares[c])
        ths = [threading.Thread(target=body, args=(c,)) for c in range(len(shares))]
        [t.start() for t in ths]
        time.sleep(0.002)
        t_start = time.perf_counter()
        gun.set()
        [t.join() for t in ths]
        torch.cuda.synchronize(dev)
        return time.perf_counter() - t_start

    def split(n, k):
        return [n // k + (1 if c < n % k else 0) for c in range(k)]
    share = split(args.steps, NCALLERS)
    # warm-up with the same concurrency as the timed region: the library grows its pool of pinned staging
    # slots on demand, and callers running together need more of them than one caller alone
    run_callers(caller, [args.warmup] * NCALLERS)
    barrier()
    e2e_s = run_callers(caller, share)
    barrier()
    for c in range(NCALLERS):
        if share[c]:
            assert np.array_equal(h_in[c][3].numpy(), w["expect"]), "end-to-end results differ from expectation"

    # ---- the box's host->device copy rate (context for the end-to-end legs: they move 292-373 B per verify) ----
    hb = torch.empty(256 << 20, dtype=torch.uint8).pin_memory()
    db = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    db.copy_(hb, non_blocking=True)
    torch.cuda.synchronize(dev)
    c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    c0.record()
    for _ in range(4):
        db.copy_(hb, non_blocking=True)
    c1.record()
    torch.cuda.synchronize(dev)
    h2d_gbps = 4 * (256 << 20) / (c0.elapsed_time(c1) * 1e-3) / 1e9
    del hb, db

    # ---- end-to-end leg through the reference-facing operator: Signature.Verify's batch form ---------
    # What bftkv hands to crypto.Signature.Verify (crypto_pgp.go:319-330): the signed bytes and a
    # SignaturePacket.Data holding one detached OpenPGP v4 signature packet, against a keyring of OpenPGP key
    # blocks.  One call per step over the whole batch, error codes out.  The blobs live in page-locked host memory
    # from bftq_host_alloc — the buffers the Go shim's aggregator appends each request to (Go memory itself can never
    # be DMA'd) — so the library DMAs them in place: per step H2D of the raw packets + offsets, K0 (OpenPGP parse +
    # issuer lookup + digest + hash-tag check on the GPU; flagged items through the host packer + K4), K1, D2H.
    # Nothing is precomputed outside the timed region.  `e2e_pageable` is the same call on pageable blobs.
    os.environ.setdefault("BFTQ_HOST_THREADS", str(min(16, max(1, cores_rank - 2))))       # leave the callers' own threads inside the CPU quota
    pw = workload.make_pgp_verify_batch(ITEMS, NKEYS, seed=0xBF7C0002 + rank, corrupt_seed=0xBF7C0003 + rank, threads=cores_rank)
    kr = Keyring(eng)
    kr.register(pw["keyring"])
    ptb, pto = _blob(pw["tbs"])
    psb, pso = _blob(pw["sigs"])
    pin = [eng.host_copy(a) for a in (ptb, pto, psb, pso)]
    # each caller brings one helper thread (K0 path): on a rank that owns few host cores more callers only spin
    PCALLERS = max(1, min(args.pgp_callers, cores_rank // 2))
    perr = [np.zeros(ITEMS, np.int32) for _ in range(PCALLERS)]

    def make_pgp_caller(blobs):
        def f(c, n):
            eng.bind_thread()
            for _ in range(n):
                L_.check(eng._lib.bftq_signature_verify_batch(kr._h, vp(blobs[0]), vp(blobs[1]), vp(blobs[2]), vp(blobs[3]), ITEMS, vp(perr[c])))
        return f
    pgp_pinned, pgp_pageable = make_pgp_caller(pin), make_pgp_caller((ptb, pto, psb, pso))
    run_callers(pgp_pinned, [args.warmup] * PCALLERS)
    pshare = split(args.steps, PCALLERS)
    st0, thr0 = eng.stats(), cgroup_throttled()
    barrier()
    pgp_s = run_callers(pgp_pinned, pshare)
    barrier()
    st1, thr1 = eng.stats(), cgroup_throttled()
    for c in range(PCALLERS):
        if pshare[c]:
            assert np.array_equal(perr[c] == 0, pw["expect_ok"]), "packet-level results differ from expectation"
    # sustained: the same callers for >= SUSTAIN seconds
    n_e2e_sus = max(args.steps, int(args.sustain / max(pgp_s / args.steps, 1e-6)) + 1)
    barrier()
    m2 = sampler.mark()
    pgp_sus_s = run_callers(pgp_pinned, split(n_e2e_sus, PCALLERS))
    m3 = sampler.mark()
    barrier()
    t0 = time.perf_counter()
    pgp_pinned(0, 3)
    pgp_single_ms = (time.perf_counter() - t0) / 3 * 1e3
    # pageable blobs (the library bounces them through its own pinned staging: round 1's headline leg)
    run_callers(pgp_pageable, [args.warmup] * PCALLERS)
    sp0 = eng.stats()
    barrier()
    pgp_pageable_s = run_callers(pgp_pageable, pshare)
    barrier()
    sp1 = eng.stats()
    # the same leg with the packets parsed by the host packer (BFTQ_GPU_PARSE=0) instead of K0, for context
    os.environ["BFTQ_GPU_PARSE"] = "0"
    run_callers(pgp_pinned, [args.warmup] * PCALLERS)
    host_packer_s = run_callers(pgp_pinned, pshare)
    del os.environ["BFTQ_GPU_PARSE"]
    for c in range(PCALLERS):
        if pshare[c]:
            assert np.array_equal(perr[c] == 0, pw["expect_ok"]), "packet-level results differ from expectation"
    tms = lambda a, b: {k: (b["packer_%s_ns" % k] - a["packer_%s_ns" % k]) / args.steps * 1e-6 for k in ("parse", "stage", "wait")}
    pgp_info = {"h2d": (st1["h2d_bytes"] - st0["h2d_bytes"]) // args.steps, "d2h": (st1["d2h_bytes"] - st0["d2h_bytes"]) // args.steps,
                "launches": (st1["launches"] - st0["launches"]) // args.steps, "threads": int(os.environ["BFTQ_HOST_THREADS"]),
                "chunks": (st1["packer_chunks"] - st0["packer_chunks"]) // args.steps, "callers": PCALLERS, "single_ms": pgp_single_ms,
                "host_packer_rate": ITEMS * args.steps / host_packer_s, "thread_ms": tms(st0, st1), "thread_ms_pageable": tms(sp0, sp1),
                "throttled": None if thr0 is None or thr1 is None else {"nr_throttled": thr1[0] - thr0[0], "throttled_usec": thr1[1] - thr0[1]}}
    kr.close()
    for a in pin:
        eng.host_free(a)

    # ---- server-side write path: CollectiveSignature.Verify's batch form (crypto_pgp.go:485-500, protocol/server.go:300) ---------
    # Each item: one TBSS string and a collective signature of 11 detached OpenPGP signature packets by members of a
    # 16-node clique (n = 16: f = 5, suff = 11; 2 % of the packets corrupted, so some items fall below suff).  The host
    # frames the packets (headers only), K0 parses + hashes every packet against its item's signed bytes, K1 verifies,
    # K2 decides IsSufficient per item.  Signed templates: 8 TBSS variants x 16 keys; items draw from them.
    from bftkv_b200.crypto_gpu import QCIds
    NC, NSIG = args.coll_items, 11
    crng = np.random.default_rng(0xBF7C0008 + rank)
    ckeys = workload.load_keys(16)
    cblocks, ckids = [], []
    for i, k in enumerate(ckeys):
        b_, kid_ = workload.pgp_public_key_block(k, workload._private_key(k), b"a%02d (http://localhost:57%02d) <a%02d@bftq.test>" % (i, i, i))
        cblocks.append(b_); ckids.append(kid_)
    ctbs = [workload.tbs_packet(bytes([j]) * 16, bytes([j + 1]) * 32, 1000 + j) for j in range(8)]
    csig = [[workload.sig_packet_v4(ckeys[i], ckids[i], 8, ctbs[j], 0x5F000000 + i) for i in range(16)] for j in range(8)]
    c_tbs, c_ss, c_expect = [], [], []
    for it in range(NC):
        j = int(crng.integers(0, 8))
        mem = crng.permutation(16)[:NSIG]
        parts, good = [], 0
        for i in mem:
            pkt = csig[j][int(i)]
            if crng.random() < 0.02:
                bb = bytearray(pkt); bb[-1 - int(crng.integers(0, 200))] ^= 0x04; pkt = bytes(bb)
            else:
                good += 1
            parts.append(pkt)
        c_tbs.append(ctbs[j]); c_ss.append(b"".join(parts)); c_expect.append(good >= 11)
    krc = Keyring(eng)
    krc.register(b"".join(cblocks))
    ctb, cto = _blob(c_tbs)
    csb, cso = _blob(c_ss)
    cpin = [eng.host_copy(a) for a in (ctb, cto, csb, cso)]
    carr = (QCIds * 1)(QCIds(5, 16, 11, 11, 0, 16))
    cmem = np.asarray(ckids, np.uint64)
    cerr = np.zeros(NC, np.int32)

    def cstep():
        L_.check(eng._lib.bftq_collective_verify_batch(krc._h, C.cast(carr, C.c_void_p), 1, vp(cmem), 16, vp(cpin[0]), vp(cpin[1]), vp(cpin[2]), vp(cpin[3]), NC, vp(cerr)))
    cstep()
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        cstep()
    coll_s = time.perf_counter() - t0
    barrier()
    assert np.array_equal(cerr == 0, np.array(c_expect)), "collective results differ from expectation"
    coll_accept = int((cerr == 0).sum())
    krc.close()
    for a in cpin:
        eng.host_free(a)

    # ---- secondary: quorum-certified read ops (BASELINE configs[2]), device-resident ----------------------------
    # 65536 read ops x 16 replicas: verify every response + wotqs read tally (K1 + K2, one stream).
    # Signed tuples are drawn from this rank's 65536-signature pool (each slot gets a genuine
    # signature by its replica's key; 1 M distinct signatures would take minutes to make).
    R, M = 16, 65536
    ro = workload.make_read_ops(w_pool_clean(w), M, R, seed=0xBF7C0004 + rank)
    quorum = eng.quorum_create([(5, 16, 6, 11, list(range(16)))])           # n=16: f=5, READ threshold 6, suff 11
    NQ = M * R
    dq = {k: torch.from_numpy(v).to(dev) for k, v in [("off", ro["op_off"].astype(np.int32)), ("idx", ro["key_idx"].astype(np.int32)),
                                                     ("sig", ro["sig"]), ("dig", ro["digest"]), ("pre", ro["pre_status"]),
                                                     ("ts", ro["ts"].astype(np.int64)), ("val", ro["value_id"].astype(np.int32))]}
    dq_st = torch.empty(NQ, dtype=torch.uint8, device=dev)
    dq_bits = torch.empty(M, dtype=torch.uint8, device=dev)
    dq_win = torch.empty(M, dtype=torch.int32, device=dev)

    def qstep():
        eng.verify_tally_batch_dev(quorum, dq["off"], dq["idx"], dq["sig"], dq["dig"], M, NQ, dq_st, dq_bits, d_pre=dq["pre"],
                                   d_ts=dq["ts"], d_value_id=dq["val"], d_winner=dq_win, stream=stream.cuda_stream)
    for _ in range(2):
        qstep()
    barrier()
    q0, q1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    q0.record(stream)
    for _ in range(args.steps):
        qstep()
    q1.record(stream)
    stream.synchronize()
    barrier()
    q_ms = q0.elapsed_time(q1)
    assert np.array_equal(dq_st.cpu().numpy(), ro["expect_status"]), "config-3 statuses differ from expectation"
    accepted = int((dq_win.cpu().numpy().astype(np.uint32) != 0xFFFFFFFF).sum())
    # K2 alone on the verified statuses (n_items = 0 skips K1): the tally's own HBM roofline
    k0e, k1e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    k2_reps = 20
    k0e.record(stream)
    for _ in range(k2_reps):
        eng.verify_tally_batch_dev(quorum, dq["off"], dq["idx"], dq["sig"], dq["dig"], M, 0, dq_st, dq_bits, d_ts=dq["ts"], d_value_id=dq["val"],
                                   d_winner=dq_win, stream=stream.cuda_stream)
    k1e.record(stream)
    stream.synchronize()
    k2_ms = k0e.elapsed_time(k1e) / k2_reps
    del dq, dq_st, dq_bits, dq_win
    eng.quorum_destroy(quorum)

    # ---- quorum-certified read ops END TO END: this rank's shard of BASELINE configs[4] --------------------------------
    # 1 048 576 read ops x 31 replicas sharded contiguously over 8 GPUs (shard.op_range) = 131 072 ops x 31 = 4 063 232
    # tuples per GPU (weak scaling: every rank runs one such shard at any N; N = 8 is the configuration itself).  The flat
    # tuples (key index, padded signature, digest, pre-status, t, value id) sit in page-locked host memory; one
    # bftq_verify_read_batch call per step moves them to the GPU in chunks, verifies (K1) and decides every operation as
    # Client.Read does (K2, arrival order), and brings statuses + decisions back.
    from bftkv_b200 import shard
    R5, M5_TOTAL = 31, 1048576
    lo5, hi5 = shard.op_range(M5_TOTAL, 8, rank % 8)
    M5 = hi5 - lo5
    pool5 = workload.make_verify_batch(args.pool5, n_keys=R5, seed=0xBF7C0010 + rank, corrupt_rate=0.0, unknown_rate=0.0, threads=cores_rank)
    eng5 = Engine(local_rank)                      # its own key table: replica r answers with key r
    eng5.bind_thread()
    eng5.register_rsa_keys([k["n"] for k in pool5["keys"]], [k["e"] for k in pool5["keys"]])
    ro5 = workload.make_read_ops(pool5, M5, R5, seed=0xBF7C0006 + rank, mix=workload.HARD_MIX, shuffle_arrival=True)
    qcs5 = [(10, 31, 11, 21, list(range(31)))]
    quorum5 = eng5.quorum_create(qcs5)             # n=31: f=10, READ threshold 11, suff 21
    NQ5 = M5 * R5
    pin5 = {k: eng5.host_copy(ro5[k]) for k in ("op_off", "key_idx", "sig", "digest", "pre_status", "ts", "value_id")}
    out5 = (eng5.host_alloc(NQ5, np.uint8), eng5.host_alloc(M5, np.uint8), eng5.host_alloc(M5, np.uint32), eng5.host_alloc(M5, np.uint32))
    h2d5 = sum(int(pin5[k].nbytes) for k in pin5)
    d2h5 = sum(int(a.nbytes) for a in out5)

    def q5step():
        eng5.verify_read_batch(quorum5, pin5["op_off"], pin5["key_idx"], pin5["sig"], pin5["digest"], pin5["ts"], pin5["value_id"],
                               pre_status=pin5["pre_status"], out_status=out5[0], out_decision=out5[1], out_winner=out5[2], out_decided_at=out5[3])
    q5step()
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        q5step()
    torch.cuda.synchronize(dev)
    q5_s = time.perf_counter() - t0
    barrier()
    assert np.array_equal(out5[0], ro5["expect_status"]), "config-5 statuses differ from expectation"
    dec_hist = {k: int((out5[1] == v).sum()) for k, v in (("value", 0), ("rejected", 1), ("exhausted", 2))}
    if rank == 0:                                  # decisions against the oracle (checker only, after the timed region)
        from oracle import c_oracle
        rd, rw, ra = c_oracle.read_decide_batch(qcs5, ro5["op_off"], ro5["key_idx"].astype(np.uint64), ro5["expect_status"], ro5["ts"], ro5["value_id"])
        assert np.array_equal(out5[1], rd) and np.array_equal(out5[2], rw) and np.array_equal(out5[3], ra), "config-5 decisions differ from the oracle"
    for a in list(pin5.values()) + list(out5):
        eng5.host_free(a)
    eng5.quorum_destroy(quorum5)
    eng5.close()
    del ro5, pool5

    # ---- quorum-certified read ops from RAW ANSWERS: packets in, decisions out ------------------------------------------------
    # BASELINE configs[2]'s shape (16-replica quorum) in the form Client.Read receives it: every answer is the decrypted
    # transport message (one-pass signature, partial-length literal data whose FileName carries the nonce, signature) around
    # the replica's stored packet <x, v, t, sig, ss> with an 11-signature collective signature — about 3.9 kB per answer.
    # One bftq_read_responses_batch call per step: H2D of the raw answers, K0m (parse, de-chunk, nonce check, packet.Parse,
    # SHA-256 of the body, hash-tag check), K1, K2m (values compared byte for byte, arrival-order decision), D2H.
    from bftkv_b200.crypto_gpu import read_responses_batch
    R6, M6 = 16, args.ops6
    ra = workload.make_read_answers(M6, R6, seed=0xBF7C0007 + rank, mix=workload.HARD_MIX)
    eng6 = Engine(local_rank)
    eng6.bind_thread()
    kr6 = Keyring(eng6)
    kr6.register(ra["keyring"])
    qcs6 = [(5, 16, 6, 11, ra["ids"])]
    blob6, off6 = _blob(ra["msgs"])
    pin6 = (eng6.host_copy(blob6), eng6.host_copy(off6))
    N6 = M6 * R6

    def q6step():
        return read_responses_batch(kr6, qcs6, ra["op_off"], ra["peer_ids"], None, ra["nonces"], pre_status=ra["pre_status"], blobs=pin6)
    q6step()
    s60 = eng6.stats()
    barrier()
    t0 = time.perf_counter()
    q6_each = []
    for _ in range(args.steps):
        t1 = time.perf_counter()
        got6 = q6step()
        q6_each.append((time.perf_counter() - t1) * 1e3)
    q6_s = time.perf_counter() - t0
    barrier()
    s61 = eng6.stats()
    assert np.array_equal(got6["status"] != 0, ra["expect_status"] != 0), "raw-answer statuses differ from expectation"
    if rank == 0:
        from oracle import c_oracle
        rd, rw, ra_ = c_oracle.read_decide_batch([(5, 16, 6, 11, list(range(16)))], ra["op_off"], ra["key_idx"].astype(np.uint64), ra["expect_status"],
                                                 ra["ts"], ra["value_id"])
        assert np.array_equal(got6["decision"], rd) and np.array_equal(got6["winner"], rw) and np.array_equal(got6["decided_at"], ra_), \
            "raw-answer decisions differ from the oracle"
    q6_info = {"bytes_per_answer": int(off6[-1]) // max(1, int((ra["pre_status"] == 0).sum())), "h2d_bytes_per_step": (s61["h2d_bytes"] - s60["h2d_bytes"]) // args.steps,
               "gpu_parsed": (s61["msg_gpu_items"] - s60["msg_gpu_items"]) // args.steps, "host_parsed": (s61["msg_host_items"] - s60["msg_host_items"]) // args.steps,
               "decisions": {k: int((got6["decision"] == v).sum()) for k, v in (("value", 0), ("rejected", 1), ("exhausted", 2))}}
    kr6.close()
    for a in pin6:
        eng6.host_free(a)
    eng6.close()
    del ra, blob6

    # ---- secondary: BASELINE configs[3] — 262144 Ed25519 verifies (K = 15 keys) + Lagrange combines ----
    # (the reference itself cannot verify Ed25519, SURVEY F5; reported for completeness of the configs)
    ed = None
    if rank == 0 and not args.skip_ed25519:
        from cryptography.hazmat.primitives import serialization
        from cryptography.hazmat.primitives.asymmetric.ed25519 import Ed25519PrivateKey
        from concurrent.futures import ThreadPoolExecutor
        import random as _r
        rg = _r.Random(0xBF7C0005)
        sks = [Ed25519PrivateKey.from_private_bytes(bytes(rg.randrange(256) for _ in range(32))) for _ in range(15)]
        pk_arr = np.frombuffer(b"".join(k.public_key().public_bytes(serialization.Encoding.Raw, serialization.PublicFormat.Raw) for k in sks),
                               np.uint8).reshape(15, 32).copy()
        NE = 262144
        e_idx = np.random.default_rng(5).integers(0, 15, NE).astype(np.uint32)
        e_msg = np.random.default_rng(6).integers(0, 256, (NE, 32), dtype=np.uint8)
        e_sig = np.empty((NE, 64), np.uint8)

        def sign_range(lo_hi):
            for i in range(*lo_hi):
                e_sig[i] = np.frombuffer(sks[e_idx[i]].sign(e_msg[i].tobytes()), np.uint8)
        nth = max(1, host_cores())
        with ThreadPoolExecutor(nth) as ex:
            list(ex.map(sign_range, [(lo, min(NE, lo + 4096)) for lo in range(0, NE, 4096)]))
        e_sig[::97, 7] ^= 1                                        # 1 % corrupted
        de = [torch.from_numpy(x).to(dev) for x in (pk_arr, e_idx.astype(np.int32), e_sig, e_msg)]
        de_st = torch.empty(NE, dtype=torch.uint8, device=dev)

        def estep():
            L_.check(eng._lib.bftq_ed25519_verify_batch_dev(eng._h, pk_arr.ctypes.data_as(C.c_void_p), 15, C.c_void_p(de[1].data_ptr()),
                                                            C.c_void_p(de[2].data_ptr()), C.c_void_p(de[3].data_ptr()), NE,
                                                            C.c_void_p(de_st.data_ptr()), C.c_void_p(stream.cuda_stream)))
        estep()
        stream.synchronize()
        a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a0.record(stream)
        for _ in range(args.steps):
            estep()
        a1.record(stream)
        stream.synchronize()
        e_ms = a0.elapsed_time(a1) / args.steps
        bad = int((de_st != 0).sum())
        assert bad == len(range(0, NE, 97)), "Ed25519 statuses differ from expectation"
        # Lagrange combine, 2t = 10 of n = 15 shares over the P-256 group order: host API incl. copies, and K3 alone
        from oracle import sss_oracle as sss_
        q256 = 0xFFFFFFFF00000000FFFFFFFFFFFFFFFFBCE6FAADA7179E84F3B9CAC2FC632551
        Bc, kc = NE // 15, 10
        rgen = np.random.default_rng(7)
        xs = np.stack([rgen.permutation(15)[:kc] + 1 for _ in range(Bc)]).astype(np.int32)
        ysb = rgen.integers(0, 256, (Bc, kc, 32), dtype=np.uint8)
        ysb[:, :, 0] &= 0x7F
        eng.lagrange_combine_batch(q256, xs[:64], ysb[:64])
        t0c = time.perf_counter()
        outc, stc = eng.lagrange_combine_batch(q256, xs, ysb)
        c_s = time.perf_counter() - t0c
        j = 12345 % Bc
        exp_j = sss_.calculate_secret([(int(xs[j, i]), int.from_bytes(ysb[j, i].tobytes(), "big")) for i in range(kc)], q256)
        assert int.from_bytes(outc[j].tobytes(), "big") == exp_j and not stc.any()
        dl = [torch.from_numpy(x).to(dev) for x in (xs, ysb)]
        dl_out, dl_st = torch.empty((Bc, 32), dtype=torch.uint8, device=dev), torch.empty(Bc, dtype=torch.uint8, device=dev)
        mb = np.frombuffer(q256.to_bytes(32, "big"), np.uint8).copy()

        def lstep():
            L_.check(eng._lib.bftq_lagrange_combine_batch_dev(eng._h, vp(mb), 32, kc, C.c_void_p(dl[0].data_ptr()), C.c_void_p(dl[1].data_ptr()), Bc,
                                                              C.c_void_p(dl_out.data_ptr()), C.c_void_p(dl_st.data_ptr()), C.c_void_p(stream.cuda_stream)))
        lstep()
        stream.synchronize()
        l0, l1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        l0.record(stream)
        for _ in range(10):
            lstep()
        l1.record(stream)
        stream.synchronize()
        k3_ms = l0.elapsed_time(l1) / 10
        assert np.array_equal(dl_out.cpu().numpy(), outc)
        ed = {"metric": "ed25519_verifies_per_sec", "value": NE / (e_ms * 1e-3), "unit": "verifies/s", "ms_per_step": e_ms,
              "config": {"workload": "262144 Ed25519 verifies over 15 keys, 32-byte messages (BASELINE configs[3]); 1% corrupted",
                         "note": "no reference behaviour exists: x/crypto/openpgp has no EdDSA (SURVEY F5); checked against OpenSSL and libsodium. "
                                 "Flat API only — there is no reference-facing path for this config (the reference skips EdDSA keys)"},
              "lagrange_combines_per_sec": Bc / c_s, "lagrange_config": "%d combines, 10 of 15 shares, P-256 order, host API incl. copies" % Bc,
              "k3_kernel_ms": k3_ms, "k3_items": Bc}
    clocks = sampler.stop() if rank == 0 else None

    t = torch.tensor([dev_ms, e2e_s * 1e3, q_ms, pgp_s * 1e3, sus_ms / n_sus, pgp_sus_s * 1e3 / n_e2e_sus, q5_s * 1e3, pgp_pageable_s * 1e3,
                      pgp_info["thread_ms"]["stage"], pgp_info["thread_ms"]["wait"], q6_s * 1e3, coll_s * 1e3], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    dev_ms, e2e_ms, q_ms, pgp_ms, sus_ms_step, pgp_sus_ms_step, q5_ms, pgp_pageable_ms, stage_ms_max, wait_ms_max, q6_ms, coll_ms = [float(x) for x in t]
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    total_items = ITEMS * world * args.steps
    value = total_items / (dev_ms * 1e-3)
    e2e_v = total_items / (e2e_ms * 1e-3)
    k_avg_ms = dev_ms / args.steps
    achieved = MACS_PER_VERIFY * ITEMS / (k_avg_ms * 1e-3)
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        hbm_peak, hbm_src = peaks["hbm_gbs"], "measured"
    except Exception:
        hbm_peak, hbm_src = 6650.0, "fallback"
    hbm_ach = BYTES_PER_VERIFY * ITEMS / (k_avg_ms * 1e-3) / 1e9
    k2_bytes = M * (3 * R + 1 + 4) + NQ * (8 + 4)     # SURVEY §8d unit (3R B in, 1 B out) + the read tally's t (8 B) and value id (4 B) per responder, winner 4 B
    out = {
        "metric": "rsa2048_signature_verifies_per_sec", "value": value, "unit": "verifies/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": dev_ms / args.steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "u32 limbs / u64 products (integer)", "data": "synthetic",
        "config": {"workload": WORKLOAD,
                   "per_gpu_batch": ITEMS, "l2": "inputs rotated over %d distinct device copies (%d MB > 126 MB L2)"
                   % (copies, copies * ITEMS * 292 // 2 ** 20), "lanes_per_signature": int(os.environ.get("BFTQ_RSA_T", "4")), "streams_in_flight": NSTREAMS,
                   "kernel": os.environ.get("BFTQ_RSA_KERNEL", "r32sq (default: radix 2^32, dedicated squaring, unified exponent loop, in-block barrier per product)"),
                   "numa_node": numa_node, "host_cores_per_rank": cores_rank},
        "gpu_launches": int(gpu_launches),
        "sustained": {"value": ITEMS * world / (sus_ms_step * 1e-3), "unit": "verifies/s", "launches": n_sus, "seconds": sus_ms * 1e-3,
                      "clocks": sampler.window(m0, m1), "note": "the `value` leg repeated for >= %.1f s; `value` itself is the K-step region the contract asks for" % args.sustain},
        "e2e": {"value": total_items / (pgp_ms * 1e-3), "unit": "verifies/s", "ms_per_step": pgp_ms / args.steps,
                "h2d_bytes_per_step": int(pgp_info["h2d"]), "d2h_bytes_per_step": int(pgp_info["d2h"]),
                "api": "bftq_signature_verify_batch = crypto.Signature.Verify's batch form (crypto_pgp.go:319-330): OpenPGP signature packets + "
                       "signed bytes in page-locked host blobs (bftq_host_alloc — the buffers the shim's aggregator fills) in, error codes out; "
                       "H2D of the raw packets, packet parsing + issuer lookup + digest + hash-tag check (K0 on the GPU, flagged items through the "
                       "host packer + K4), K1 verify and D2H inside the timed region; %d concurrent callers (one batch each per step)" % pgp_info["callers"],
                "sustained": {"value": ITEMS * world / (pgp_sus_ms_step * 1e-3), "steps": n_e2e_sus, "seconds": pgp_sus_s, "clocks": sampler.window(m2, m3)},
                "one_caller_ms_per_batch": pgp_info["single_ms"],
                "gpu_parse": os.environ.get("BFTQ_GPU_PARSE", "1") != "0",
                "host_packer_verifies_per_sec_rank0": pgp_info["host_packer_rate"],
                "kernels_per_step": int(pgp_info["launches"]), "host_threads": pgp_info["threads"], "chunks_per_step": int(pgp_info["chunks"]),
                "worker_thread_ms_per_step": pgp_info["thread_ms"], "stage_ms_per_step_max_over_ranks": stage_ms_max,
                "wait_ms_per_step_max_over_ranks": wait_ms_max, "cgroup_cpu_throttled_rank0": pgp_info["throttled"],
                "h2d_gbps_this_box": h2d_gbps, "copy_bound_verifies_per_sec": h2d_gbps * 1e9 / max(pgp_info["h2d"] / ITEMS, 1)},
        "e2e_pageable": {"value": total_items / (pgp_pageable_ms * 1e-3), "unit": "verifies/s", "ms_per_step": pgp_pageable_ms / args.steps,
                         "api": "the same call with the blobs in pageable memory: the library copies each chunk into its pinned staging first "
                                "(round 1's headline leg)", "worker_thread_ms_per_step": pgp_info["thread_ms_pageable"]},
        "e2e_flat": {"value": e2e_v, "unit": "verifies/s", "h2d_bytes_per_step": ITEMS * (256 + 32 + 4), "d2h_bytes_per_step": ITEMS,
                     "api": "bftq_rsa_verify_batch (flat tuples: key index, padded signature, precomputed digest; pinned host buffers), "
                            "%d concurrent callers" % NCALLERS,
                     "ms_per_step": e2e_ms / args.steps},
        "collective": {"metric": "collective_signature_verifies_per_sec", "value": NC * world * args.steps / (coll_ms * 1e-3), "unit": "collective verifies/s",
                       "signature_verifies_per_sec": NC * NSIG * world * args.steps / (coll_ms * 1e-3), "steps": args.steps, "ms_per_step": coll_ms / args.steps,
                       "api": "bftq_collective_verify_batch = crypto.CollectiveSignature.Verify's batch form (crypto_pgp.go:485-500): TBSS strings + concatenated "
                              "OpenPGP signature packets in page-locked host blobs in, nil / ErrInsufficientNumberOfSignatures out; packets framed on the host, "
                              "K0 + K1 + K2 (IsSufficient) on the GPU",
                       "config": {"workload": "%d collective signatures x 11 packets by members of a 16-node clique (f = 5, suff = 11), 2%% of the packets corrupted" % NC,
                                  "accepted_rank0": coll_accept, "data": "synthetic; packets drawn from 8 x 16 genuine signatures"}},
        "quorum_ops": {"metric": "quorum_certified_read_ops_per_sec", "value": M * world * args.steps / (q_ms * 1e-3), "unit": "ops/s",
                       "verifies_per_sec": NQ * world * args.steps / (q_ms * 1e-3), "steps": args.steps, "ms_per_step": q_ms / args.steps,
                       "config": {"workload": "batch 65536 read ops x 16-replica quorum, verify + wotqs read tally (BASELINE configs[2]), device-resident",
                                  "quorum": "n=16 f=5 READ threshold 6", "accepted_ops_rank0": accepted,
                                  "data": "synthetic; 1,048,576 tuples drawn from a pool of 65,536 genuine signatures"},
                       "kernels_per_step": 2,
                       "e2e": {"metric": "quorum_certified_read_ops_per_sec", "value": M5 * world * args.steps / (q5_ms * 1e-3), "unit": "ops/s",
                               "verifies_per_sec": NQ5 * world * args.steps / (q5_ms * 1e-3), "steps": args.steps, "ms_per_step": q5_ms / args.steps,
                               "h2d_bytes_per_step": h2d5, "d2h_bytes_per_step": d2h5,
                               "api": "bftq_verify_read_batch: flat tuples in page-locked host memory in, per-tuple status + per-op Client.Read decision "
                                      "(value / rejected / exhausted, winner, decided_at) out; chunked H2D + K1 + K2 + D2H inside the timed region",
                               "config": {"workload": "BASELINE configs[4]: 1M (1,048,576) read ops x 31-replica Byzantine quorum sharded across 8 GPUs by contiguous "
                                                      "op ranges (shard.op_range) = %d ops x 31 = %d verifies per GPU; every rank runs one such shard (weak scaling; "
                                                      "N = 8 is the configuration itself)" % (M5, NQ5),
                                          "quorum": "n=31 f=10 READ threshold 11",
                                          "responses": "per-op mix: 80% as SURVEY config 3 (0.90 ok / 0.05 stale / 0.03 bad / 0.02 missing), 20% degraded classes "
                                                       "(workload.HARD_MIX); responses arrive in seeded random order",
                                          "decisions_rank0": dec_hist, "checked": "statuses vs expectation on every rank; decisions vs the C oracle on rank 0",
                                          "data": "synthetic; tuples drawn from a pool of %d genuine signatures over 31 keys" % args.pool5}},
                       "e2e_packets": {"metric": "quorum_certified_read_ops_per_sec", "value": M6 * world * args.steps / (q6_ms * 1e-3), "unit": "ops/s",
                                       "answers_per_sec": N6 * world * args.steps / (q6_ms * 1e-3), "steps": args.steps, "ms_per_step": q6_ms / args.steps, "ms_each_step_rank0": [round(x, 3) for x in q6_each],
                                       "h2d_bytes_per_step": int(q6_info["h2d_bytes_per_step"]), "bytes_per_answer": q6_info["bytes_per_answer"],
                                       "h2d_gbps_achieved": q6_info["h2d_bytes_per_step"] * args.steps / (q6_ms * 1e-3) / 1e9,
                                       "api": "bftq_read_responses_batch: the decrypted transport answers (one-pass signature, partial-length literal data, signature) in "
                                              "page-locked host memory in, per-answer status + per-op Client.Read decision out; message parsing, de-chunking, nonce check, "
                                              "packet.Parse, SHA-256, RSA verify and the tally all on the GPU",
                                       "config": {"workload": "%d read ops x 16-replica quorum per GPU, every answer a ~3.9 kB transport message around the stored packet "
                                                              "<x, v, t, sig, ss(11 signatures)>; response mix workload.HARD_MIX, random arrival order" % M6,
                                                  "answers_parsed_on_gpu_rank0": int(q6_info["gpu_parsed"]), "answers_through_host_packer_rank0": int(q6_info["host_parsed"]),
                                                  "decisions_rank0": q6_info["decisions"], "checked": "statuses vs expectation on every rank; decisions vs the C oracle on rank 0",
                                                  "data": "synthetic; one signed template per (replica, current / stale value), the nonce in the unsigned FileName differs per answer"}}},
        "roofline": {"bound": "int_alu", "achieved": achieved / 1e12, "peak": int_peak / 1e12, "unit": "Tmac/s (32x32+64 IMAD.WIDE on the FMA-heavy pipe)",
                     "frac": achieved / int_peak, "traffic": NCU_DRAM_BYTES_PER_LAUNCH,
                     "traffic_source": "dram__bytes_read.sum + dram__bytes_write.sum of one rsa_verify_r32_kernel launch (65536 items) in "
                                       "profiles/ncu_rsa_verify_r02c_unified.txt (ncu --set full); algorithmic bytes per launch = %d" % (BYTES_PER_VERIFY * ITEMS),
                     "peak_source": "measured live on this GPU: dependency-free fused IMAD.WIDE.U32 stream, 64 warps/SM (bftq_measure_int_peak)",
                     "kernel": "rsa_verify_r32_kernel<128, 4, SQ>", "kernel_ms_avg": k_avg_ms, "kernel_ms_alone": serial_ms[len(serial_ms) // 2],
                     "kernel_ms_note": "avg = timed region / launches (launches alternate over %d streams); alone = median of the serial warm-up launches" % NSTREAMS,
                     "algorithmic_macs_per_verify": MACS_PER_VERIFY, "executed_macs_per_verify": EXECUTED_MACS_PER_VERIFY,
                     "frac_executed": EXECUTED_MACS_PER_VERIFY * ITEMS / (k_avg_ms * 1e-3) / int_peak,
                     "note": "`frac` uses SURVEY §8(d)'s ALGORITHMIC count (19 schoolbook products); the kernel executes fewer multiplies (18 products, "
                             "16 of them triangular squarings), so frac can exceed the share of pipe cycles it occupies — `frac_executed` is that share",
                     "hbm": {"achieved": hbm_ach, "peak": hbm_peak, "unit": "GB/s", "frac": hbm_ach / hbm_peak,
                             "peak_source": hbm_src + " (MEASURED_PEAKS.json)", "algorithmic_bytes_per_verify": BYTES_PER_VERIFY}},
        "roofline_secondary": {
            "k2_read_tally": {"bound": "hbm", "achieved": k2_bytes / (k2_ms * 1e-3) / 1e9, "peak": hbm_peak, "unit": "GB/s",
                              "frac": k2_bytes / (k2_ms * 1e-3) / 1e9 / hbm_peak, "kernel_ms": k2_ms,
                              "bytes_per_launch": k2_bytes, "note": "read_tally_kernel alone on 65536 ops x 16 responders (17 B per responder + 5 B per op); "
                                                                     "1.1 MB of inputs stay L2-resident between launches, so this is launch/latency bound, not HBM bound"}},
        "clocks": clocks,
        "ed25519": ed,
    }
    if ed:
        out["roofline_secondary"]["k1b_ed25519"] = {
            "bound": "int_alu", "achieved": ED25519_MACS * ed["value"] / 1e12, "peak": int_peak / 1e12, "unit": "Tmac/s",
            "frac": ED25519_MACS * ed["value"] / int_peak, "executed_macs_per_verify": ED25519_MACS,
            "note": "cached window tables (radix 2^12 base point, radix 2^10 keys): expected 47.4 mixed additions x 7 field products x 100 IMAD.WIDE + Barrett reduction (126) in "
                    "ed25519_accumulate_kernel, 5 products + 1/8 inversion per signature in ed25519_finish_kernel; SHA-512 and the 19*g / 2*f "
                    "pre-scalings (plain IMAD) not counted; the first K1b executed 134 970 per verification"}
        k3_bytes = ed["k3_items"] * (10 * (4 + 32) + 32 + 1)
        out["roofline_secondary"]["k3_lagrange"] = {
            "bound": "hbm", "achieved": k3_bytes / (ed["k3_kernel_ms"] * 1e-3) / 1e9, "peak": hbm_peak, "unit": "GB/s",
            "frac": k3_bytes / (ed["k3_kernel_ms"] * 1e-3) / 1e9 / hbm_peak, "kernel_ms": ed["k3_kernel_ms"], "bytes_per_launch": k3_bytes,
            "note": "lagrange_combine_kernel<8> on %d combines of 10 shares mod the P-256 order: 393 B per combine (SURVEY §8d); one thread per "
                    "combine (small-integer inversions + about 80 Montgomery products), under one wave: latency-bound, HBM idle" % ed["k3_items"]}
    if world == 1:
        from oracle import c_oracle
        threads = host_cores()
        reps = 4
        have_lc = c_oracle.libcrypto_available()
        if have_lc:
            lc_rate, st = cpu_verify(w, threads, reps, "libcrypto")
            assert (st == w["expect"]).all()
        port_rate, st = cpu_verify(w, threads, reps, "port")
        assert (st == w["expect"]).all()
        kind = "libcrypto" if have_lc else "port"
        out["cpu_baseline"] = {"value": lc_rate if have_lc else port_rate, "unit": "verifies/s", "cores": threads, "kind": "port",
                               "implementation": kind,
                               "sample": "%d passes over the same 65536-item batch (%d verifies) on %d host threads; %s"
                               % (reps, reps * ITEMS, threads, CPU_KIND_TEXT[kind])}
        out["cpu_baseline_port"] = {"value": port_rate, "unit": "verifies/s", "cores": threads, "kind": "port", "implementation": "port",
                                    "sample": "%d passes over the same batch; %s" % (reps, CPU_KIND_TEXT["port"])}
    real_stdout.write(json.dumps(out) + "\n")
    real_stdout.flush()
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--copies", type=int, default=8)
    ap.add_argument("--streams", type=int, default=2, help="streams the device-resident launches alternate over")
    ap.add_argument("--callers", type=int, default=2, help="concurrent host callers in the flat end-to-end leg")
    ap.add_argument("--pgp-callers", type=int, default=2, help="concurrent host callers in the packet-level end-to-end leg")
    ap.add_argument("--sustain", type=float, default=2.2, help="seconds of the sustained legs")
    ap.add_argument("--pool5", type=int, default=32768, help="genuine signatures in the configs[4] pool")
    ap.add_argument("--ops6", type=int, default=8192, help="read operations per GPU in the raw-answer leg")
    ap.add_argument("--coll-items", type=int, default=16384, help="collective signatures per step in the server-side leg")
    ap.add_argument("--skip-ed25519", action="store_true", help="skip the BASELINE configs[3] secondary measurement")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's status bytes to DIR/status.npy (float32)")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank, world)
    else:
        run_gpu(args, rank, local_rank, world)


if __name__ == "__main__":
    main()
