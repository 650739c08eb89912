#!/usr/bin/env python3
"""A/B of every host-buffer entry point of two builds of libzkpair.so on the same seeded inputs.

Each library runs in a fresh process with ZKPAIR_LIB pointing at it.  The first library also generates the inputs
(points, field elements, Groth16 and KZG workloads, blobs, cells) into a temporary directory, so that both see the
same bytes.  Every call runs once from pageable (numpy) and once from pinned (torch) host buffers, with outputs
pre-filled with 0xA5.  Compared per call: the output bytes, the return code, zkp_last_error() and the growth of
zkp_launch_count().  Sizes straddle one and two chunk boundaries of a build with
-DZKP_CHUNK=1024 -DZKP_BLOB_CHUNK=8 -DZKP_CELLS_CHUNK=4 -DZKP_CELL_PROOF_CHUNK=2 -DZKP_CELLS_RECOVER_CHUNK=4
-DZKP_CELL_VERIFY_CHUNK=64; inputs include n = 0, n = 1 and invalid elements (off-curve points, limbs >= p, scalars
>= r, bad cell indices and counts).  Prints one line per call and exits non-zero on any difference.
Usage: python tools/ab_host_calls.py LIB_A LIB_B [--devices N]   (N devices per context; default 1)"""
import ctypes
import hashlib
import json
import os
import subprocess
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

NP = 6400          # points in the pool: 2049 checks of 3 pairs
N_PAIR = [0, 1, 1025, 2049]
N_BLOB = [0, 1, 9, 17]
N_CELLS = [0, 1, 5, 9]
N_CELL_PROOF = [0, 1, 3, 5]
N_VERIFY = [0, 1, 65, 129, 256]


def fr_rows(rng, n):   # n scalars < r as (n, 4) little-endian u64
    v = rng.integers(0, 2**64, size=(n, 4), dtype=np.uint64)
    v[:, 3] &= np.uint64(0x3FFFFFFFFFFFFFFF)
    return v


def gen(d):
    import zkvm_pairings_b200 as z
    from zkvm_pairings_b200 import workloads as w
    rng = np.random.default_rng(0xAB)
    eng = z.PairingEngine([0])
    g1, i1, g2, i2 = eng.gen_points(0x5EED, 0, NP)
    i1[::97] = 1
    i2[::89] = 1
    fp = np.concatenate([g1.reshape(-1), g2.reshape(-1)]).reshape(-1, 6)   # canonical Fp
    out = {"g1": g1, "i1": i1, "g2": g2, "i2": i2, "fp": fp, "fr": fr_rows(rng, NP)}
    g16 = w.groth16_proofs(eng, 2049, 3, seed=0x16)
    for k in ("alpha", "beta", "gamma", "delta", "ic", "proofs", "inputs"):
        out["g16_" + k] = g16[k]
    g16b = w.groth16_proofs(eng, 1025, 20, seed=0x17)
    for k in ("alpha", "beta", "gamma", "delta", "ic", "proofs", "inputs"):
        out["g16b_" + k] = g16b[k]
    kz = w.kzg_proofs(eng, 2049)
    out.update(kzg_tau=kz["tau_g2"], kzg_proofs=kz["proofs"], kzg_zy=kz["zy"])
    bl = w.kzg_blob_proofs(eng, 17, distinct=4)
    out.update(blob_tau=bl["tau_g2"], blobs=bl["blobs"], blob_proofs=bl["proofs"])
    _, g2m, g1m, lag = w.kzg_cell_setup(eng)
    out.update(g2m=g2m, g1m=g1m, lag=lag)
    with eng.kzg_setup_cells(g2m, g1m, lag) as s:
        cells, pr, pi, _ = eng.kzg_compute_cells_and_proofs_batch(s, bl["blobs"][:2])
        com, _, _ = eng.kzg_blob_to_commitment_batch(s, bl["blobs"][:2])
        cells9 = eng.kzg_compute_cells_batch(s, bl["blobs"][:9])[0]
    out.update(vc_cells=cells.reshape(256, -1), vc_proofs=pr.reshape(256, 12), vc_com=np.repeat(com, 128, axis=0),
               vc_idx=np.tile(np.arange(128, dtype=np.uint64), 2))
    idx = np.zeros((9, 128), np.uint64)
    rc = np.zeros((9, 128, cells9.shape[-1]), np.uint8)
    num = np.zeros(9, np.uint64)
    for b in range(9):   # 64 .. 128 cells present, the first num entries in ascending order
        m = int(rng.integers(64, 129))
        keep = np.sort(rng.choice(128, size=m, replace=False))
        idx[b, :m], rc[b, :m], num[b] = keep, cells9[b, keep], m
    out.update(rec_idx=idx, rec_cells=rc, rec_num=num)
    eng.close()
    np.savez(os.path.join(d, "inputs.npz"), **out)


def run(d, ndev):
    import torch
    import zkvm_pairings_b200 as z
    from zkvm_pairings_b200 import engine as E
    I = dict(np.load(os.path.join(d, "inputs.npz")))
    eng = z.PairingEngine(list(range(ndev)))
    lib, ctx = eng._lib, eng._ctx
    g1, i1, g2, i2, fp, fr = I["g1"], I["i1"], I["g2"], I["i2"], I["fp"], I["fr"]

    def fpn(k, off=0):   # k canonical Fp as (k, 6)
        return np.resize(np.roll(fp, -off, axis=0), (k, 6))

    bad_g1 = g1.copy()
    bad_g1[7, 1] ^= np.uint64(1)            # off the curve
    nc_g1 = g1.copy()
    nc_g1[1030, :6] = np.uint64(2**64 - 1)   # x >= p
    bad_fr = fr.copy()
    bad_fr[3] = np.uint64(2**64 - 1)        # >= r
    vk = eng.groth16_prepare_vk(*(I["g16_" + k] for k in ("alpha", "beta", "gamma", "delta", "ic")))
    vkb = eng.groth16_prepare_vk(*(I["g16b_" + k] for k in ("alpha", "beta", "gamma", "delta", "ic")))
    ks = eng.kzg_setup(I["kzg_tau"])
    bs = eng.kzg_setup(I["blob_tau"])
    cs = eng.kzg_setup_cells(I["g2m"], I["g1m"], I["lag"])
    blobs = I["blobs"]
    bad_blobs = blobs.copy()
    bad_blobs[5, :32] = 0xFF                # an element >= r
    tables = eng.g2_prepare_batch(g2[:3])
    tinf = np.array([0, 1, 0], np.uint8)

    cases = []   # (name, symbol, args): "ctx", ("h", handle), ("v", ctype value), ("i", array | None), ("o", shape, dtype)

    def add(name, sym, *args):
        cases.append((name, sym, args))

    O8, O64 = np.uint8, np.uint64
    for op, (na, nb, nr) in (("fp_mul", (1, 1, 1)), ("fp2_inv", (2, 0, 2)), ("fp_sqrt", (1, 0, 1)), ("fp12_mul", (12, 12, 12)),
                             ("fp12_pow", (12, 1, 12)), ("fp12_mul_by_014", (12, 6, 12)), ("fp6_mul_by_01", (6, 4, 6))):
        for n in N_PAIR:
            a, b = fpn(n * na).reshape(n, 6 * na), (fpn(n * nb, 5).reshape(n, 6 * nb) if nb else None)
            add("tower %s n=%d" % (op, n), "zkp_tower_op_batch", "ctx", ("v", ctypes.c_int32(E.TOWER_OPS[op])), ("i", a), ("i", b),
                ("o", (n, 6 * nr), O64), ("o", (n,), O8), ("v", ctypes.c_size_t(n)))
    nca = fpn(1025).copy()
    nca[1024] = np.uint64(2**64 - 1)
    add("tower fp_mul non-canonical", "zkp_tower_op_batch", "ctx", ("v", ctypes.c_int32(3)), ("i", nca), ("i", fpn(1025, 1)),
        ("o", (1025, 6), O64), ("o", (1025,), O8), ("v", ctypes.c_size_t(1025)))
    for n in N_PAIR:
        add("fp_mul n=%d" % n, "zkp_fp_mul_batch", "ctx", ("i", fpn(n)), ("i", fpn(n, 3)), ("o", (n, 6), O64), ("v", ctypes.c_size_t(n)))
        add("fp12_mul n=%d" % n, "zkp_fp12_mul_batch", "ctx", ("i", fpn(12 * n)), ("i", fpn(12 * n, 3)), ("o", (n, 72), O64),
            ("v", ctypes.c_size_t(n)))
        add("mul_by_014 n=%d" % n, "zkp_fp12_mul_by_014_batch", "ctx", ("i", fpn(12 * n)), ("i", fpn(6 * n, 3)), ("o", (n, 72), O64),
            ("v", ctypes.c_size_t(n)))
    for op in (0, 1):
        add("sys_bigint op=%d" % op, "zkp_sys_bigint", "ctx", ("o", (12,), np.uint32), ("v", ctypes.c_uint32(op)),
            ("i", fpn(1).view(np.uint32).reshape(-1)), ("i", fpn(1, 9).view(np.uint32).reshape(-1)))
    for sym, mode in (("zkp_miller_loop_batch", "miller"), ("zkp_pairing_batch", "pairing")):
        for n in N_PAIR:
            for fl in (0, 1):
                add("%s n=%d flags=%d" % (mode, n, fl), sym, "ctx", ("i", g1[:n]), ("i", i1[:n] if fl else None), ("i", g2[:n]),
                    ("i", i2[:n] if fl else None), ("v", ctypes.c_size_t(n)), ("o", (n, 72), O64))
    add("pairing non-canonical", "zkp_pairing_batch", "ctx", ("i", nc_g1[:2049]), ("i", None), ("i", g2[:2049]), ("i", None),
        ("v", ctypes.c_size_t(2049)), ("o", (2049, 72), O64))
    for n in N_PAIR:
        for fl in (0, 1):
            a1, a2 = (i1[:3 * n], i2[:3 * n]) if fl else (None, None)
            add("multi_miller k=3 n=%d flags=%d" % (n, fl), "zkp_multi_miller_loop_batch", "ctx", ("i", g1[:3 * n]), ("i", a1),
                ("i", g2[:3 * n]), ("i", a2), ("v", ctypes.c_size_t(n)), ("v", ctypes.c_int32(3)), ("o", (n, 72), O64))
            add("multi_pairing k=3 n=%d flags=%d" % (n, fl), "zkp_multi_pairing_batch", "ctx", ("i", g1[:3 * n]), ("i", a1),
                ("i", g2[:3 * n]), ("i", a2), ("v", ctypes.c_size_t(n)), ("v", ctypes.c_int32(3)), ("o", (n, 72), O64), ("o", (n,), O8))
    add("multi_pairing k=9", "zkp_multi_pairing_batch", "ctx", ("i", g1[:9]), ("i", None), ("i", g2[:9]), ("i", None),
        ("v", ctypes.c_size_t(1)), ("v", ctypes.c_int32(9)), ("o", (1, 72), O64), ("o", (1,), O8))
    for n in N_PAIR:
        add("final_exp n=%d" % n, "zkp_final_exp_batch", "ctx", ("i", fpn(12 * n, 2)), ("v", ctypes.c_size_t(n)), ("o", (n, 72), O64))
        add("gen_points n=%d" % n, "zkp_gen_points", "ctx", ("v", ctypes.c_uint64(77)), ("v", ctypes.c_uint64(5)), ("v", ctypes.c_size_t(n)),
            ("o", (n, 12), O64), ("o", (n,), O8), ("o", (n, 24), O64), ("o", (n,), O8))
    ncf = fpn(12 * 1025, 2).copy()
    ncf[12 * 1024 + 3] = np.uint64(2**64 - 1)
    add("final_exp non-canonical", "zkp_final_exp_batch", "ctx", ("i", ncf), ("v", ctypes.c_size_t(1025)), ("o", (1025, 72), O64))
    for kf in (0, 1, 3):
        for ti in (0, 1):
            if ti and not kf:
                continue
            for n in (1, 1025, 2049):
                kv = 3 - kf
                add("prepared k=3 kf=%d tables_inf=%d n=%d" % (kf, ti, n), "zkp_multi_pairing_prepared_batch", "ctx", ("i", g1[:3 * n]),
                    ("i", i1[:3 * n]), ("i", g2[:kv * n] if kv else None), ("i", i2[:kv * n] if kv else None), ("v", ctypes.c_size_t(n)),
                    ("v", ctypes.c_int32(3)), ("i", tables[:kf] if kf else None), ("i", tinf[:kf] if ti else None), ("v", ctypes.c_int32(kf)),
                    ("o", (n, 72), O64), ("o", (n,), O8))
    for n in (0, 1, 2049, 6147):
        for mp in (1, 0):
            for fl in (0, 1):
                add("multi_miller_product n=%d miller=%d flags=%d" % (n, mp, fl), "zkp_multi_miller_product", "ctx", ("i", g1[:n]),
                    ("i", i1[:n] if fl else None), ("i", g2[:n]), ("i", i2[:n] if fl else None), ("v", ctypes.c_size_t(n)),
                    ("o", (72,), O64) if mp else ("i", None), ("o", (72,), O64))
    for n in N_PAIR:
        for G, w, src, ssrc in (("g1", 12, g1, bad_g1), ("g2", 24, g2, g2)):
            add("%s_add n=%d" % (G, n), "zkp_%s_add_batch" % G, "ctx", ("i", src[:n]), ("i", i1[:n]), ("i", src[7:7 + n]), ("i", i2[:n]),
                ("v", ctypes.c_size_t(n)), ("o", (n, w), O64), ("o", (n,), O8))
            add("%s_add noflags n=%d" % (G, n), "zkp_%s_add_batch" % G, "ctx", ("i", src[:n]), ("i", None), ("i", src[7:7 + n]), ("i", None),
                ("v", ctypes.c_size_t(n)), ("o", (n, w), O64), ("o", (n,), O8))
            add("%s_check n=%d" % (G, n), "zkp_%s_check_batch" % G, "ctx", ("i", ssrc[:n]), ("i", i1[:n]), ("v", ctypes.c_size_t(n)),
                ("o", (n,), O8))
            add("%s_mul n=%d" % (G, n), "zkp_%s_mul_batch" % G, "ctx", ("i", ssrc[:n]), ("i", i2[:n]), ("i", fr[:n]), ("v", ctypes.c_size_t(n)),
                ("o", (n, w), O64), ("o", (n,), O8))
    add("g1_check non-canonical", "zkp_g1_check_batch", "ctx", ("i", nc_g1[:2049]), ("i", None), ("v", ctypes.c_size_t(2049)), ("o", (2049,), O8))
    for tag, h, P in (("np3", vk, "g16_"), ("np20", vkb, "g16b_")):
        pf, xs = I[P + "proofs"], I[P + "inputs"]
        bad_x = xs.copy()
        bad_x[2, :4] = np.uint64(2**64 - 1)
        pinf = np.zeros((len(pf), 3), np.uint8)
        pinf[4::50, 1] = 1
        for n in [m for m in N_PAIR if m <= len(pf)]:
            for fl in (0, 1):
                add("groth16 %s n=%d flags=%d" % (tag, n, fl), "zkp_groth16_verify_batch", "ctx", ("h", h), ("i", pf[:n]),
                    ("i", pinf[:n] if fl else None), ("i", (bad_x if fl else xs)[:n]), ("v", ctypes.c_size_t(n)), ("o", (n,), O8))
    kp, kzy = I["kzg_proofs"], I["kzg_zy"]
    bad_zy = kzy.copy()
    bad_zy[9, :4] = np.uint64(2**64 - 1)
    kinf = np.zeros((len(kp), 2), np.uint8)
    kinf[3::40, 0] = 1
    for n in N_PAIR:
        for fl in (0, 1):
            add("kzg_verify n=%d flags=%d" % (n, fl), "zkp_kzg_verify_batch", "ctx", ("h", ks), ("i", kp[:n]), ("i", kinf[:n] if fl else None),
                ("i", (bad_zy if fl else kzy)[:n]), ("v", ctypes.c_size_t(n)), ("o", (n,), O8))
    bp = I["blob_proofs"]
    binf = np.zeros((17, 2), np.uint8)
    binf[2, 1] = 1
    for n in N_BLOB:
        for fl in (0, 1):
            for zy in (0, 1):
                add("blob_verify n=%d flags=%d zy=%d" % (n, fl, zy), "zkp_kzg_verify_blob_batch", "ctx", ("h", bs),
                    ("i", (bad_blobs if fl else blobs)[:n]), ("i", bp[:n]), ("i", binf[:n] if fl else None), ("v", ctypes.c_size_t(n)),
                    ("o", (n,), O8), ("o", (n, 8), O64) if zy else ("i", None))
    cinf = np.zeros(17, np.uint8)
    cinf[4] = 1
    for n in N_BLOB:
        src = bad_blobs[:n]
        add("commitment n=%d" % n, "zkp_kzg_blob_to_commitment_batch", "ctx", ("h", cs), ("i", src), ("v", ctypes.c_size_t(n)),
            ("o", (n, 12), O64), ("o", (n,), O8), ("o", (n,), O8))
        zz = bad_fr[:n].copy()
        add("compute_proof n=%d" % n, "zkp_kzg_compute_proof_batch", "ctx", ("h", cs), ("i", src), ("i", zz), ("v", ctypes.c_size_t(n)),
            ("o", (n, 12), O64), ("o", (n,), O8), ("o", (n, 4), O64), ("o", (n,), O8))
        for fl in (0, 1):
            for zy in (0, 1):
                add("blob_proof n=%d flags=%d zy=%d" % (n, fl, zy), "zkp_kzg_compute_blob_proof_batch", "ctx", ("h", cs), ("i", src),
                    ("i", bp[:n, :12]), ("i", cinf[:n] if fl else None), ("v", ctypes.c_size_t(n)), ("o", (n, 12), O64), ("o", (n,), O8),
                    ("o", (n,), O8), ("o", (n, 8), O64) if zy else ("i", None))
    CB = 128 * 2048
    for n in N_CELLS:
        add("cells n=%d" % n, "zkp_kzg_compute_cells_batch", "ctx", ("h", cs), ("i", bad_blobs[:n]), ("v", ctypes.c_size_t(n)),
            ("o", (n, CB), O8), ("o", (n,), O8))
    for n in N_CELL_PROOF:
        add("cells_and_proofs n=%d" % n, "zkp_kzg_compute_cells_and_proofs_batch", "ctx", ("h", cs), ("i", bad_blobs[:n]),
            ("v", ctypes.c_size_t(n)), ("o", (n, CB), O8), ("o", (n, 128, 12), O64), ("o", (n, 128), O8), ("o", (n,), O8))
    vcc, vci, vcp, vcm = I["vc_com"], I["vc_idx"].copy(), I["vc_proofs"], I["vc_cells"].copy()
    vci[70] = 128                 # an index >= 128
    vci[71] = 2**64 - 1
    vcm[100, :32] = 0xFF          # an element >= r
    vflag = np.zeros(256, np.uint8)
    vflag[5::60] = 1
    for n in N_VERIFY:
        for fl in (0, 1):
            add("verify_cell n=%d flags=%d" % (n, fl), "zkp_kzg_verify_cell_batch", "ctx", ("h", cs), ("i", vcc[:n]), ("i", vflag[:n] if fl else None),
                ("i", vci[:n]), ("i", vcm[:n]), ("i", vcp[:n]), ("i", vflag[:n] if fl else None), ("v", ctypes.c_size_t(n)), ("o", (n,), O8))
    ridx, rcl, rnum = I["rec_idx"], I["rec_cells"], I["rec_num"]
    bidx, bnum = ridx.copy(), rnum.copy()
    bnum[1] = 63                  # too few cells
    bidx[2, :2] = bidx[2, 1::-1]  # not ascending
    bidx[3, 0] = 200              # out of range
    for bad in (0, 1):
        xi, xn = (bidx, bnum) if bad else (ridx, rnum)
        for n in (0, 1, 5, 9):
            add("recover n=%d bad=%d" % (n, bad), "zkp_kzg_recover_cells_batch", "ctx", ("h", cs), ("i", xi[:n]), ("i", rcl[:n]), ("i", xn[:n]),
                ("v", ctypes.c_size_t(n)), ("o", (n, CB), O8), ("o", (n,), O8))
        for n in (0, 1, 3, 5):
            add("recover_and_proofs n=%d bad=%d" % (n, bad), "zkp_kzg_recover_cells_and_proofs_batch", "ctx", ("h", cs), ("i", xi[:n]),
                ("i", rcl[:n]), ("i", xn[:n]), ("v", ctypes.c_size_t(n)), ("o", (n, CB), O8), ("o", (n, 128, 12), O64), ("o", (n, 128), O8),
                ("o", (n,), O8))

    def pinned_like(shape, dtype):
        nb = int(np.prod(shape)) * np.dtype(dtype).itemsize
        return torch.empty(max(nb, 1), dtype=torch.uint8, pin_memory=True).numpy()[:nb].view(dtype).reshape(shape)

    res = {}
    for name, sym, args in cases:
        for mem in ("pageable", "pinned"):
            cargs, outs, keep = [], [], []
            for a in args:
                if a == "ctx":
                    cargs.append(ctx)
                elif a[0] == "h":
                    cargs.append(a[1].handle)
                elif a[0] == "v":
                    cargs.append(a[1])
                elif a[1] is None:
                    cargs.append(None)
                elif a[0] == "i":
                    x = np.ascontiguousarray(a[1])
                    if mem == "pinned":
                        x, p = pinned_like(x.shape, x.dtype), x
                        x[...] = p
                    keep.append(x)
                    cargs.append(ctypes.c_void_p(x.ctypes.data))
                else:
                    o = np.empty(a[1], a[2]) if mem == "pageable" else pinned_like(a[1], a[2])
                    o.view(np.uint8)[...] = 0xA5
                    outs.append(o)
                    cargs.append(ctypes.c_void_p(o.ctypes.data))
            l0 = lib.zkp_launch_count(ctx)
            rc = getattr(lib, sym)(*cargs)
            dl = lib.zkp_launch_count(ctx) - l0
            err = lib.zkp_last_error().decode() if rc else ""
            h = hashlib.sha256()
            for o in outs:
                h.update(o.tobytes())
            res["%s [%s]" % (name, mem)] = [rc, err, dl, h.hexdigest()[:16]]
    for o in (vk, vkb, ks, bs, cs):
        o.close()
    eng.close()
    print(json.dumps(res))


def main():
    if sys.argv[1] == "--gen":
        gen(sys.argv[2])
        return
    if sys.argv[1] == "--run":
        run(sys.argv[2], int(sys.argv[3]))
        return
    libs = [os.path.abspath(p) for p in sys.argv[1:3]]
    ndev = int(sys.argv[sys.argv.index("--devices") + 1]) if "--devices" in sys.argv else 1
    me = os.path.abspath(__file__)
    with tempfile.TemporaryDirectory() as d:
        env = dict(os.environ, ZKPAIR_LIB=libs[0])
        subprocess.run([sys.executable, me, "--gen", d], env=env, check=True)
        res = []
        for lib in libs:
            r = subprocess.run([sys.executable, me, "--run", d, str(ndev)], env=dict(os.environ, ZKPAIR_LIB=lib), capture_output=True, text=True)
            if r.returncode != 0:
                print("run with %s failed:\n%s" % (lib, r.stderr[-3000:]))
                sys.exit(2)
            res.append(json.loads(r.stdout.strip().splitlines()[-1]))
    a, b = res
    bad = 0
    for k in sorted(set(a) | set(b)):
        same = a.get(k) == b.get(k)
        bad += not same
        rc, err, dl, h = a.get(k) or [None] * 4
        line = "%s %s  rc=%s launches=%s out=%s" % ("same" if same else "DIFF", k, rc, dl, h)
        if err:
            line += "  err=%r" % err
        if not same:
            line += "  vs  %s" % (b.get(k),)
        print(line)
    print("%d calls, %d differences (devices per context: %d)" % (len(set(a) | set(b)), bad, ndev))
    sys.exit(1 if bad else 0)


if __name__ == "__main__":
    main()
