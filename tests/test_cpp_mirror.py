"""The C++ host mirror (include/nova_b200.hpp): compiles and links against the C ABI on the CPU
box; on the GPU box runs commits concurrently from 8 threads and checks every result against the
oracle."""
import os
import struct
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EXE = os.path.join(ROOT, "tests", "cpp", "host_mirror_test")


def build():
    src = os.path.join(ROOT, "tests", "cpp", "host_mirror_test.cpp")
    hdrs = [os.path.join(ROOT, "include", f) for f in ("nova_b200.hpp", "nova_b200.h")]
    lib = os.path.join(ROOT, "nova_b200", "libnova_b200.so")
    if not os.path.exists(EXE) or any(os.path.getmtime(p) > os.path.getmtime(EXE) for p in [src, lib] + hdrs):
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-pthread", src, "-o", EXE, "-L" + os.path.dirname(lib),
                               "-lnova_b200", "-Wl,-rpath," + os.path.dirname(lib)])


def test_cpp_mirror_compiles_and_links():
    build()
    out = subprocess.check_output([EXE, "--compile-check"], text=True)
    assert "nova_b200" in out


@pytest.mark.gpu
def test_cpp_mirror_concurrent_commits(oracle, tmp_path):
    build()
    check_concurrent_commits(EXE, oracle, tmp_path)


def check_concurrent_commits(exe, oracle, tmp_path):
    from oracle.pyref import CURVES
    cid, c = 0, CURVES[0]
    n = 6000
    bases = oracle.gen_bases(cid, n + 1)
    sc = oracle.gen_scalars(c.scalar_field, 11, n)
    r = oracle.gen_scalars(c.scalar_field, 12, 1)
    case = tmp_path / "case.bin"
    with open(case, "wb") as f:
        for blob, sz in ((bases[:64 * n], 64), (bases[64 * n:], 64), (sc, 32), (r, 32)):
            f.write(struct.pack("<Q", len(blob) // sz))
            f.write(blob)
    out = subprocess.run([exe, str(case)], capture_output=True, text=True)
    assert out.returncode == 0, out.stdout + out.stderr
    raw = open(str(case) + ".out", "rb").read()
    (k,) = struct.unpack_from("<Q", raw, 0)
    pts = [raw[8 + 96 * i:8 + 96 * i + 96] for i in range(k)]
    off = 8 + 96 * k
    aff = lambda b: c.affine_from_bytes(oracle.jacobian_to_affine(cid, b))
    assert aff(pts[0]) == c.affine_from_bytes(oracle.msm_naive(cid, sc + r, bases))
    for j in range(32):  # 8 threads x 4 commits, prefix lengths n / (1 + j % 5)
        ln = n // (1 + j % 5)
        assert aff(pts[1 + j]) == c.affine_from_bytes(oracle.msm(cid, sc[:32 * ln], bases[:64 * ln])), j
    (nf,) = struct.unpack_from("<Q", raw, off)
    folded = raw[off + 8:off + 8 + 32 * nf]
    assert folded == oracle.axpy(c.scalar_field, sc, sc, r)
    off += 8 + 32 * nf
    (nz,) = struct.unpack_from("<Q", raw, off)
    assert raw[off + 8:off + 8 + 32 * nz] == oracle.bind_top(c.scalar_field, sc[:32 * (n & ~1)], r)


# ---- the same executable source against the CPU emulation of the library (tests/cpp/emulated_b200.cpp) ----
EXE_EMUL = os.path.join(ROOT, "tests", "cpp", "host_mirror_test_emul")
EMUL_SO = os.path.join(ROOT, "tests", "cpp", "libemulated_b200.so")


def build_emulated():
    """host_mirror_test linked against libemulated_b200.so (C-ABI symbols answered by the C oracle): the C++
    host layer of include/nova_b200.hpp runs on the CPU box."""
    from oracle import coracle
    coracle.lib()  # makes sure oracle/liboracle.so exists
    odir = os.path.join(ROOT, "oracle")
    cdir = os.path.join(ROOT, "tests", "cpp")
    esrc = os.path.join(cdir, "emulated_b200.cpp")
    hdrs = [os.path.join(ROOT, "include", f) for f in ("nova_b200.hpp", "nova_b200.h")]
    if not os.path.exists(EMUL_SO) or any(os.path.getmtime(p) > os.path.getmtime(EMUL_SO) for p in [esrc] + hdrs):
        hdir = os.path.join(ROOT, "tests", "hostcheck")  # host build of the device round kernel (hc_sc_round)
        hsrc, hso = os.path.join(hdir, "hostcheck.cpp"), os.path.join(hdir, "libhostcheck.so")
        csrc = os.path.join(ROOT, "nova_b200", "csrc")
        hdeps = [hsrc] + [os.path.join(csrc, f) for f in os.listdir(csrc) if f.endswith(".cuh")]
        if not os.path.exists(hso) or any(os.path.getmtime(p) > os.path.getmtime(hso) for p in hdeps):
            subprocess.check_call(["g++", "-O2", "-std=c++17", "-pthread", "-shared", "-fPIC", "-x", "c++", hsrc, "-o", hso])
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", esrc, "-o", EMUL_SO, "-L" + odir, "-loracle",
                               "-L" + hdir, "-lhostcheck", "-Wl,-rpath," + odir, "-Wl,-rpath," + hdir])
    src = os.path.join(cdir, "host_mirror_test.cpp")
    if not os.path.exists(EXE_EMUL) or any(os.path.getmtime(p) > os.path.getmtime(EXE_EMUL) for p in [src, EMUL_SO] + hdrs):
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-pthread", src, "-o", EXE_EMUL, "-L" + cdir, "-lemulated_b200",
                               "-Wl,-rpath," + cdir, "-Wl,-rpath," + odir,
                               "-Wl,-rpath," + os.path.join(ROOT, "tests", "hostcheck")])


def test_cpp_mirror_host_logic_concurrent_commits_cpu(oracle, tmp_path):
    """The C++ layer's commit / MSM / fold / bind wrappers, with commits issued from 8 threads, on the CPU."""
    build_emulated()
    check_concurrent_commits(EXE_EMUL, oracle, tmp_path)


def test_cpp_mirror_host_logic_resident_folding_step_cpu(oracle, tmp_path):
    """DeviceVec, WitnessStream, validate_key, R1CSShapeDev::commit_T and fold_witness_resident on the CPU."""
    build_emulated()
    check_fold(EXE_EMUL, oracle, tmp_path)


def check_fold(exe, oracle, tmp_path):
    """host_mirror_test --fold: the streamed commitment, T, comm_T and the folded W / E equal the oracle's
    (r1cs/mod.rs:578-627, 1044-1069)."""
    from oracle.ppsnark_ref import random_instance
    from oracle.pyref import CURVES, SplitMix64, mont_bytes
    from snark_parity import csr
    cid, c = 0, CURVES[0]
    fid, p = c.scalar_field, c.q
    pack = lambda xs: b"".join(mont_bytes(p, x) for x in xs)
    num_cons, num_vars, num_io = 128, 64, 2
    rng = SplitMix64(2024)
    S, W, u1, X1 = random_instance(p, rng, num_cons, num_vars, num_io)
    W1, E1 = W["W"], W["E"]
    W2 = [rng.field(p) for _ in range(num_vars)]
    X2 = [rng.field(p) for _ in range(num_io)]
    r, r_T, r_W = rng.field(p), rng.field(p), rng.field(p)
    n_key = max(num_cons, num_vars)
    bases = oracle.gen_bases(cid, n_key + 1)
    case = tmp_path / "fold.bin"

    def blob(b, sz):
        return struct.pack("<Q", len(b) // sz) + b

    def u64s(xs):
        return struct.pack("<Q", len(xs)) + struct.pack(f"<{len(xs)}Q", *xs)
    with open(case, "wb") as f:
        f.write(u64s([num_cons, num_vars, num_io]))
        for name in "ABC":
            d, idx, ptr = csr(S[name], num_cons)
            f.write(blob(pack(d), 32) + u64s(idx) + u64s(ptr))
        for v in (W1, E1, W2, X1, X2, [u1, (u1 + 1) % p, r, r_T, r_W, 1]):
            f.write(blob(pack(v), 32))
        f.write(blob(bases[:64 * n_key], 64) + blob(bases[64 * n_key:], 64))
    out = subprocess.run([exe, "--fold", str(case)], capture_output=True, text=True, timeout=120)
    assert out.returncode == 0, out.stdout + out.stderr
    raw = open(str(case) + ".out", "rb").read()
    off = 0

    def take(sz):
        nonlocal off
        (n,) = struct.unpack_from("<Q", raw, off)
        b = raw[off + 8:off + 8 + n * sz]
        off += 8 + n * sz
        return b
    bad, rejected_at = take(8), take(8)
    comm_W2, comm_T, T, Wf, Ef = take(96), take(96), take(32), take(32), take(32)
    assert struct.unpack("<Q", bad)[0] == (1 << 64) - 1  # every base is on the curve
    # the untrusted-key constructor refused the copy whose middle point was corrupted, naming that point
    assert struct.unpack("<Q", rejected_at)[0] == n_key // 2
    h = bases[64 * n_key:]
    aff = lambda jac: c.affine_from_bytes(oracle.jacobian_to_affine(cid, jac))
    assert aff(comm_W2) == c.affine_from_bytes(oracle.msm(cid, pack(W2 + [r_W]), bases[:64 * num_vars] + h))
    Z = pack([(a + b) % p for a, b in zip(W1 + [u1] + X1, W2 + [1] + X2)])
    az, bz, cz = (oracle.spmv(fid, pack(d), idx, ptr, Z) for (d, idx, ptr) in (csr(S[k], num_cons) for k in "ABC"))
    T_exp = oracle.cross_term(fid, az, bz, cz, pack(E1), None, pack([(u1 + 1) % p]))
    assert T == T_exp
    assert aff(comm_T) == c.affine_from_bytes(oracle.msm(cid, T_exp + pack([r_T]), bases[:64 * num_cons] + h))
    assert Wf == oracle.axpy(fid, pack(W1), pack(W2), pack([r]))
    assert Ef == oracle.axpy(fid, pack(E1), T_exp, pack([r]))


def test_cpp_mirror_host_logic_sumcheck_loops_cpu(oracle, tmp_path):
    """prove_quad_prod / prove_cubic_with_three_inputs of include/nova_b200.hpp (TranscriptState with pending absorbs)
    on the CPU: the emulated library strings the host build of the device round kernel together."""
    build_emulated()
    check_sumcheck(EXE_EMUL, oracle, tmp_path)


def check_sumcheck(exe, oracle, tmp_path):
    from oracle.pyref import (FIELD_MODULUS, Keccak256Transcript, SplitMix64, from_mont_bytes, mont_bytes,
                              prove_cubic_with_three_inputs, prove_quad_prod)
    fid, l = 0, 6
    p = FIELD_MODULUS[fid]
    pack = lambda xs: b"".join(mont_bytes(p, x) for x in xs)
    rng = SplitMix64(606)
    n = 1 << l
    A, B, C = ([rng.field(p) for _ in range(n)] for _ in range(3))
    taus = [rng.field(p) for _ in range(l)]
    taus[2] = 0  # a tau = 0 round
    cq, cc = rng.field(p), rng.field(p)

    def fresh():
        t = Keccak256Transcript(p, b"cpp")
        t.absorb_scalar(b"a", 5)
        t.squeeze(b"x")
        t.absorb_scalar(b"b", 7)  # left pending
        return t
    t0 = fresh()
    case = tmp_path / "sc.bin"
    blob = lambda b, sz: struct.pack("<Q", len(b) // sz) + b
    with open(case, "wb") as f:
        f.write(struct.pack("<QQ", 1, l))
        for v in (A, B, C, taus, [cq, cc]):
            f.write(blob(pack(v), 32))
        f.write(blob(struct.pack("<Q", t0.round) + t0.state, 8))
        f.write(blob(t0.buf, 1))
    out = subprocess.run([exe, "--sumcheck", str(case)], capture_output=True, text=True, timeout=120)
    assert out.returncode == 0, out.stdout + out.stderr
    raw = open(str(case) + ".out", "rb").read()
    off = 0

    def take(sz):
        nonlocal off
        (k,) = struct.unpack_from("<Q", raw, off)
        b = raw[off + 8:off + 8 + k * sz]
        off += 8 + k * sz
        return b
    canon = lambda b: [int.from_bytes(b[i:i + 32], "little") for i in range(0, len(b), 32)]
    mont = lambda b: [from_mont_bytes(p, b[i:i + 32]) for i in range(0, len(b), 32)]
    for which, ncoef in ((0, 2), (1, 3)):
        t = fresh()
        exp = prove_quad_prod(p, cq, l, A, B, t) if which == 0 else prove_cubic_with_three_inputs(p, cc, taus, A, B, C, t)
        polys, rs, finals, trb, left = take(32), take(32), take(32), take(72), take(8)
        flat = canon(polys)
        assert [flat[ncoef * j:ncoef * (j + 1)] for j in range(l)] == [list(q) for q in exp[0]]
        assert mont(rs) == list(exp[1]) and mont(finals) == list(exp[2])
        assert struct.unpack("<Q", trb[:8])[0] == t.round and trb[8:] == t.state and struct.unpack("<Q", left)[0] == 0


@pytest.mark.gpu
@pytest.mark.parametrize("log2n", [14, 18])
def test_cpp_concurrent_commits_overlap_and_agree(log2n, tmp_path):
    """host_mirror_test --concurrency: 4 commitments issued from one thread in turn and from 4 threads at once
    (rayon in the reference: ppsnark.rs:457-470) give the same points; each call takes its own host slot (workspace +
    streams) of the key, so the calls overlap on the device -- the measured ratio is printed (profiles/r02e)."""
    import json

    from nova_b200.provider import Curve, _jac_to_affine
    build()
    points = tmp_path / "concurrency_points.bin"
    out = subprocess.check_output([EXE, "--concurrency", str(log2n), "4", str(points)], text=True, timeout=300)
    res = json.loads(out.strip().splitlines()[-1])
    raw = points.read_bytes()
    pts = [_jac_to_affine(Curve(0), raw[96 * i:96 * i + 96]) for i in range(8)]
    assert pts[:4] == pts[4:] and len(set(pts[:4])) == 4
    assert res["ms_serial"] > 0 and res["ms_concurrent"] > 0
    print(res)


def check_mgpu(exe, oracle, tmp_path, ndev):
    """host_mirror_test --mgpu: MultiGpuCommitmentKey == CommitmentKey on the same inputs (and == the oracle)"""
    from nova_b200.provider import Curve, _jac_to_affine
    from oracle.pyref import CURVES
    cid, c = 0, CURVES[0]
    n = 9000
    bases = oracle.gen_bases(cid, n + 1)
    sc = oracle.gen_scalars(c.scalar_field, 21, n)
    r = oracle.gen_scalars(c.scalar_field, 22, 1)
    case = tmp_path / "mgpu.bin"
    with open(case, "wb") as f:
        for blob, size in ((bases[:64 * n], 64), (bases[64 * n:], 64), (sc, 32), (r, 32)):
            f.write((len(blob) // size).to_bytes(8, "little") + blob)
    out = subprocess.check_output([exe, "--mgpu", str(case), str(ndev)], text=True, timeout=300)
    assert "mgpu ok" in out
    raw = open(str(case) + ".out", "rb").read()
    k = int.from_bytes(raw[:8], "little")
    pts = [_jac_to_affine(Curve(cid), raw[8 + 96 * i:8 + 96 * i + 96]) for i in range(2 * k)]
    assert pts[:k] == pts[k:]
    assert pts[1] == c.affine_from_bytes(oracle.msm(cid, sc, bases[:64 * n]))


def test_cpp_mirror_multi_gpu_key_host_logic_cpu(oracle, tmp_path):
    build_emulated()
    check_mgpu(EXE_EMUL, oracle, tmp_path, 3)


@pytest.mark.gpu
@pytest.mark.parametrize("ndev", [1, 3])
def test_cpp_mirror_multi_gpu_key(oracle, tmp_path, ndev):
    build()
    check_mgpu(EXE, oracle, tmp_path, ndev)
