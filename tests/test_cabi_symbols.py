"""CPU: the C-ABI library builds for sm_100a, loads, and exports every symbol include/tts_b200.h
declares (no compute calls without a GPU)."""
import ctypes as C
import os
import re

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared_symbols():
    src = open(os.path.join(ROOT, "include", "tts_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(tts_[a-z0-9_]+)\s*\(", src)))


def test_header_symbols_all_exported_and_bound():
    from transformer_tacotron2_b200 import _lib
    lib = _lib.load()
    names = _declared_symbols()
    assert len(names) >= 18
    for n in names:
        assert hasattr(lib, n), n
        assert n in _lib.SIGNATURES, f"{n} declared in the header but not bound in _lib.SIGNATURES"
    assert set(_lib.SIGNATURES) == set(names)
    assert b"sm_100a" in lib.tts_version()


def test_library_contains_sm100a_code():
    import subprocess
    from transformer_tacotron2_b200 import _lib
    _lib.load()
    out = subprocess.run(["cuobjdump", "-lelf", _lib.LIB_PATH], capture_output=True, text=True).stdout
    assert "sm_100a" in out


def test_no_gpu_means_loud_failure_not_fallback():
    import pytest
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from transformer_tacotron2_b200 import TransformerTTS
    m = TransformerTTS()
    with pytest.raises(RuntimeError):
        m.inference(torch.zeros(1, 4, dtype=torch.int64), torch.tensor([4]), max_len=2)
    # tts_create itself refuses without an sm_100 device
    from transformer_tacotron2_b200 import _lib
    lib = _lib.load()
    cc = _lib.TtsConfig(C.sizeof(_lib.TtsConfig), 128, 512, 8, 6, 6, 2048, 80, 256, 3, 5, 512, 5, 2048, 1e-5, 1e-5)
    h = C.c_void_p()
    assert lib.tts_create(C.byref(cc), 0, C.byref(h)) != 0


def test_training_without_gpu_fails_loudly_too():
    import pytest
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from transformer_tacotron2_b200 import TransformerTTS
    from transformer_tacotron2_b200.training import Trainer
    with pytest.raises(RuntimeError):
        Trainer(TransformerTTS())
    # the training entry points refuse a null handle instead of crashing
    from transformer_tacotron2_b200 import _lib
    lib = _lib.load()
    assert lib.tts_train_begin(None) != 0
    assert lib.tts_train_num_tensors(None) == -1
    assert lib.tts_train_workspace_bytes(None, 4, 10, 20) == 0


def test_product_package_never_imports_oracle():
    pkg = os.path.join(ROOT, "transformer_tacotron2_b200")
    for dp, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                txt = open(os.path.join(dp, f)).read()
                assert "import oracle" not in txt and "from oracle" not in txt, f


def test_kv_cache_block_layout():
    """The decode kernel's cache block layout (host arithmetic of the shipped library, no GPU): a bijection onto 8192 elements;
    rows [0, 16 n) of K and V together fill exactly the first 16 n * 128 elements (so any ring stage is ONE contiguous copy);
    K rows are row-major inside a 16-row sub-chunk; the V half of a sub-chunk is in mma.m16n8k16 A-fragment order of V^T."""
    from transformer_tacotron2_b200 import _lib
    lib = _lib.load()
    idx = {(w, r, d): lib.tts_debug_kv_index(r, d, w) for w in (0, 1) for r in range(64) for d in range(64)}
    assert sorted(idx.values()) == list(range(8192))
    assert lib.tts_debug_kv_index(64, 0, 0) == -1 and lib.tts_debug_kv_index(0, 64, 1) == -1 and lib.tts_debug_kv_index(0, 0, 2) == -1
    for n in range(1, 5):
        got = sorted(v for (w, r, d), v in idx.items() if r < 16 * n)
        assert got == list(range(16 * n * 128))
    for r in range(64):
        base = (r // 16) * 2048 + (r % 16) * 64
        assert [idx[(0, r, d)] for d in range(64)] == list(range(base, base + 64))
    for s in range(4):                     # 16-row sub-chunk
        for dt in range(4):                # 16-dim tile of V^T
            for g in range(8):
                for t4 in range(4):
                    base = s * 2048 + 1024 + (dt * 32 + g * 4 + t4) * 8
                    want = [(16 * s + 4 * t4 + 0, 16 * dt + g), (16 * s + 4 * t4 + 1, 16 * dt + g),            # a0: A[g][2 t4, 2 t4 + 1]
                            (16 * s + 4 * t4 + 0, 16 * dt + g + 8), (16 * s + 4 * t4 + 1, 16 * dt + g + 8),    # a1: A[g + 8][..]
                            (16 * s + 4 * t4 + 2, 16 * dt + g), (16 * s + 4 * t4 + 3, 16 * dt + g),            # a2: A[g][2 t4 + 8, + 9]
                            (16 * s + 4 * t4 + 2, 16 * dt + g + 8), (16 * s + 4 * t4 + 3, 16 * dt + g + 8)]    # a3
                    assert [idx[(1, r, d)] for r, d in want] == list(range(base, base + 8))


def _pack(lib, w, rows, kp_base, KP, TW):
    import ctypes as C
    import numpy as np
    w = np.ascontiguousarray(w, dtype=np.float32)
    rows = np.ascontiguousarray(rows, dtype=np.int32)
    need = lib.tts_debug_pack_segment(w.ctypes.data, w.shape[0], w.shape[1], rows.ctypes.data, len(rows), kp_base, KP, TW, None, 0)
    assert need == len(rows) // 16 * KP * 1024
    out = np.zeros(need, dtype=np.uint8)
    got = lib.tts_debug_pack_segment(w.ctypes.data, w.shape[0], w.shape[1], rows.ctypes.data, len(rows), kp_base, KP, TW, out.ctypes.data, need)
    assert got == need
    return out.view(np.uint16)                  # bf16 bit patterns


def _bf16_bits(x):
    import numpy as np
    import torch
    return torch.from_numpy(np.ascontiguousarray(x, dtype=np.float32)).to(torch.bfloat16).view(torch.int16).numpy().view(np.uint16)


def _read_fragment_block(stream16, byte_off, lane, ks):
    """The four 32-bit registers lane `lane` loads for k-step `ks` of the 1 KB block at byte_off (kernel: wp[(block * 2 + ks) * 32 + lane])
    -> bf16 bit patterns [a0.lo, a0.hi, a1.lo, a1.hi, a2.lo, a2.hi, a3.lo, a3.hi]."""
    e = byte_off // 2 + (ks * 32 + lane) * 8
    return stream16[e:e + 8]


def test_decode_weight_stream_matches_kernel_addressing():
    """Host packer (tts_finalize_weights -> pack_cluster_segment) against the addressing of the decode kernel's GEMMs, on CPU:
    wide GEMMs read their K range in two halves (cl_gemm<KP, TW, 2>), narrow ones as 4 tiles x 4 K quarters (cl_gemm_ksplit<4, 16, 4>),
    FFN2 two tiles per warp over a K slice.  Every fragment register must hold W[row][k] of the mma.m16n8k16 A layout."""
    import numpy as np
    from transformer_tacotron2_b200 import _lib
    lib = _lib.load()
    rng = np.random.default_rng(5)

    def check(stream, W, rows, tile, kp, byte_off):
        want = _bf16_bits(W)
        for ks in range(2):
            for lane in range(32):
                g, t4 = lane >> 2, lane & 3
                k0 = kp * 32 + ks * 16 + t4 * 2
                r0, r1 = rows[tile * 16 + g], rows[tile * 16 + g + 8]
                regs = _read_fragment_block(stream, byte_off, lane, ks)
                exp = [want[r0, k0], want[r0, k0 + 1], want[r1, k0], want[r1, k0 + 1],
                       want[r0, k0 + 8], want[r0, k0 + 9], want[r1, k0 + 8], want[r1, k0 + 9]]
                assert list(regs) == exp, (tile, kp, ks, lane)

    # ---- wide GEMM, FFN1-like slice of rank 3: 256 rows (16 tiles = 16 warps), K = 512, two halves of 8 k-pairs
    W = rng.standard_normal((2048, 512)).astype(np.float32)
    rows = np.arange(256 * 3, 256 * 4)
    stream = np.concatenate([_pack(lib, W, rows, 0, 8, 1), _pack(lib, W, rows, 8, 8, 1)])
    KH, BW = 8, 8 * 1024
    for warp in (0, 5, 15):
        for h in range(2):
            run = (h * 16 + warp) * BW                         # stage (h * nst + warp / WPS), offset (warp % WPS) * BW: contiguous runs
            for kl in (0, 3, 7):
                check(stream, W, rows, warp, h * KH + kl, run + kl * 1024)      # TW = 1: block index kl * TW + j = kl
    # ---- narrow GEMM, O-projection slice of rank 6: 64 rows (4 tiles), K = 512; warp w -> tile w % 4, quarter w / 4, run = tile * 4 + quarter
    W = rng.standard_normal((512, 512)).astype(np.float32)
    rows = np.arange(64 * 6, 64 * 7)
    stream = _pack(lib, W, rows, 0, 16, 1)
    for warp in range(16):
        tile, kq = warp % 4, warp // 4
        run = (tile * 4 + kq) * 4096
        for ku in range(4):
            check(stream, W, rows, tile, kq * 4 + ku, run + ku * 1024)
    # ---- FFN2 (K-split over ranks): all 512 rows, K slice [256 r, 256 r + 256) of d_ff, two tiles per warp, two halves of 4 k-pairs
    W = rng.standard_normal((512, 2048)).astype(np.float32)
    rows = np.arange(512)
    r = 5
    stream = np.concatenate([_pack(lib, W, rows, 8 * r, 4, 2), _pack(lib, W, rows, 8 * r + 4, 4, 2)])
    KH, TW, BW = 4, 2, 2 * 4 * 1024
    for warp in (0, 9, 15):
        for h in range(2):
            run = (h * 16 + warp) * BW
            for kl in range(KH):
                for j in range(TW):
                    check(stream, W, rows, warp * TW + j, 8 * r + h * KH + kl, run + (kl * TW + j) * 1024)
    # ---- zero rows (the head segment pads 81 -> 96 columns) and K padding (prenet fc1: K = 80 -> 128)
    W = rng.standard_normal((81, 512)).astype(np.float32)
    rows = np.array([16 * 5 + i if 16 * 5 + i < 81 else -1 for i in range(16)], dtype=np.int32)
    stream = _pack(lib, W, rows, 0, 16, 1)
    assert _read_fragment_block(stream, 0, 0, 0)[0] == _bf16_bits(W)[80, 0]              # row 80 (stop) is lane g = 0
    assert not _read_fragment_block(stream, 0, 4, 0)[:2].any()                            # g = 1 -> row 81: zero
    W = rng.standard_normal((256, 80)).astype(np.float32)
    stream = _pack(lib, W, np.arange(32), 0, 4, 1)
    assert not _read_fragment_block(stream, 2 * 1024, 0, 1)[:2].any()                     # k = 2 * 32 + 16 = 80: padding


def test_sequence_test_entry_points_validate_on_the_host():
    """tts_k_gemm_epi and tts_k_attention_strided refuse layouts their kernels cannot handle before any device work (the
    addresses below are never dereferenced)."""
    import pytest
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present: tests/test_gpu_seq_kernels.py checks the same with real buffers")
    from transformer_tacotron2_b200 import _lib
    lib = _lib.load()
    fake = 1 << 20

    def gemm(**kw):
        a = _lib.TtsKGemm()
        a.struct_size = C.sizeof(_lib.TtsKGemm)
        base = dict(A=fake, lda=512, W=fake, ldw=512, M=74, N=6144, K=512, taps=1, T=37, bias=fake, drop_site=-1, dropw_site=-1,
                    scatter=1, out_bf16=fake, B=2, Lpad=48)
        for k, v in dict(base, **kw).items():
            setattr(a, k, v)
        return lib.tts_k_gemm_epi(C.byref(a), None)
    assert gemm(struct_size=8) == -1
    assert gemm(Lpad=40) == -1                          # row-major cache: Lpad a multiple of 16
    assert gemm(Lpad=32) == -1                          # Lpad < T
    assert gemm(N=5632) == -1                           # cross K/V: N a multiple of 1024
    assert gemm(scatter=3) == -1                        # blocked cache: Lpad a multiple of 64
    assert gemm(B=3) == -1                              # B * T != M
    assert gemm(T=36) == -1                             # M % T
    assert gemm(scatter=2, N=80, out_f32=fake, out2_f32=fake) == -1      # heads: N = 81
    assert gemm(scatter=0, N=512, ldo=500) == -1        # ldo < N
    assert gemm(scatter=0, N=1024, ldo=1024, pe=fake) == -1              # pe rows are 512 wide
    assert gemm(bias=fake + 2) == -1                    # not even element-aligned
    assert gemm(lda=500) == -1                          # TMA row stride: a multiple of 8 elements
    assert gemm(taps=3) == -1
    st = (C.c_int64 * 12)(*([64 * 1536, 64, 1536] * 3 + [64 * 512, 64, 516]))
    assert lib.tts_k_attention_strided(fake, fake, fake, fake, None, None, st, 2, 8, 64, 64, 0, None) == -1
    st = (C.c_int64 * 12)(*([64 * 1536, 64, 1536] * 3 + [64 * 512, 64, 512]))
    assert lib.tts_k_attention_strided(fake + 2, fake, fake, fake, None, None, st, 2, 8, 64, 64, 0, None) == -1
