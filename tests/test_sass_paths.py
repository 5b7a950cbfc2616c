"""`tools/sass_paths.py` (instruction counts of the march loop's paths) on a hand-made SASS listing with the
shape of the inline-shading kernel: a work loop around the march loop, which holds the extra-fetch loop, the
sigma test's branch over the shading block and the loop tail."""
import os
import sys

sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tools"))
import sass_paths  # noqa: E402

LISTING = """
        /*0000*/                   MOV R1, c[0x0][0x28] ;                                   /* 0x00000a0000017a02 */
        /*0010*/                   FFMA2 R24, R4.F32, R16.F32x2.HI_LO, R18.F32x2.HI_LO ;    /* 0x0000000000000000 */
        /*0020*/                   LDS R27, [R38+0x10] ;                                    /* 0x0000000000000000 */
        /*0030*/                   LDG.E.CONSTANT R41, desc[UR8][R28.64] ;                  /* 0x0000000000000000 */
        /*0040*/                   ISETP.GE.AND P0, PT, R41, RZ, PT ;                       /* 0x0000000000000000 */
        /*0050*/              @!P0 BRA 0x90 ;                                               /* 0x0000000000000000 */
        /*0060*/                   STS [R42+0x210], R41 ;                                   /* 0x0000000000000000 */
        /*0070*/                   LDG.E.CONSTANT R41, desc[UR8][R28.64] ;                  /* 0x0000000000000000 */
        /*0080*/               @P0 BRA 0x60 ;                                               /* 0x0000000000000000 */
        /*0090*/                   FADD2 R26, -R26.F32x2.HI_LO, 8388608 ;                   /* 0x0000000000000000 */
        /*00a0*/              @!P0 BRA 0xe0 ;                                               /* 0x0000000000000000 */
        /*00b0*/                   LDG.E.NA.EFL2.256.CONSTANT R12, R28, desc[UR8][R20.64] ; /* 0x0000000000000000 */
        /*00c0*/                   FFMA2 R30, R45.F32, R30.F32x2.HI_LO, R32.F32x2.HI_LO ;   /* 0x0000000000000000 */
        /*00d0*/              @!P0 BRA 0x110 ;                                              /* 0x0000000000000000 */
        /*00e0*/                   FADD R4, R42, R4 ;                                       /* 0x0000000000000000 */
        /*00f0*/                   FSETP.GEU.AND P0, PT, R4, R56, PT ;                      /* 0x0000000000000000 */
        /*0100*/              @!P0 BRA 0x10 ;                                               /* 0x0000000000000000 */
        /*0110*/                   BRA.U !UP0, 0x0 ;                                        /* 0x0000000000000000 */
        /*0120*/                   EXIT ;                                                   /* 0x0000000000000000 */
"""


def test_parse_and_branch_targets():
    insns = sass_paths.parse_sass(LISTING)
    assert len(insns) == 19 and insns[1] == (0x10, "FFMA2 R24, R4.F32, R16.F32x2.HI_LO, R18.F32x2.HI_LO")
    assert sass_paths.branch_target("@!P0 BRA 0x90") == 0x90
    assert sass_paths.branch_target("BRA.U !UP0, 0x140") == 0x140
    assert sass_paths.branch_target("@!P1 BRA P0, 0x9f0") == 0x9f0
    assert sass_paths.branch_target("FADD R4, R42, R4") is None


def test_path_counts():
    r = sass_paths.analyse(sass_paths.parse_sass(LISTING))
    assert r["march_loop"] == ["0x10", "0x100"]
    assert r["fetch"] == 3          # 0x60..0x80
    assert r["shade"] == 3          # 0xb0..0xd0
    assert r["empty"] == 10         # 0x10..0x50, 0x90, 0xa0, 0xe0..0x100
    assert r["paired_loop"] == 3 and r["paired_kernel"] == 3
