"""Builds tests/simt/_build/libapk_simt_corr.so: the device part of astrild_b200/csrc/corr.cu (plane-symmetrising fill,
real-space binning in its four instantiations, fold), unchanged, compiled by g++ against tests/simt/simt.h with the
helpers of build_simt.py.  Tests only."""
import os

import build_simt as bs


def corr_device_part(path: str) -> str:
    """corr.cu without its host code and C entry points (everything from ``using namespace apk;`` on); the dynamic
    shared memory declaration points at the emulator's buffer and the two inline-PTX RED helpers become plain adds."""
    text = open(path).read()
    text = text[:text.index("using namespace apk;")]
    assert text.count(bs.DYN_SMEM_DECL) == 1
    text = text.replace(bs.DYN_SMEM_DECL, "unsigned char *smem_raw = simt::dyn_smem;")
    for ptx in ('asm volatile("red.global.add.f64 [%0], %1;" ::"l"(addr), "d"(v) : "memory");',
                'asm volatile("red.global.add.u64 [%0], %1;" ::"l"(addr), "l"(v) : "memory");'):
        assert text.count(ptx) == 1
        text = text.replace(ptx, "*addr += v;")
    return text


def build_corr(force: bool = False) -> str:
    """-> tests/simt/_build/libapk_simt_corr.so (xi_fill_kernel, xi_bin_kernel, xi_fold_kernel on CPU fibers)"""
    so = os.path.join(bs.OUT_DIR, "libapk_simt_corr.so")
    srcs = [os.path.join(bs.CSRC, f) for f in ("corr.cu", "apk_common.cuh")]
    srcs += [os.path.join(bs.HERE, f) for f in ("simt.h", "corr_host.cpp", "build_simt.py", "build_simt_corr.py")]
    if not force and bs._fresh(so, srcs):
        return so
    os.makedirs(bs.OUT_DIR, exist_ok=True)
    with open(os.path.join(bs.OUT_DIR, "corr_kernels.inc"), "w") as f:
        f.write(corr_device_part(srcs[0]))
    return bs._gxx("corr_host.cpp", bs.OUT_DIR, so)


if __name__ == "__main__":
    print(build_corr(force=True))
