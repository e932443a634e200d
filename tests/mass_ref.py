"""CPU reference of the mass operator IProductWRTBase_w o BwdTrans: the composition of the two oracle operators
(oracle/__init__.py), whose contract the fused kernels match bit for bit."""
import oracle


def mass_quad(nq, nelmt, b0, b1, inp, w=None):
    return oracle.iproduct_quad(nq, nq, nelmt, b0, b1, oracle.bwdtrans_quad(nq, nq, nelmt, b0, b1, inp), w)


def mass_hex(nq, nelmt, b0, b1, b2, inp, w=None):
    return oracle.iproduct_hex(nq, nq, nq, nelmt, b0, b1, b2, oracle.bwdtrans_hex(nq, nq, nq, nelmt, b0, b1, b2, inp), w)
