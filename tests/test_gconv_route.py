"""CPU: the engine routes of the generalised convolution (csrc/gconv.cu) for the layers of UNet(1,2) and UNet_S at
512x512, B = 16.  The _supported queries and unetb200_gconv_wgrad_plan are host code (148 SMs assumed without a GPU),
and what they answer decides which kernels a step launches and how ops.py names them in profiles (algo_used)."""
import ctypes as C

from unetb200 import _lib

TAPS3 = [(kh - 1, kw - 1) for kh in range(3) for kw in range(3)]
MODES = ((_lib.BF16, _lib.ALGO_AUTO), (_lib.F32, _lib.ALGO_PREFER_TC), (_lib.F32, _lib.ALGO_SIMT))

# (C_in, N, output H = W, ConvTranspose2d) -> per mode of MODES: (affine_relu, affine_relu_pool, affine_relu_outconv
# with 2 classes, dgrad_bnbwd, wgrad_plan splits, wgrad_plan algo_used), 16-byte aligned pointers
TABLE = {
    (1, 16, 512, 0): ((1, 0, 0, 0, 296, 1), (0, 0, 0, 0, 888, 1), (0, 0, 0, 0, 888, 1)),
    (1, 64, 512, 0): ((1, 0, 0, 0, 888, 1), (0, 0, 0, 0, 888, 1), (0, 0, 0, 0, 888, 1)),
    (16, 16, 512, 0): ((1, 1, 0, 1, 296, 2), (1, 0, 0, 0, 2368, 1), (0, 0, 0, 0, 2368, 1)),
    (16, 32, 256, 0): ((1, 1, 0, 1, 296, 2), (1, 0, 0, 0, 1184, 1), (0, 0, 0, 0, 1184, 1)),
    (32, 16, 512, 0): ((1, 1, 0, 1, 296, 2), (1, 0, 0, 0, 1184, 1), (0, 0, 0, 0, 1184, 1)),
    (32, 32, 256, 0): ((1, 1, 0, 1, 296, 2), (1, 0, 0, 0, 592, 1), (0, 0, 0, 0, 592, 1)),
    (32, 64, 128, 0): ((1, 1, 0, 0, 148, 2), (1, 0, 0, 1, 148, 2), (0, 0, 0, 0, 296, 1)),
    (32, 64, 512, 1): ((0, 0, 0, 0, 296, 2), (0, 0, 0, 0, 888, 1), (0, 0, 0, 0, 888, 1)),
    (64, 32, 256, 0): ((1, 1, 0, 1, 148, 2), (0, 0, 0, 0, 296, 1), (0, 0, 0, 0, 296, 1)),
    (64, 64, 128, 0): ((1, 1, 1, 1, 148, 2), (1, 0, 0, 1, 148, 2), (0, 0, 0, 0, 99, 1)),
    (64, 64, 512, 0): ((1, 1, 1, 1, 296, 2), (1, 0, 0, 1, 148, 2), (0, 0, 0, 0, 99, 1)),
    (64, 128, 64, 0): ((1, 1, 0, 1, 64, 2), (1, 0, 0, 1, 64, 2), (0, 0, 0, 0, 50, 1)),
    (64, 128, 256, 0): ((1, 1, 0, 1, 148, 2), (1, 0, 0, 1, 148, 2), (0, 0, 0, 0, 50, 1)),
    (64, 128, 256, 1): ((0, 0, 0, 0, 296, 2), (0, 0, 0, 0, 444, 1), (0, 0, 0, 0, 444, 1)),
    (128, 64, 128, 0): ((1, 1, 1, 1, 148, 2), (1, 0, 0, 1, 148, 2), (0, 0, 0, 0, 50, 1)),
    (128, 64, 512, 0): ((1, 1, 1, 1, 148, 2), (1, 0, 0, 1, 148, 2), (0, 0, 0, 0, 50, 1)),
    (128, 128, 64, 0): ((1, 1, 0, 1, 37, 2), (1, 0, 0, 1, 49, 2), (0, 0, 0, 0, 25, 1)),
    (128, 128, 256, 0): ((1, 1, 0, 1, 74, 2), (1, 0, 0, 1, 148, 2), (0, 0, 0, 0, 25, 1)),
    (128, 256, 32, 0): ((1, 1, 0, 1, 16, 2), (1, 0, 0, 1, 16, 2), (0, 0, 0, 0, 13, 1)),
    (128, 256, 128, 0): ((1, 1, 0, 1, 37, 2), (1, 0, 0, 1, 74, 2), (0, 0, 0, 0, 13, 1)),
    (128, 256, 128, 1): ((0, 0, 0, 0, 37, 2), (0, 0, 0, 0, 37, 2), (0, 0, 0, 0, 111, 1)),
    (128, 256, 512, 1): ((0, 0, 0, 0, 74, 2), (0, 0, 0, 0, 74, 2), (0, 0, 0, 0, 111, 1)),
    (256, 128, 64, 0): ((1, 1, 0, 1, 49, 2), (1, 0, 0, 1, 49, 2), (0, 0, 0, 0, 13, 1)),
    (256, 128, 256, 0): ((1, 1, 0, 1, 74, 2), (1, 0, 0, 1, 74, 2), (0, 0, 0, 0, 13, 1)),
    (256, 256, 32, 0): ((1, 1, 0, 1, 12, 2), (1, 0, 0, 1, 12, 2), (0, 0, 0, 0, 7, 1)),
    (256, 256, 128, 0): ((1, 1, 0, 1, 37, 2), (1, 0, 0, 1, 37, 2), (0, 0, 0, 0, 7, 1)),
    (256, 512, 64, 0): ((1, 1, 0, 1, 12, 2), (1, 0, 0, 1, 12, 2), (0, 0, 0, 0, 4, 1)),
    (256, 512, 64, 1): ((0, 0, 0, 0, 16, 2), (0, 0, 0, 0, 16, 2), (0, 0, 0, 0, 28, 1)),
    (256, 512, 256, 1): ((0, 0, 0, 0, 37, 2), (0, 0, 0, 0, 37, 2), (0, 0, 0, 0, 28, 1)),
    (512, 256, 128, 0): ((1, 1, 0, 1, 12, 2), (1, 0, 0, 1, 12, 2), (0, 0, 0, 0, 4, 1)),
    (512, 512, 64, 0): ((1, 1, 0, 1, 6, 2), (1, 0, 0, 1, 6, 2), (0, 0, 0, 0, 2, 1)),
    (512, 1024, 32, 0): ((1, 1, 0, 1, 3, 2), (1, 0, 0, 1, 3, 2), (0, 0, 0, 0, 1, 1)),
    (512, 1024, 128, 1): ((0, 0, 0, 0, 9, 2), (0, 0, 0, 0, 9, 2), (0, 0, 0, 0, 7, 1)),
    (1024, 512, 64, 0): ((1, 1, 0, 1, 3, 2), (1, 0, 0, 1, 3, 2), (0, 0, 0, 0, 1, 1)),
    (1024, 1024, 32, 0): ((1, 1, 0, 1, 3, 2), (1, 0, 0, 1, 3, 2), (0, 0, 0, 0, 1, 1)),
    (1024, 2048, 64, 1): ((0, 0, 0, 0, 2, 2), (0, 0, 0, 0, 2, 2), (0, 0, 0, 0, 2, 1)),
}


def test_routes_of_the_unet_layers():
    lib = _lib.load()
    P = 1 << 20
    for (cin, n, hw, conv_t), want in TABLE.items():
        for (dt, algo), expect in zip(MODES, want):
            d = _lib.GConv()
            d.dtype, d.algo, d.B, d.Cin, d.ld_in, d.in_scale, d.N = dt, algo, 16, cin, cin, 1, n
            if conv_t:      # ConvTranspose2d(k2, s2) fprop into the upper half of a concat buffer
                d.Hm = d.Wm = d.Hin = d.Win = hw // 2
                d.ntaps, d.nquad, d.out_scale, d.Hout, d.Wout, d.ld_out = 1, 4, 2, hw, hw, n // 2
            else:
                d.Hm = d.Wm = d.Hin = d.Win = d.Hout = d.Wout = hw
                d.ntaps, d.nquad, d.out_scale, d.ld_out = 9, 1, 1, n
                for t, (dy, dx) in enumerate(TAPS3):
                    d.tap_dy[t], d.tap_dx[t] = dy, dx
            bd = C.byref(d)
            splits, used = C.c_int(0), C.c_int(0)
            assert lib.unetb200_gconv_wgrad_plan(bd, C.byref(splits), C.byref(used)) == 0
            got = (lib.unetb200_gconv_fprop_affine_relu_supported(bd, P, P, P),
                   lib.unetb200_gconv_fprop_affine_relu_pool_supported(bd, P, P, P, P, n),
                   lib.unetb200_gconv_fprop_affine_relu_outconv_supported(bd, P, P, 2),
                   lib.unetb200_gconv_dgrad_bnbwd_supported(bd, P, P, P), splits.value, used.value)
            assert got == expect, ((cin, n, hw, conv_t), dt, algo)
