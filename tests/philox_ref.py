"""numpy reference of the in-kernel sampler (csrc/common.cuh): Philox4x32-10 and the uniform / normal draws built on it.

Vectorised over elements in uint64 arithmetic, so it runs on whole edge / node arrays.  Layout, as the kernels use it:
  counter = (elem_lo, elem_hi, step, 0)   (last word 1 for the normal draw)
  key     = (seed_lo, seed_hi)
  uniform = (x >> 8) * 2^-24                                   exact in fp32
  normal  = sqrt(-2 ln u1) cos(2 pi u2),  u1 = ((x >> 8) + 0.5) * 2^-24 in fp32,  u2 = (y >> 8) * 2^-24"""
import numpy as np

M32 = np.uint64(0xFFFFFFFF)
_M0, _M1 = np.uint64(0xD2511F53), np.uint64(0xCD9E8D57)
_W0, _W1 = np.uint64(0x9E3779B9), np.uint64(0xBB67AE85)


def philox4x32_10(ctr, key):
  """ctr: 4 arrays (or ints) of 32-bit words, key: 2 words -> 4 uint64 arrays holding the 32-bit output words."""
  c = [np.asarray(x, dtype=np.uint64) & M32 for x in ctr]
  c = np.broadcast_arrays(*c)
  c0, c1, c2, c3 = [x.copy() for x in c]
  k0, k1 = np.uint64(int(key[0]) & 0xFFFFFFFF), np.uint64(int(key[1]) & 0xFFFFFFFF)
  for _ in range(10):
    p0, p1 = _M0 * c0, _M1 * c2                  # 32 x 32 -> 64 bit: no overflow in uint64
    hi0, lo0 = p0 >> np.uint64(32), p0 & M32
    hi1, lo1 = p1 >> np.uint64(32), p1 & M32
    c0, c1, c2, c3 = hi1 ^ c1 ^ k0, lo1, hi0 ^ c3 ^ k1, lo0
    k0, k1 = (k0 + _W0) & M32, (k1 + _W1) & M32
  return c0, c1, c2, c3


def _words(seed, step, elem, last):
  elem = np.asarray(elem, dtype=np.uint64)
  seed = int(seed) & 0xFFFFFFFFFFFFFFFF
  return philox4x32_10((elem & M32, elem >> np.uint64(32), np.uint64(int(step) & 0xFFFFFFFF), np.uint64(last)),
                       (seed & 0xFFFFFFFF, seed >> 32))


def _unit24(x):
  return (x >> np.uint64(8)).astype(np.float32) * np.float32(2.0 ** -24)


def uniform(seed, step, elem):
  """philox_uniform: U[0,1) with 24 random bits, bit-exact fp32."""
  return _unit24(_words(seed, step, elem, 0)[0])


def normal_uniforms(seed, step, elem, counter_word3=1):
  """(u1, u2) of philox_normal in fp32, rounded exactly as the kernel rounds them ((x >> 8) + 0.5f is one fp32 add).
  counter_word3 is 1 in the kernel; other values only serve to show what a layout error would change."""
  x, y = _words(seed, step, elem, counter_word3)[:2]
  u1 = ((x >> np.uint64(8)).astype(np.float32) + np.float32(0.5)) * np.float32(2.0 ** -24)
  return u1, _unit24(y)


def box_muller(u1, u2):
  return np.sqrt(-2.0 * np.log(np.asarray(u1, np.float64))) * np.cos(2.0 * np.pi * np.asarray(u2, np.float64))


def normal(seed, step, elem):
  """philox_normal evaluated in float64 from the kernel's fp32 u1 / u2: differs from the device value only by the
  error of the device logf / cospif / sqrtf (a few fp32 ulp)."""
  return box_muller(*normal_uniforms(seed, step, elem))
