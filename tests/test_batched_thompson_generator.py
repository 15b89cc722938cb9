"""CPU: a numpy restatement of the batched Thompson stage's normal generator (csrc/batched_thompson.cu, bt_normal):
Philox4x32-10 keyed by the run's 64-bit seed at counter (row, agent, iteration, 0), Box-Muller on its 128 output bits.
The GPU tests compare the device's normals with it."""
import numpy as np

M32 = np.uint64(0xFFFFFFFF)


def philox4x32_10(c, k):
    """Philox4x32-10 (Salmon, Moraes, Dror and Shaw, SC'11) on arrays of 32-bit words: c[4], k[2] -> 4 output words."""
    c = [np.asarray(v, dtype=np.uint64) & M32 for v in c]
    k = [np.asarray(v, dtype=np.uint64) & M32 for v in k]
    for _ in range(10):
        p0 = np.uint64(0xD2511F53) * c[0]
        p1 = np.uint64(0xCD9E8D57) * c[2]
        c = [(p1 >> np.uint64(32)) ^ c[1] ^ k[0], p1 & M32, (p0 >> np.uint64(32)) ^ c[3] ^ k[1], p0 & M32]
        k = [(k[0] + np.uint64(0x9E3779B9)) & M32, (k[1] + np.uint64(0xBB67AE85)) & M32]
    return c


def device_normals_reference(seed, iteration, row, agent):
    """The standard normal the device draws for (seed, iteration, row, agent); arrays broadcast."""
    seed = int(seed)
    row, agent = np.asarray(row, dtype=np.uint64), np.asarray(agent, dtype=np.uint64)
    c = philox4x32_10((row, agent, np.full_like(row, iteration), np.zeros_like(row)), (seed & 0xFFFFFFFF, seed >> 32))
    a = ((c[0] << np.uint64(32)) | c[1]) >> np.uint64(11)
    b = ((c[2] << np.uint64(32)) | c[3]) >> np.uint64(11)
    u1 = (a + np.uint64(1)).astype(np.float64) * 2.0 ** -53
    u2 = b.astype(np.float64) * 2.0 ** -53
    return np.sqrt(-2.0 * np.log(u1)) * np.cos(2.0 * np.pi * u2)


def test_philox_restatement_reproduces_the_published_known_answers():
    kat = [((0, 0, 0, 0), (0, 0), (0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8)),
           ((0xffffffff,) * 4, (0xffffffff,) * 2, (0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd)),
           ((0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344), (0xa4093822, 0x299f31d0),
            (0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1))]
    for c, k, want in kat:
        assert tuple(int(v) for v in philox4x32_10(c, k)) == want


def test_reference_normals_are_standard_normal_and_keyed_by_every_counter_word():
    rows = np.arange(200_000, dtype=np.uint64)
    x = device_normals_reference(2 ** 64 - 1, 3, rows, 0)
    n = x.size
    assert abs(x.mean()) <= 5 / np.sqrt(n) and abs(x.var() - 1) <= 6 * np.sqrt(2 / n)
    assert np.all(np.isfinite(x))
    others = [device_normals_reference(2 ** 64 - 2, 3, rows, 0), device_normals_reference(2 ** 64 - 1, 4, rows, 0),
              device_normals_reference(2 ** 64 - 1, 3, rows, 1), device_normals_reference(2 ** 64 - 1, 3, rows + 1, 0)]
    for y in others:
        assert abs(float(np.corrcoef(x, y)[0, 1])) <= 6 / np.sqrt(n)
