"""The CPU reference of the device generator (oracle/device_rng.py) on its own: Philox4x32-10 against the Random123
known-answer vectors, and the properties the GPU comparisons in test_device_rng.py rely on (no GPU needed)."""
import numpy as np
import pytest

from oracle import device_rng as R

# Random123 kat_vectors, philox4x32_10: counter, key, result
KAT = [
    ((0x00000000, 0x00000000, 0x00000000, 0x00000000), (0x00000000, 0x00000000),
     (0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8)),
    ((0xffffffff, 0xffffffff, 0xffffffff, 0xffffffff), (0xffffffff, 0xffffffff),
     (0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd)),
    ((0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344), (0xa4093822, 0x299f31d0),
     (0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1)),
]


@pytest.mark.parametrize("ctr,key,want", KAT, ids=["zeros", "ones", "pi"])
def test_philox_known_answers(ctr, key, want):
    got = R.philox4x32_10(*ctr, *key)
    assert tuple(int(w) for w in got) == want
    # vectorised: the same call at every position of a batch
    batch = R.philox4x32_10(*(np.full(5, c, dtype=np.uint32) for c in ctr), *key)
    assert all((b == w).all() and b.dtype == np.uint32 for b, w in zip(batch, want))


def test_split_of_signed_and_unsigned_64bit_values():
    assert R.split64(0x9E3779B97F4A7C15) == (0x7F4A7C15, 0x9E3779B9)
    assert R.split64(0x9E3779B97F4A7C15 - (1 << 64)) == (0x7F4A7C15, 0x9E3779B9)      # as the device stores it
    assert R.split64(-1) == (0xFFFFFFFF, 0xFFFFFFFF) and R.split64(1 << 32) == (0, 1)


def test_uniforms_are_exact_top_24_bits():
    w = np.array([0, 0xFF, 0x100, 0xFFFFFFFF, 0x80000000], dtype=np.uint32)
    u = R.uniforms(w)
    assert u.dtype == np.float32
    assert u.tolist() == [0.0, 0.0, 2.0 ** -24, 1.0 - 2.0 ** -24, 0.5]


def test_box_muller_word_roles():
    """Radius from words x / z, angle from words y / w, output order (r0 cos, r0 sin, r1 cos, r1 sin)."""
    top = 0xFFFFFF00                              # (top 24 bits + 1) * 2^-24 = 1: radius 0
    half = 0x7FFFFF00                             # u = 0.5
    quarter = 0x40000000                          # angle pi / 2
    z = R.normals4(np.uint32(half), np.uint32(0), np.uint32(top), np.uint32(quarter))
    r = np.sqrt(-2.0 * np.log(0.5))
    np.testing.assert_allclose(z, [r, 0.0, 0.0, 0.0], atol=1e-7)
    z = R.normals4(np.uint32(top), np.uint32(0), np.uint32(half), np.uint32(quarter))
    np.testing.assert_allclose(z, [0.0, 0.0, 0.0, r], atol=1e-6)


def test_env_draws_follow_the_slot_layout():
    key, step, n = 0xC0FFEE0012345678 | (1 << 63), (1 << 32) + 5, 37
    for ndof, nobs in ((10, 41), (12, 47), (18, 65)):
        f = R.env_draws(key, step, n, ndof, nobs)
        shapes = dict(u_delay=(n, 1), z_action=(n, ndof), u_cmd=(n, 3), u_push=(n, 5), u_reset=(n, ndof + 5), z_obs=(n, nobs))
        for name, shape in shapes.items():
            assert tuple(getattr(f, name).shape) == shape, name
        # the root-xy / command part of the reset draws continues the dof jitter's words (rng_uniforms with first = NDOF)
        words = R.philox4x32_10(np.arange(n)[:, None], R.SLOT_U_RESET + np.arange(8)[None, :], *R.split64(step), *R.split64(key))
        flat = R.uniforms(np.stack(words, axis=-1)).reshape(n, -1)
        np.testing.assert_array_equal(f.u_reset.numpy(), flat[:, :ndof + 5])
        np.testing.assert_array_equal(f.u_reset.numpy()[:, ndof:], flat[:, ndof:ndof + 5])
        # distinct slots, distinct envs: no two blocks of draws share a Philox call
        assert not np.array_equal(f.u_cmd.numpy(), f.u_push.numpy()[:, :3])
        assert len(np.unique(f.z_obs.numpy()[:, 0])) == n
    # the counter's upper word and the key's upper word both matter
    base = R.env_draws(key, step, n, 10, 41).z_obs.numpy()
    assert not np.array_equal(base, R.env_draws(key, step & 0xFFFFFFFF, n, 10, 41).z_obs.numpy())
    assert not np.array_equal(base, R.env_draws(key & 0xFFFFFFFF, step, n, 10, 41).z_obs.numpy())
    with pytest.raises(ValueError):
        R.env_draws(key, step, n, 25, 41)


def test_ppo_normals_are_standard_normal_and_prefix_stable():
    z = R.ppo_normals(0x9E3779B97F4A7C15, 3, 200003)
    assert z.dtype == np.float32 and z.shape == (200003,) and np.isfinite(z).all()
    assert abs(z.mean()) < 0.01 and abs(z.std() - 1.0) < 0.01 and abs((z.astype(np.float64) ** 4).mean() - 3.0) < 0.1
    np.testing.assert_array_equal(R.ppo_normals(0x9E3779B97F4A7C15, 3, 5), z[:5])
    assert not np.array_equal(R.ppo_normals(0x9E3779B97F4A7C15, 4, 5), z[:5])
    assert not np.array_equal(R.ppo_normals(0x9E3779B97F4A7C15, 3 + (1 << 32), 5), z[:5])
