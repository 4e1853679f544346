// Scramble with the action stream generated ON the device (SURVEY 8d C2: "full run may generate on device from the same
// counter-based stream"): no action bytes cross PCIe or HBM, 20 B per cube leave the chip.
//
// The stream is Philox4x32-10 (Salmon, Moraes, Dror, Shaw: "Parallel random numbers: as easy as 1, 2, 3", SC'11 -- the
// counter-based generator of Random123 and cuRAND), key = the 64-bit seed, counter = (block j, 0, cube id lo, cube id hi):
// every cube owns one Philox subsequence, so the result for cube c does not depend on how cubes are sharded over launches,
// streams or GPUs.  One 32-bit output word gives THREE moves: t = (word * 1728) >> 32 is uniform on [0, 12^3) (bias
// < 1728 / 2^32 = 4e-7) and its base-12 digits are three independent uniform action indices -- each move uniform over 6 faces
// x 2 directions as in the reference's draw (cube.py:208-209: randint(6) faces, randint(2) directions):
//     move 3q     = t_q / 144        move 3q + 1 = t_q / 12 % 12        move 3q + 2 = t_q % 12
//     t_q = word (q % 4) of Philox block (q / 4) of the cube's subsequence;  a sequence of depth d uses moves 0 .. d-1
// (so a shorter scramble with the same seed is a prefix of a longer one).  t_q is used as it is as the row index of the
// 3-move table of rb_scramble_macro.cuh (the later move is the low digit there too).  k_seeded_actions writes the same
// stream out as action bytes: parity is checked by replaying those bytes on the CPU oracle (tests/test_gpu_seeded.py), and
// oracle/cube_oracle.py restates the generator in numpy (pinned on the Random123 known-answer vectors).
//
// The kernel is the slot-major macro-move kernel without its action buffers: thread per cube, 32 consecutive cubes per
// warp, table rows from 4 copies in shared memory (Rows3), results staged per warp and written as 640 contiguous bytes.
#pragma once
#include "rb_scramble_macro.cuh"

namespace rbs {

struct PhiloxKeys {                              // the ten round keys of one seed (key schedule: += golden-ratio constants)
	uint32_t k0[10], k1[10];
};

static inline PhiloxKeys philox_keys(uint64_t seed) {
	PhiloxKeys k;
	uint32_t a = (uint32_t)seed, b = (uint32_t)(seed >> 32);
	for (int r = 0; r < 10; ++r) {
		k.k0[r] = a; k.k1[r] = b;
		a += 0x9E3779B9u; b += 0xBB67AE85u;
	}
	return k;
}

__device__ __forceinline__ void philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, const PhiloxKeys& k, uint32_t (&x)[4]) {
#pragma unroll
	for (int r = 0; r < 10; ++r) {
		const uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
		const uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
		c0 = hi1 ^ c1 ^ k.k0[r];
		c2 = hi0 ^ c3 ^ k.k1[r];
		c1 = lo1;
		c3 = lo0;
	}
	x[0] = c0; x[1] = c1; x[2] = c2; x[3] = c3;
}

__device__ __forceinline__ uint32_t triple_of(uint32_t word) { return __umulhi(word, 1728u); }

// The action bytes of the stream: actions[i][m] for cubes first_cube .. first_cube + n - 1 (thread per cube and Philox block).
__global__ void __launch_bounds__(256)
k_seeded_actions(PhiloxKeys keys, uint64_t first_cube, uint8_t* __restrict__ actions, int64_t n, int depth, int blocks_per_cube) {
	const int64_t stride = (int64_t)gridDim.x * blockDim.x, total = n * blocks_per_cube;
	for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += stride) {
		const int64_t i = t / blocks_per_cube;
		const int j = (int)(t - i * blocks_per_cube);
		const uint64_t cube = first_cube + (uint64_t)i;
		uint32_t x[4];
		philox4x32_10((uint32_t)j, 0u, (uint32_t)cube, (uint32_t)(cube >> 32), keys, x);
		uint8_t* row = actions + i * depth;
#pragma unroll
		for (int k = 0; k < 4; ++k) {
			const uint32_t tr = triple_of(x[k]);
			const int m = 3 * (4 * j + k);
			if (m < depth) row[m] = (uint8_t)(tr / 144u);
			if (m + 1 < depth) row[m + 1] = (uint8_t)(tr / 12u % 12u);
			if (m + 2 < depth) row[m + 2] = (uint8_t)(tr % 12u);
		}
	}
}

constexpr int kSeedStage = 640;                  // result staging per warp: 32 cubes x 20 B
constexpr int kSeedSmem = kTableBytes3 + kMaxThreads / 32 * kSeedStage;

__global__ void __launch_bounds__(kMaxThreads, 1)
k_scramble_seeded(PhiloxKeys keys, uint64_t first_cube, int8_t* __restrict__ out, int64_t n, int depth, int out_pitch, uint32_t p2_stride,
                  uint32_t n_warps) {
	// n_warps <= blockDim.x / 32 warps work (small n is spread over all SMs); the whole CTA stages the table
	extern __shared__ __align__(128) uint8_t smem[];
	uint8_t* table = smem;                                              // [P1: 4 copies of the 16-byte part | P2 | 2-move tail | staging]
	const uint32_t lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
	uint32_t* stage = reinterpret_cast<uint32_t*>(smem + kTableBytes3 + wib * kSeedStage);
	const Rows3<false> t(table, lane, 0u, p2_stride);

	stage_table3(table);
	__syncthreads();
	if (wib >= n_warps) return;

	const int Q = depth / 3, rem = depth - 3 * Q;                       // Q whole triples, rem trailing moves (from triple Q)
	const int n_words = Q + (rem ? 1 : 0), n_blocks = (n_words + 3) >> 2;
	const int64_t n_chunks = (n + 31) / 32, stride = (int64_t)gridDim.x * n_warps;
	for (int64_t chunk = (int64_t)blockIdx.x * n_warps + wib; chunk < n_chunks; chunk += stride) {
		const int cnt = (int)min((int64_t)32, n - chunk * 32);
		uint32_t res[5] = {0u, 0u, 0u, 0u, 0u};
		if ((int)lane < cnt) {
			const uint64_t cube = first_cube + (uint64_t)(chunk * 32 + lane);
			const uint32_t c2 = (uint32_t)cube, c3 = (uint32_t)(cube >> 32);
			Slots s{0x60402000u, 0xe0c0a080u, 0x03020100u, 0x07060504u, 0x0b0a0908u};
			// as in k_scramble_macro3 the INVERSE moves are multiplied in REVERSE order (the tables are laid out for it): the last
			// Philox block first, inside a block the last triple first, before everything the trailing rem moves
			{                                                                    // the last block: may be partial, may hold the trailing moves
				const int j = n_blocks - 1;
				uint32_t x[4];
				if (j >= 0) philox4x32_10((uint32_t)j, 0u, c2, c3, keys, x);
#pragma unroll
				for (int k = 3; k >= 0; --k) {
					const int q = 4 * j + k;
					if (j < 0 || q > Q || (q == Q && rem == 0)) continue;
					const uint32_t tr = triple_of(x[k]);
					if (q == Q) {                                                  // 1 or 2 moves: 2-move table, index = later + 13 * earlier (12 = none)
						const uint32_t m0 = tr / 144u, m1 = tr / 12u % 12u;
						t.apply_tail(s, rem == 1 ? m0 + 13u * 12u : m1 + 13u * m0);
					} else {
						t.apply3(s, tr);
					}
				}
			}
			int since = 1;                                                       // blocks applied since the last fold: <= 8 rows (+ the tail row) between folds
			for (int j = n_blocks - 2; j >= 0; --j) {
				uint32_t x[4];
				philox4x32_10((uint32_t)j, 0u, c2, c3, keys, x);
				t.apply3(s, triple_of(x[3])); t.apply3(s, triple_of(x[2])); t.apply3(s, triple_of(x[1])); t.apply3(s, triple_of(x[0]));
				if (++since == 2) { fold(s); since = 0; }
			}
			fold(s);
			cubie_major(s, res);
		}
		if ((int)lane < cnt) {
#pragma unroll
			for (int k = 0; k < 5; ++k) stage[lane * 5 + k] = res[k];
		}
		__syncwarp();
		uint32_t outw[5];
#pragma unroll
		for (int k = 0; k < 5; ++k) {
			const int j = lane + 32 * k;
			outw[k] = j < cnt * 5 ? stage[j] : 0u;
		}
		__syncwarp();
		store_results<32>(out, chunk * 32, out_pitch, cnt, lane, outw);
	}
}

static int launch_seeded(uint64_t seed, uint64_t first_cube, int8_t* out, int64_t n, int depth, cudaStream_t st, int out_pitch) {
	int rc = ensure_device();
	if (rc != RB_OK) return rc;
	const int64_t chunks = (n + 31) / 32;
	int64_t warps = (chunks + RB_NUM_SMS - 1) / RB_NUM_SMS;                 // small n: one chunk per warp on as many SMs as possible
	if (warps > kMaxThreads / 32) warps = kMaxThreads / 32;
	const int64_t ctas = (chunks + warps - 1) / warps;
	const int grid = (int)(ctas < RB_NUM_SMS ? ctas : RB_NUM_SMS);
	k_scramble_seeded<<<grid, kMaxThreads, kSeedSmem, st>>>(philox_keys(seed), first_cube, out, n, depth, out_pitch, 4u, (uint32_t)warps);
	RB_LAUNCHED("scramble_seeded_2024");
	return RB_OK;
}

static int launch_seeded_actions(uint64_t seed, uint64_t first_cube, uint8_t* actions, int64_t n, int depth, cudaStream_t st) {
	const int blocks_per_cube = ((depth + 2) / 3 + 3) / 4;
	k_seeded_actions<<<rb_grid(n * blocks_per_cube, 256, 8), 256, 0, st>>>(philox_keys(seed), first_cube, actions, n, depth, blocks_per_cube);
	RB_LAUNCHED("seeded_actions");
	return RB_OK;
}

}  // namespace rbs
