// rt_checksum.h -- the 64-bit multiply-xorshift checksum of the library's files (flattened scenes, accumulator
// checkpoints) and of the scene fingerprint (not installed).
#pragma once
#include <stdint.h>
#include <stddef.h>
#include <string.h>

#if defined(__CUDACC__)
#define RT_CHECKSUM_FN __host__ __device__
#else
#define RT_CHECKSUM_FN
#endif

// Over 8-byte words (tail bytes zero-padded), then the length: catches truncation and bit rot, runs at memory speed.
struct RtChecksum
{
	uint64_t h = 0x9E3779B97F4A7C15ull;
	RT_CHECKSUM_FN void Add(const void* data, size_t bytes)
	{
		const unsigned char* p = (const unsigned char*)data;
		size_t i = 0;
		for (; i + 8 <= bytes; i += 8) { uint64_t w; memcpy(&w, p + i, 8); Mix(w); }
		if (i < bytes) { uint64_t w = 0; memcpy(&w, p + i, bytes - i); Mix(w); }
		Mix((uint64_t)bytes);
	}
	RT_CHECKSUM_FN void Mix(uint64_t w) { h ^= w; h *= 0xD6E8FEB86659FD93ull; h ^= h >> 32; }
};
