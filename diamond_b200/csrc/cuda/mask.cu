// mask.cu -- dmnd_block_mask / dmnd_block_mask_fetch: launch sequence of the masking kernels (mask_kernels.cuh).
#include "ctx.cuh"
#include "mask_kernels.cuh"
#include <cub/cub.cuh>
#include <algorithm>

namespace dmnd_cuda {

int block_mask_impl(dmnd_ctx* ctx, dmnd_block* b, int algo, uint32_t s_begin, uint32_t s_end, uint64_t* n_hard) {
	if (s_begin > s_end || s_end > b->nseq) { set_error("dmnd_block_mask: bad sequence range"); return 1; }
	if (algo & ~(DMND_MASK_TANTAN | DMND_MASK_MOTIF)) { set_error("dmnd_block_mask: unknown masking algorithm"); return 1; }
	cudaStream_t st = ctx->stream;
	ctx->mask_n = 0;
	b->content_epoch = new_content_epoch();  // letters / soft table change: a seed index cached on the block is stale
	if (n_hard) *n_hard = 0;
	const size_t p_begin = (size_t)b->h_limits[s_begin], p_end = (size_t)b->h_limits[s_end];
	const size_t nlet = p_end - p_begin, nseq = s_end - s_begin;
	if (nseq == 0 || nlet == 0) { if (algo & DMND_MASK_MOTIF) b->has_soft = true; return 0; }
	if (nlet >= 0x7fffffffull) { set_error("dmnd_block_mask: ranges of 2 G letters or more are not supported (mask the block in several ranges)"); return 1; }
	const size_t w_begin = p_begin >> 5, w_end = ((p_end - 1) >> 5) + 1;
	if (ctx->b_mask_cov.ensure(((b->raw_len >> 5) + 4) * 4) || ctx->b_counters.ensure(96 * sizeof(unsigned long long))) return 1;
	uint32_t* d_bits = ctx->b_mask_cov.as<uint32_t>();
	unsigned long long* d_cnt = ctx->b_counters.as<unsigned long long>();
	PhaseTimer timer(ctx, PH_SEED);
	if (algo & DMND_MASK_TANTAN) {
		if (ctx->b_mask_pb.ensure(nlet * 4) || ctx->b_mask_scale.ensure(((nlet >> 4) + nseq + 2) * 4)) return 1;
		DMND_CUDA_CHECK(cudaMemsetAsync(d_bits + w_begin, 0, (w_end - w_begin) * 4, st));
		DMND_CUDA_CHECK(cudaMemsetAsync(d_cnt, 0, 6 * sizeof(unsigned long long), st));
		// longest-first order of the range's sequences: the four sequences of a warp run in lock step (mask_kernels.cuh), so
		// neighbours in the order should have the same length; long sequences also start first
		if (ctx->b_keys.ensure(nseq * 4) || ctx->b_keys2.ensure(nseq * 4) || ctx->b_vals.ensure(nseq * 4) || ctx->b_vals2.ensure(nseq * 4)) return 1;
		seq_len_kernel<<<(unsigned)((nseq + 255) / 256), 256, 0, st>>>(b->limits, s_begin, (uint32_t)nseq, ctx->b_keys.as<uint32_t>(), ctx->b_vals.as<uint32_t>());
		{
			size_t tmp = 0;
			cub::DeviceRadixSort::SortPairsDescending(nullptr, tmp, ctx->b_keys.as<uint32_t>(), ctx->b_keys2.as<uint32_t>(), ctx->b_vals.as<uint32_t>(), ctx->b_vals2.as<uint32_t>(), (int)nseq, 0, 32, st);
			if (ctx->b_cub.ensure(tmp)) return 1;
			DMND_CUDA_CHECK(cub::DeviceRadixSort::SortPairsDescending(ctx->b_cub.p, tmp, ctx->b_keys.as<uint32_t>(), ctx->b_keys2.as<uint32_t>(), ctx->b_vals.as<uint32_t>(), ctx->b_vals2.as<uint32_t>(), (int)nseq, 0, 32, st));
		}
		// forward pass of everything; it also decides which sequences need the backward pass at all (mask_kernels.cuh); the
		// compacted longest-first list of those goes through the backward kernel, whose grid covers the worst case
		if (ctx->b_mask_zinv.ensure(nseq * 4) || ctx->b_mask_need.ensure(nseq + 16)) return 1;
		int* d_nneed = (int*)(d_cnt + 2);
		tantan_forward_kernel<<<(unsigned)((nseq + 15) / 16), 128, 0, st>>>(b->letters, b->limits, ctx->b_vals2.as<uint32_t>(), (uint32_t)nseq, ctx->d_params,
			ctx->b_mask_pb.as<float>(), ctx->b_mask_scale.as<float>(), (int64_t)p_begin, s_begin, ctx->b_mask_zinv.as<float>(), ctx->b_mask_need.as<uint8_t>());
		{
			size_t tmp = 0;
			cub::DeviceSelect::Flagged(nullptr, tmp, ctx->b_vals2.as<uint32_t>(), ctx->b_mask_need.as<uint8_t>(), ctx->b_keys2.as<uint32_t>(), d_nneed, (int)nseq, st);
			if (ctx->b_cub.ensure(tmp)) return 1;
			DMND_CUDA_CHECK(cub::DeviceSelect::Flagged(ctx->b_cub.p, tmp, ctx->b_vals2.as<uint32_t>(), ctx->b_mask_need.as<uint8_t>(), ctx->b_keys2.as<uint32_t>(), d_nneed, (int)nseq, st));
		}
		tantan_backward_kernel<<<(unsigned)((nseq + 15) / 16), 128, 0, st>>>(b->letters, b->limits, ctx->b_keys2.as<uint32_t>(), d_nneed, ctx->d_params,
			ctx->b_mask_pb.as<float>(), ctx->b_mask_scale.as<float>(), (int64_t)p_begin, s_begin, ctx->b_mask_zinv.as<float>(), d_bits);
		ctx->launches += 8;
		popc_kernel<<<(unsigned)((w_end - w_begin + 255) / 256), 256, 0, st>>>(d_bits, w_begin, w_end, d_cnt);
		ctx->launches += 2;
		DMND_CUDA_CHECK(cudaGetLastError());
		DMND_CUDA_CHECK(cudaMemcpyAsync(ctx->h_pinned, d_cnt, sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
		DMND_CUDA_CHECK(stream_wait(ctx, st));
		const unsigned long long n = *(const unsigned long long*)ctx->h_pinned;
		if (n) {
			// ascending offsets of the set bits: stream compaction of a counting sequence (no sort needed)
			if (ctx->b_mask_pos.ensure((size_t)n * 8)) return 1;
			cub::CountingInputIterator<uint64_t> first((uint64_t)p_begin);
			size_t tmp = 0;
			int* d_num = (int*)(d_cnt + 4);
			cub::DeviceSelect::If(nullptr, tmp, first, ctx->b_mask_pos.as<uint64_t>(), d_num, (int)nlet, BitSet{ d_bits }, st);
			if (ctx->b_cub.ensure(tmp)) return 1;
			DMND_CUDA_CHECK(cub::DeviceSelect::If(ctx->b_cub.p, tmp, first, ctx->b_mask_pos.as<uint64_t>(), d_num, (int)nlet, BitSet{ d_bits }, st));
			ctx->launches += 2;
		}
		ctx->mask_n = n;
		if (n_hard) *n_hard = n;
	}
	if (algo & DMND_MASK_MOTIF) {
		if (ctx->b_mask_flag.ensure(((size_t)b->nseq / 32 + 2) * 4) || ctx->b_mask_seqs.ensure((nseq + 1) * 4) || ctx->b_mask_pos2.ensure(DMND_MOTIF_COUNT * 8)) return 1;
		uint32_t* d_flag = ctx->b_mask_flag.as<uint32_t>();
		unsigned int* d_nlist = (unsigned int*)(d_cnt + 3);
		DMND_CUDA_CHECK(cudaMemcpyAsync(ctx->b_mask_pos2.p, DMND_MOTIF_CODES, DMND_MOTIF_COUNT * 8, cudaMemcpyHostToDevice, st));
		DMND_CUDA_CHECK(cudaMemsetAsync(d_bits + w_begin, 0, (w_end - w_begin + 1) * 4, st));
		DMND_CUDA_CHECK(cudaMemsetAsync(d_flag, 0, ((size_t)b->nseq / 32 + 2) * 4, st));
		DMND_CUDA_CHECK(cudaMemsetAsync(d_nlist, 0, sizeof(unsigned int), st));
		clear_bits_kernel<<<(unsigned)((w_end - w_begin + 255) / 256), 256, 0, st>>>(b->soft, p_begin, p_end);
		motif_hit_kernel<<<(unsigned)((nlet + MOTIF_TILE - 1) / MOTIF_TILE), 256, 0, st>>>(b->letters, b->raw_len, p_begin, p_end, ctx->b_mask_pos2.as<uint64_t>(), d_bits,
			b->limits, s_begin, s_end, d_flag, ctx->b_mask_seqs.as<uint32_t>(), d_nlist);
		// sequences with a hit are rare; the grid covers the worst case and surplus threads leave at once
		motif_apply_kernel<<<(unsigned)((nseq + 127) / 128), 128, 0, st>>>(b->limits, ctx->b_mask_seqs.as<uint32_t>(), d_nlist, d_bits, b->soft, ctx->params.max_motif_len);
		ctx->launches += 3;
		DMND_CUDA_CHECK(cudaGetLastError());
		b->has_soft = true;
	}
	timer.stop();
	return 0;
}

int block_mask_fetch_impl(dmnd_ctx* ctx, uint64_t* positions, size_t cap) {
	if (cap < ctx->mask_n) { set_error("dmnd_block_mask_fetch: buffer too small"); return 1; }
	if (ctx->mask_n == 0) return 0;
	PhaseTimer t(ctx, PH_D2H);
	DMND_CUDA_CHECK(cudaMemcpyAsync(positions, ctx->b_mask_pos.p, (size_t)ctx->mask_n * 8, cudaMemcpyDeviceToHost, ctx->stream));
	t.stop();
	ctx->d2h_bytes += (size_t)ctx->mask_n * 8;
	return 0;
}

}  // namespace dmnd_cuda
