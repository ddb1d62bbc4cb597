// comm.cu -- the one collective of the path (SURVEY 8e): the packed reference block travels once from one rank to all others
// over NVLink, straight from the root's resident block into a freshly allocated block on every other rank (no host bounce).
// One process per GPU; every rank calls with its own context.  NCCL is loaded at run time (dlopen) so that the library has no
// link-time dependency on it: DMND_NCCL_LIB, then libnccl.so.2 / libnccl.so on the loader path.  The 128-byte unique id is
// exchanged by the caller (torch.distributed, MPI, a file): dmnd_comm_unique_id on rank 0, dmnd_comm_init on every rank.
#include "ctx.cuh"
#include <dlfcn.h>
#include <cstdlib>
#include <cstring>

namespace {

typedef struct { char internal[128]; } nccl_uid;
typedef void* nccl_comm;
struct Nccl {
	void* h = nullptr;
	int (*GetUniqueId)(nccl_uid*) = nullptr;
	int (*CommInitRank)(nccl_comm*, int, nccl_uid, int) = nullptr;
	int (*Broadcast)(const void*, void*, size_t, int /*ncclDataType_t*/, int, nccl_comm, cudaStream_t) = nullptr;
	int (*CommDestroy)(nccl_comm) = nullptr;
	const char* (*GetErrorString)(int) = nullptr;
	bool load() {
		if (h) return true;
		const char* names[] = { getenv("DMND_NCCL_LIB"), "libnccl.so.2", "libnccl.so" };
		for (const char* n : names) {
			if (!n || !*n) continue;
			h = dlopen(n, RTLD_NOW | RTLD_GLOBAL);
			if (h) break;
		}
		if (!h) return false;
		GetUniqueId = (int (*)(nccl_uid*))dlsym(h, "ncclGetUniqueId");
		CommInitRank = (int (*)(nccl_comm*, int, nccl_uid, int))dlsym(h, "ncclCommInitRank");
		Broadcast = (int (*)(const void*, void*, size_t, int, int, nccl_comm, cudaStream_t))dlsym(h, "ncclBroadcast");
		CommDestroy = (int (*)(nccl_comm))dlsym(h, "ncclCommDestroy");
		GetErrorString = (const char* (*)(int))dlsym(h, "ncclGetErrorString");
		return GetUniqueId && CommInitRank && Broadcast && CommDestroy;
	}
};
Nccl g_nccl;
constexpr int NCCL_INT8 = 0, NCCL_INT64 = 4;  // ncclDataType_t

int nccl_fail(const char* what, int rc) {
	dmnd_cuda::set_error(std::string(what) + ": " + (g_nccl.GetErrorString ? g_nccl.GetErrorString(rc) : "NCCL error") + " (" + std::to_string(rc) + ")");
	return 1;
}

}  // namespace

extern "C" {

int dmnd_comm_unique_id(void* out128) {
	if (!g_nccl.load()) { dmnd_cuda::set_error("dmnd_comm_unique_id: cannot load NCCL (set DMND_NCCL_LIB to libnccl.so.2)"); return 1; }
	nccl_uid id;
	if (int rc = g_nccl.GetUniqueId(&id)) return nccl_fail("ncclGetUniqueId", rc);
	std::memcpy(out128, &id, sizeof id);
	return 0;
}

int dmnd_comm_init(dmnd_ctx* ctx, int rank, int nranks, const void* unique_id128) {
	DMND_CUDA_CHECK(cudaSetDevice(ctx->device));
	if (!g_nccl.load()) { dmnd_cuda::set_error("dmnd_comm_init: cannot load NCCL (set DMND_NCCL_LIB to libnccl.so.2)"); return 1; }
	if (rank < 0 || rank >= nranks) { dmnd_cuda::set_error("dmnd_comm_init: bad rank"); return 1; }
	if (ctx->comm) { g_nccl.CommDestroy((nccl_comm)ctx->comm); ctx->comm = nullptr; }
	nccl_uid id;
	std::memcpy(&id, unique_id128, sizeof id);
	nccl_comm c = nullptr;
	if (int rc = g_nccl.CommInitRank(&c, nranks, id, rank)) return nccl_fail("ncclCommInitRank", rc);
	ctx->comm = c; ctx->comm_rank = rank; ctx->comm_size = nranks;
	return 0;
}

void dmnd_comm_destroy(dmnd_ctx* ctx) {
	if (ctx->comm && g_nccl.CommDestroy) g_nccl.CommDestroy((nccl_comm)ctx->comm);
	ctx->comm = nullptr;
}

int dmnd_block_broadcast(dmnd_ctx* ctx, int root, dmnd_block* src, dmnd_block** out) {
	DMND_CUDA_CHECK(cudaSetDevice(ctx->device));
	if (!ctx->comm) { dmnd_cuda::set_error("dmnd_block_broadcast: dmnd_comm_init has not been called on this context"); return 1; }
	const bool is_root = ctx->comm_rank == root;
	if (is_root && !src) { dmnd_cuda::set_error("dmnd_block_broadcast: the root rank must pass its resident block"); return 1; }
	nccl_comm comm = (nccl_comm)ctx->comm;
	cudaStream_t st = ctx->stream;
	// ---- header: raw length, sequence count, masking state
	if (ctx->b_counters.ensure(64)) return 1;
	int64_t hdr[4] = { 0, 0, 0, 0 };
	if (is_root) { hdr[0] = (int64_t)src->raw_len; hdr[1] = (int64_t)src->nseq; hdr[2] = src->has_soft ? 1 : 0; }
	int64_t* d_hdr = ctx->b_counters.as<int64_t>();
	if (is_root) DMND_CUDA_CHECK(cudaMemcpyAsync(d_hdr, hdr, sizeof hdr, cudaMemcpyHostToDevice, st));
	if (int rc = g_nccl.Broadcast(d_hdr, d_hdr, 4, NCCL_INT64, root, comm, st)) return nccl_fail("ncclBroadcast(header)", rc);
	DMND_CUDA_CHECK(cudaMemcpyAsync(hdr, d_hdr, sizeof hdr, cudaMemcpyDeviceToHost, st));
	DMND_CUDA_CHECK(dmnd_cuda::stream_wait(ctx, st));
	const size_t raw_len = (size_t)hdr[0];
	const uint32_t nseq = (uint32_t)hdr[1];
	dmnd_block* b = src;
	if (!is_root) {
		if (dmnd_block_alloc_empty(ctx, raw_len, nseq, &b)) return 1;
	}
	// ---- letters (incl. hard masking done on the root), limits, the per-letter soft-masking table, the bias array
	const size_t padded = (raw_len + 63) & ~(size_t)63;
	if (int rc = g_nccl.Broadcast(b->letters, b->letters, padded + 64, NCCL_INT8, root, comm, st)) return nccl_fail("ncclBroadcast(letters)", rc);
	if (int rc = g_nccl.Broadcast(b->limits, b->limits, (size_t)nseq + 1, NCCL_INT64, root, comm, st)) return nccl_fail("ncclBroadcast(limits)", rc);
	if (int rc = g_nccl.Broadcast(b->soft, b->soft, padded / 8 + 16, NCCL_INT8, root, comm, st)) return nccl_fail("ncclBroadcast(soft)", rc);
	if (int rc = g_nccl.Broadcast(b->bias, b->bias, padded + 64, NCCL_INT8, root, comm, st)) return nccl_fail("ncclBroadcast(bias)", rc);
	if (!is_root) {
		b->has_soft = hdr[2] != 0;
		b->content_epoch = dmnd_cuda::new_content_epoch();
		b->h_limits.resize((size_t)nseq + 1);
		DMND_CUDA_CHECK(cudaMemcpyAsync(b->h_limits.data(), b->limits, sizeof(int64_t) * ((size_t)nseq + 1), cudaMemcpyDeviceToHost, st));
	}
	DMND_CUDA_CHECK(dmnd_cuda::stream_wait(ctx, st));
	ctx->launches += 5;
	*out = b;
	return 0;
}

}  // extern "C"
