// conv_bank.cuh -- a convolver bank spread over several GPUs of one box (include/neo_b200.h: neo_b200_bank_*).
//
// The reference has one private convolver per channel (src/neo/convolution/uniform_partitioned_convolver.hpp:28-34, one instance per
// channel in extra/cli/src/convolver.cpp:37-40), so channels shard with no communication; and the delay line is linear in the input
// (fdl_index.hpp:24-36 pairs partition p with the spectrum of p blocks ago), so the partitions of one long filter shard too, at the
// price of ONE sum of partial spectra per block. The bank lays its N = Gc x Gp ranks out in two dimensions:
//
//   rank = gc * Gp + gp      gc: channel group   -- channels [gc*C/Gc, (gc+1)*C/Gc) (matrix topology: OUTPUT channels)
//                            gp: partition shard -- partitions [lo_gp, hi_gp) of every filter of the group
//
// Per step (one call of T blocks) and rank:
//   1. input rows: every rank brings in only its own 1/N of the rows (host -> device over its own PCIe link, or device -> device),
//      then the ranks that need the same rows (the Gp shards of a group; everyone in the matrix topology) exchange them over NVLink
//      (all-gather) into a ring of time-domain input slots;
//   2. forward: window + r2c + delay line + spectral MAC of the rank's partitions -> PARTIAL spectra [group channels][T][B]. In frame
//      mode shard gp > 0 reads the ring slot of lo_gp/T frames ago instead of keeping a deeper ring of frame spectra
//      (neo_b200_conv_config::input_delayed): its newest frame spectrum then comes from registers exactly as on shard 0;
//   3. reduction + inverse: the Gp partial spectra of a group are summed and rank (gc, gp) runs c2r + overlap handling for its
//      1/Gp of the group's channels;
//   4. output rows: each rank returns its own 1/N of the rows.
//
// Two transports for steps 1 and 3:
//   peer : every rank lives in this process (neo_b200_bank_create with devices[]). Step 1 pushes rows with peer copies; step 3 is
//          FUSED into the c2r kernel, which loads the Gp partial spectra through peer-mapped pointers (conv_c2r_sum_io) -- no
//          separate reduction pass, no extra HBM round trip. Ordering is by CUDA events across the devices' streams. The same device
//          may be named several times (tests on a one-GPU box run the whole multi-rank logic that way).
//   nccl : one rank per process (neo_b200_bank_create_rank; torchrun / MPI launchers). Step 1 is ncclAllGather, step 3
//          ncclReduceScatter (sum) followed by the plain c2r kernel. NCCL is loaded at run time (libnccl.so.2), so the library has
//          no link-time dependency on it and single-GPU users never touch it.
//
// Steps are software-pipelined: submit() only enqueues (four streams per rank: input, forward, reduction, output; every buffer a
// step writes is double-buffered), so the input copy of step i+1 and the output copy of step i-1 overlap the kernels of step i.
#pragma once

#include <dlfcn.h>

#include <array>
#include <deque>

namespace neo_b200 {
namespace {

// ---- NCCL, resolved at run time -------------------------------------------------------------------------------------------------------
// Minimal declarations of the stable NCCL 2 ABI (nccl.h): opaque communicator, 128-byte unique id, result code 0 = success.
struct nccl_api
{
    using comm_t = void*;
    struct unique_id
    {
        char internal[128];
    };
    static constexpr int k_float32 = 7, k_float64 = 8, k_sum = 0;  // ncclFloat32, ncclFloat64, ncclSum

    int (*GetUniqueId)(unique_id*)                                                        = nullptr;
    int (*CommInitRank)(comm_t*, int, unique_id, int)                                     = nullptr;
    int (*CommSplit)(comm_t, int, int, comm_t*, void*)                                    = nullptr;
    int (*CommDestroy)(comm_t)                                                            = nullptr;
    int (*AllGather)(void const*, void*, size_t, int, comm_t, cudaStream_t)               = nullptr;
    int (*ReduceScatter)(void const*, void*, size_t, int, int, comm_t, cudaStream_t)      = nullptr;
    char const* (*GetErrorString)(int)                                                    = nullptr;
    int (*GetVersion)(int*)                                                               = nullptr;
    void* lib                                                                             = nullptr;

    static nccl_api* get()
    {
        static nccl_api api;
        static bool tried = false;
        if (!tried) {
            tried = true;
            char const* names[] = {std::getenv("NEO_B200_NCCL_LIB"), "libnccl.so.2", "libnccl.so"};
            for (char const* name : names) {
                if (name == nullptr || *name == 0) { continue; }
                api.lib = dlopen(name, RTLD_NOW | RTLD_GLOBAL);
                if (api.lib != nullptr) { break; }
            }
            if (api.lib != nullptr) {
                auto sym = [&](char const* s) { return dlsym(api.lib, s); };
                api.GetUniqueId    = reinterpret_cast<decltype(api.GetUniqueId)>(sym("ncclGetUniqueId"));
                api.CommInitRank   = reinterpret_cast<decltype(api.CommInitRank)>(sym("ncclCommInitRank"));
                api.CommSplit      = reinterpret_cast<decltype(api.CommSplit)>(sym("ncclCommSplit"));
                api.CommDestroy    = reinterpret_cast<decltype(api.CommDestroy)>(sym("ncclCommDestroy"));
                api.AllGather      = reinterpret_cast<decltype(api.AllGather)>(sym("ncclAllGather"));
                api.ReduceScatter  = reinterpret_cast<decltype(api.ReduceScatter)>(sym("ncclReduceScatter"));
                api.GetErrorString = reinterpret_cast<decltype(api.GetErrorString)>(sym("ncclGetErrorString"));
                api.GetVersion     = reinterpret_cast<decltype(api.GetVersion)>(sym("ncclGetVersion"));
            }
        }
        bool const ok = api.lib != nullptr && api.GetUniqueId != nullptr && api.CommInitRank != nullptr && api.CommSplit != nullptr
                     && api.CommDestroy != nullptr && api.AllGather != nullptr && api.ReduceScatter != nullptr;
        return ok ? &api : nullptr;
    }
};

#define NEO_NCCL_TRY(api, expr)                                                                                                   \
    do {                                                                                                                           \
        int const nccl_status_ = (expr);                                                                                           \
        if (nccl_status_ != 0) {                                                                                                   \
            return fail(NEO_B200_ERR_CUDA, "NCCL: %s failed: %s", #expr,                                                           \
                        (api)->GetErrorString != nullptr ? (api)->GetErrorString(nccl_status_) : "unknown error");                 \
        }                                                                                                                          \
    } while (0)

// steps in flight: the copy-in of step i+2 and the copy-out of step i-1 overlap the kernels of step i (the spectra buffers between
// forward and inverse stay double-buffered; their reuse is ordered by events, it does not limit the depth of the I/O pipeline)
constexpr unsigned k_bank_depth = 3;

// ---- one rank of the bank that lives in this process -----------------------------------------------------------------------------------
struct bank_rank
{
    neo_b200_bank_rank_info info{};
    neo_b200_conv* conv{nullptr};  // the rank's share as an ordinary handle: group channels x its partition range
    cudaStream_t s_in{nullptr}, s_cmp{nullptr}, s_red{nullptr}, s_out{nullptr};
    device_buffer xring;           // [slots][gather_count][max_blocks * B] time-domain input rows
    size_t slots{0}, slot_elems{0};
    device_buffer red[2];          // nccl transport: reduce-scatter result [out_count][T][B] complex
    device_buffer yout[3];         // HOST calls: finished rows on the device before they go back (step mod 3)
    // per-step events, rings of four indexed by step & 3: up to three steps are in flight and a step waits on steps up to three back
    cudaEvent_t ev_in[4]{}, ev_fwd[4]{}, ev_red[4]{}, ev_c2r[4]{}, ev_out[4]{};
    cudaEvent_t t_begin{nullptr}, t_end{nullptr};  // neo_b200_bank_timer_*
    void* partial[2]{};            // partial spectra buffer the forward of (step & 1) wrote
    // push form (fused frame kernel, partition shards > 1): every shard of the group writes the partial spectra of MY channels into
    // my inbox while it computes them; slot (parity, shard) holds [out_count][T][B] complex. inbox_of[s] = base of shard s's inbox as
    // seen from this rank (its own pointer, a peer-mapped pointer, or a CUDA IPC mapping of another process's allocation)
    bool push{false};              // the fused frame kernel stores into the owners' inboxes itself (NEO_B200_BANK_EXCHANGE=kernel)
    bool dma{false};               // default: kernels write locally, the copy engines move each owner's rows into its inbox
    device_buffer inbox;
    size_t inbox_slot{0};          // complex elements per (parity, shard) slot
    void* inbox_of[k_bank_max_shards] = {};
    bool inbox_ipc[k_bank_max_shards] = {};
    device_buffer gate;            // nccl transport: one word per shard, all-gathered as a cross-process stream barrier
    // input rows by copy engine between processes: the other ranks' input rings as CUDA IPC mappings (index = position in the rank's
    // gather domain), the number of slots of each, and the gate words of the input side
    bool dma_in{false};
    std::vector<void*> xring_of;
    std::vector<size_t> xslots_of;
    device_buffer gate_in;
    size_t gather_first{0}, gather_count{0};  // input rows the rank's forward reads (global index, count)
    nccl_api::comm_t comm_world{nullptr}, comm_in{nullptr}, comm_out{nullptr};

    int create_streams()
    {
        for (cudaStream_t* s : {&s_in, &s_cmp, &s_red, &s_out}) { NEO_CUDA_TRY(cudaStreamCreateWithFlags(s, cudaStreamNonBlocking)); }
        for (int b = 0; b < 4; ++b) {
            for (cudaEvent_t* e : {&ev_in[b], &ev_fwd[b], &ev_red[b], &ev_c2r[b], &ev_out[b]}) {
                NEO_CUDA_TRY(cudaEventCreateWithFlags(e, cudaEventDisableTiming));
            }
        }
        NEO_CUDA_TRY(cudaEventCreate(&t_begin));
        NEO_CUDA_TRY(cudaEventCreate(&t_end));
        return NEO_B200_OK;
    }

    void destroy(nccl_api* api)
    {
        cudaSetDevice(info.device);
        for (cudaStream_t s : {s_in, s_cmp, s_red, s_out}) {
            if (s != nullptr) { cudaStreamSynchronize(s); }
        }
        if (api != nullptr) {
            if (comm_out != nullptr) { api->CommDestroy(comm_out); }
            if (comm_in != nullptr && comm_in != comm_world) { api->CommDestroy(comm_in); }
            if (comm_world != nullptr) { api->CommDestroy(comm_world); }
        }
        for (int s = 0; s < k_bank_max_shards; ++s) {
            if (inbox_ipc[s] && inbox_of[s] != nullptr) { cudaIpcCloseMemHandle(inbox_of[s]); }
        }
        if (dma_in) {
            for (void* p : xring_of) {
                if (p != nullptr && p != xring.ptr) { cudaIpcCloseMemHandle(p); }
            }
        }
        neo_b200_conv_destroy(conv);
        xring.release();
        for (auto& buf : red) { buf.release(); }
        for (auto& buf : yout) { buf.release(); }
        for (int b = 0; b < 4; ++b) {
            for (cudaEvent_t e : {ev_in[b], ev_fwd[b], ev_red[b], ev_c2r[b], ev_out[b]}) {
                if (e != nullptr) { cudaEventDestroy(e); }
            }
        }
        for (cudaEvent_t e : {t_begin, t_end}) {
            if (e != nullptr) { cudaEventDestroy(e); }
        }
        for (cudaStream_t s : {s_in, s_cmp, s_red, s_out}) {
            if (s != nullptr) { cudaStreamDestroy(s); }
        }
    }
};

}  // namespace
}  // namespace neo_b200

// a submitted step: its inverse side (sum of the group's partial spectra + c2r + copy-out) may still be waiting to be enqueued
struct neo_b200_bank_step
{
    std::uint64_t step{0};
    size_t blocks{0};
    int memspace{0};
    std::vector<void*> out_rows;
    bool finished{false};
};

struct neo_b200_bank
{
    neo_b200_conv_config cfg{};
    neo_b200_bank_layout layout{};
    size_t world{0};
    bool nccl{false};
    neo_b200::nccl_api* api{nullptr};
    std::deque<neo_b200::bank_rank> ranks;   // the ranks of this process, ascending (deque: a rank owns device buffers and never moves)
    std::uint64_t step{0};
    std::deque<neo_b200_bank_step> pending;  // submitted, not yet waited for
    bool has_filter{false};

    ~neo_b200_bank()
    {
        for (auto& r : ranks) { r.destroy(api); }
    }

    neo_b200::bank_rank* find(size_t rank)
    {
        for (auto& r : ranks) {
            if (size_t(r.info.rank) == rank) { return &r; }
        }
        return nullptr;
    }
};

namespace neo_b200 {
namespace {

// shard gp of Gp over the partition axis; in frame mode shards start on frame boundaries (the delay of a shard is whole frames)
inline void bank_partition_range(size_t parts, size_t frame, size_t shards, size_t gp, size_t* lo, size_t* hi)
{
    size_t const unit  = frame > 0 ? frame : 1;
    size_t const units = (parts + unit - 1) / unit;
    *lo                = std::min(parts, (gp * units / shards) * unit);
    *hi                = std::min(parts, ((gp + 1) * units / shards) * unit);
}

int bank_validate(neo_b200_conv_config& c, neo_b200_bank_layout const& l, size_t world)
{
    NEO_TRY(validate(c));
    if (!(c.partition_begin == 0 && c.partition_end == c.partitions)) {
        return fail(NEO_B200_ERR_INVALID, "a bank shards the partitions itself: leave partition_begin/partition_end at 0");
    }
    if (l.channel_groups == 0 || l.partition_shards == 0 || l.channel_groups * l.partition_shards != world) {
        return fail(NEO_B200_ERR_INVALID, "layout %zu channel groups x %zu partition shards does not match %zu ranks", l.channel_groups,
                    l.partition_shards, world);
    }
    if (l.partition_shards > size_t(k_bank_max_shards)) {
        return fail(NEO_B200_ERR_UNSUPPORTED, "at most %d partition shards", k_bank_max_shards);
    }
    if (c.outputs % world != 0 || c.inputs % world != 0) {
        return fail(NEO_B200_ERR_UNSUPPORTED, "outputs=%zu and inputs=%zu must be multiples of the %zu ranks", c.outputs, c.inputs, world);
    }
    size_t const unit  = c.frame_blocks > 0 ? c.frame_blocks : 1;
    size_t const units = (c.partitions + unit - 1) / unit;
    if (units < l.partition_shards) {
        return fail(NEO_B200_ERR_INVALID, "%zu partitions (%zu per frame) cannot be cut into %zu shards", c.partitions, unit, l.partition_shards);
    }
    return NEO_B200_OK;
}

void bank_fill_info(neo_b200_conv_config const& c, neo_b200_bank_layout const& l, size_t world, size_t rank, int device,
                    neo_b200_bank_rank_info* info)
{
    size_t const gp = rank % l.partition_shards, gc = rank / l.partition_shards;
    info->rank            = int(rank);
    info->device          = device;
    info->channel_group   = gc;
    info->partition_shard = gp;
    info->group_count     = c.outputs / l.channel_groups;
    info->group_first     = gc * info->group_count;
    info->out_count       = c.outputs / world;
    info->out_first       = rank * info->out_count;
    info->in_count        = c.inputs / world;
    info->in_first        = rank * info->in_count;
    bank_partition_range(c.partitions, c.frame_blocks, l.partition_shards, gp, &info->partition_begin, &info->partition_end);
    info->delay_blocks    = c.frame_blocks > 0 ? info->partition_begin : 0;
}

// build the rank's streams, sub-handle and buffers on its device
int bank_build_rank(neo_b200_bank* bank, bank_rank& r)
{
    neo_b200_conv_config const& c = bank->cfg;
    NEO_CUDA_TRY(cudaSetDevice(r.info.device));
    NEO_TRY(r.create_streams());
    neo_b200_conv_config sub = c;
    sub.outputs              = r.info.group_count;
    sub.inputs               = c.topology == NEO_B200_MATRIX ? c.inputs : r.info.group_count;
    sub.partition_begin      = r.info.partition_begin;
    sub.partition_end        = r.info.partition_end;
    sub.input_delayed        = r.info.delay_blocks > 0 ? 1 : 0;
    NEO_TRY(neo_b200_conv_create(&r.conv, &sub));
    r.gather_first = c.topology == NEO_B200_MATRIX ? 0 : r.info.group_first;
    r.gather_count = c.topology == NEO_B200_MATRIX ? c.inputs : r.info.group_count;
    size_t const esz = elem_size(c.dtype);
    r.slots          = (c.frame_blocks > 0 ? r.info.delay_blocks / c.frame_blocks : 0) + k_bank_depth;
    r.slot_elems     = r.gather_count * c.max_blocks * c.block;
    NEO_TRY(r.xring.reserve(r.slots * r.slot_elems * esz));
    NEO_CUDA_TRY(cudaMemsetAsync(r.xring.ptr, 0, r.xring.bytes, r.s_in));
    NEO_CUDA_TRY(cudaStreamSynchronize(r.s_in));
    bool fused = false;
    (void)with_engine(r.conv, [&](auto& e) {
        fused = e.fused;
        return NEO_B200_OK;
    });
    size_t const gp_n = bank->layout.partition_shards;
    // how the partial spectra of a group reach the rank that finishes a channel (NEO_B200_BANK_EXCHANGE):
    //   dma        (default) every shard's kernels write their partial spectra locally; the copy engines then move each owner's rows
    //              into its inbox over NVLink (no SM and no store queue of the compute kernel involved) and the c2r kernel sums its
    //              own rows and its inbox slots;
    //   kernel     the fused frame kernel stores the rows straight into the owners' inboxes (peer stores; wide frame-mode banks);
    //   collective ncclReduceScatter (rank-per-process) / peer loads inside the c2r kernel (devices[] banks).
    // measured, BASELINE config 5 on 2 GPUs (1 x 2), ms per fused step / per step: kernel 7.6 / 8.7, collective 5.5 / 8.7, dma see DESIGN.md
    char const* const how = std::getenv("NEO_B200_BANK_EXCHANGE");
    std::string const exchange = how != nullptr ? how : "dma";
    r.push = gp_n > 1 && fused && exchange == "kernel";
    r.dma  = gp_n > 1 && !r.push && exchange != "collective";
    if (r.push || r.dma) {
        r.inbox_slot = r.info.out_count * c.max_blocks * c.block;
        NEO_TRY(r.inbox.reserve(2 * gp_n * r.inbox_slot * 2 * esz));
        r.inbox_of[r.info.partition_shard] = r.inbox.ptr;
    }
    return NEO_B200_OK;
}

// push form: every rank of a group learns where the other shards' inboxes are. All ranks in one process: their pointers, readable
// and writable through peer access. One rank per process: CUDA IPC handles, exchanged with ncclAllGather on the group communicator.
inline void bank_domains(neo_b200_bank const* bank, bank_rank const& r, std::vector<size_t>* gather, std::vector<size_t>* reduce);

// rank-per-process banks, copy-engine exchange: the ranks of a gather domain map each other's input rings (CUDA IPC), so that a rank's
// input rows reach the others by cudaMemcpyAsync over NVLink instead of an SM-resident ncclAllGather kernel
int bank_connect_inputs(neo_b200_bank* bank)
{
    if (!bank->nccl) { return NEO_B200_OK; }
    char const* const how = std::getenv("NEO_B200_BANK_EXCHANGE");
    if (how != nullptr && std::string(how) == "collective") { return NEO_B200_OK; }
    for (auto& r : bank->ranks) {
        std::vector<size_t> gather;
        bank_domains(bank, r, &gather, nullptr);
        if (gather.size() <= 1) { continue; }
        NEO_CUDA_TRY(cudaSetDevice(r.info.device));
        size_t const n = gather.size();
        size_t me      = 0;
        for (size_t i = 0; i < n; ++i) {
            if (gather[i] == size_t(r.info.rank)) { me = i; }
        }
        cudaIpcMemHandle_t mine{};
        NEO_CUDA_TRY(cudaIpcGetMemHandle(&mine, r.xring.ptr));
        device_buffer staging;
        NEO_TRY(staging.reserve(n * sizeof(mine)));
        char* const slots = staging.as<char>();
        NEO_CUDA_TRY(cudaMemcpyAsync(slots + me * sizeof(mine), &mine, sizeof(mine), cudaMemcpyHostToDevice, r.s_in));
        NEO_NCCL_TRY(bank->api, bank->api->AllGather(slots + me * sizeof(mine), slots, sizeof(mine) / 4, nccl_api::k_float32, r.comm_in, r.s_in));
        std::vector<cudaIpcMemHandle_t> all(n);
        NEO_CUDA_TRY(cudaMemcpyAsync(all.data(), slots, n * sizeof(mine), cudaMemcpyDeviceToHost, r.s_in));
        NEO_CUDA_TRY(cudaStreamSynchronize(r.s_in));
        r.xring_of.assign(n, nullptr);
        r.xslots_of.assign(n, 0);
        for (size_t i = 0; i < n; ++i) {
            neo_b200_bank_rank_info peer{};
            bank_fill_info(bank->cfg, bank->layout, bank->world, gather[i], -1, &peer);
            r.xslots_of[i] = (bank->cfg.frame_blocks > 0 ? peer.delay_blocks / bank->cfg.frame_blocks : 0) + k_bank_depth;
            if (i == me) { r.xring_of[i] = r.xring.ptr; }
            else { NEO_CUDA_TRY(cudaIpcOpenMemHandle(&r.xring_of[i], all[i], cudaIpcMemLazyEnablePeerAccess)); }
        }
        NEO_TRY(r.gate_in.reserve(n * sizeof(float)));
        NEO_CUDA_TRY(cudaMemsetAsync(r.gate_in.ptr, 0, r.gate_in.bytes, r.s_in));
        NEO_CUDA_TRY(cudaStreamSynchronize(r.s_in));
        r.dma_in = true;
    }
    return NEO_B200_OK;
}

int bank_connect_inboxes(neo_b200_bank* bank)
{
    size_t const gp_n = bank->layout.partition_shards;
    for (auto& r : bank->ranks) {
        if (!r.push && !r.dma) { continue; }
        NEO_CUDA_TRY(cudaSetDevice(r.info.device));
        size_t const base = r.info.channel_group * gp_n;
        if (!bank->nccl) {
            for (size_t s = 0; s < gp_n; ++s) {
                bank_rank* const peer = bank->find(base + s);
                if (peer->push != r.push || peer->dma != r.dma) { return fail(NEO_B200_ERR_INVALID, "the ranks of a group disagree about the exchange form"); }
                r.inbox_of[s] = peer->inbox.ptr;
            }
            continue;
        }
        cudaIpcMemHandle_t mine{};
        NEO_CUDA_TRY(cudaIpcGetMemHandle(&mine, r.inbox.ptr));
        device_buffer staging;
        NEO_TRY(staging.reserve(gp_n * sizeof(mine)));
        char* const slots = staging.as<char>();
        NEO_CUDA_TRY(cudaMemcpyAsync(slots + r.info.partition_shard * sizeof(mine), &mine, sizeof(mine), cudaMemcpyHostToDevice, r.s_red));
        NEO_NCCL_TRY(bank->api, bank->api->AllGather(slots + r.info.partition_shard * sizeof(mine), slots, sizeof(mine) / 4, nccl_api::k_float32,
                                                     r.comm_out, r.s_red));
        std::vector<cudaIpcMemHandle_t> all(gp_n);
        NEO_CUDA_TRY(cudaMemcpyAsync(all.data(), slots, gp_n * sizeof(mine), cudaMemcpyDeviceToHost, r.s_red));
        NEO_CUDA_TRY(cudaStreamSynchronize(r.s_red));
        for (size_t s = 0; s < gp_n; ++s) {
            if (s == r.info.partition_shard) { continue; }
            NEO_CUDA_TRY(cudaIpcOpenMemHandle(&r.inbox_of[s], all[s], cudaIpcMemLazyEnablePeerAccess));
            r.inbox_ipc[s] = true;
        }
        NEO_TRY(r.gate.reserve(gp_n * sizeof(float)));
        NEO_CUDA_TRY(cudaMemsetAsync(r.gate.ptr, 0, r.gate.bytes, r.s_red));
        NEO_CUDA_TRY(cudaStreamSynchronize(r.s_red));
    }
    return NEO_B200_OK;
}

int bank_common_create(neo_b200_bank** out, neo_b200_conv_config const* config, neo_b200_bank_layout const* layout, size_t world,
                       std::unique_ptr<neo_b200_bank>& bank)
{
    if (out == nullptr || config == nullptr || layout == nullptr) { return fail(NEO_B200_ERR_INVALID, "null argument"); }
    *out = nullptr;
    neo_b200_conv_config c = *config;
    NEO_TRY(bank_validate(c, *layout, world));
    NEO_TRY(require_device());
    bank.reset(new (std::nothrow) neo_b200_bank{});
    if (!bank) { return fail(NEO_B200_ERR_ALLOC, "out of host memory"); }
    bank->cfg    = c;
    bank->layout = *layout;
    bank->world  = world;
    return NEO_B200_OK;
}

// ranks whose input rows rank r needs (its gather domain) / whose partial spectra it sums (its reduce group), ascending
inline void bank_domains(neo_b200_bank const* bank, bank_rank const& r, std::vector<size_t>* gather, std::vector<size_t>* reduce)
{
    size_t const gp_n = bank->layout.partition_shards;
    size_t const base = r.info.channel_group * gp_n;
    if (reduce != nullptr) {
        for (size_t j = 0; j < gp_n; ++j) { reduce->push_back(base + j); }
    }
    if (gather != nullptr) {
        if (bank->cfg.topology == NEO_B200_MATRIX) {
            for (size_t j = 0; j < bank->world; ++j) { gather->push_back(j); }
        } else {
            for (size_t j = 0; j < gp_n; ++j) { gather->push_back(base + j); }
        }
    }
}

int bank_finish(neo_b200_bank* bank, neo_b200_bank_step& st);
int bank_finish_older(neo_b200_bank* bank);

int bank_wait_oldest(neo_b200_bank* bank)
{
    if (bank->pending.empty()) { return NEO_B200_OK; }
    NEO_TRY(bank_finish(bank, bank->pending.front()));  // nobody submitted after it: its inverse side has not been enqueued yet
    int const e = int(bank->pending.front().step & 3U);
    for (auto& r : bank->ranks) {
        NEO_CUDA_TRY(cudaSetDevice(r.info.device));
        NEO_CUDA_TRY(cudaEventSynchronize(r.ev_out[e]));
    }
    bank->pending.pop_front();
    return NEO_B200_OK;
}

template<typename T>
int bank_submit_impl(neo_b200_bank* bank, void const* const* in_rows, void* const* out_rows, size_t blocks, int memspace)
{
    neo_b200_conv_config const& c = bank->cfg;
    size_t const pitch            = blocks * c.block;          // reals per row of this call
    std::uint64_t const step      = bank->step;
    int const b                   = int(step & 1U);  // parity of the double-buffered spectra (partial buffers, inbox slots)
    int const e0                  = int(step & 3U);  // this step's slot in the event rings
    // event of `back` steps ago in a ring (nullptr before the first step: nothing to wait for)
    auto const ago = [&](cudaEvent_t const (&ring)[4], unsigned back) -> cudaEvent_t { return step >= back ? ring[(step - back) & 3U] : nullptr; };
    auto const wait_for = [&](cudaStream_t s, cudaEvent_t ev) -> int {
        if (ev != nullptr) { NEO_CUDA_TRY(cudaStreamWaitEvent(s, ev, 0)); }
        return NEO_B200_OK;
    };
    size_t const gp_n             = bank->layout.partition_shards;
    bool const host               = memspace == NEO_B200_HOST;
    cudaMemcpyKind const kin      = host ? cudaMemcpyHostToDevice : cudaMemcpyDeviceToDevice;

    // ---- 1. input rows into slot (step mod slots) of every rank that needs them ----
    for (size_t l = 0; l < bank->ranks.size(); ++l) {
        bank_rank& r = bank->ranks[l];
        NEO_CUDA_TRY(cudaSetDevice(r.info.device));
        std::vector<size_t> gather;
        bank_domains(bank, r, &gather, nullptr);
        // the slot about to be overwritten was last read by the forward of k_bank_depth steps ago, on every rank it is pushed to
        if (bank->nccl) {
            NEO_TRY(wait_for(r.s_in, ago(r.ev_fwd, k_bank_depth)));
        } else {
            for (size_t p : gather) { NEO_TRY(wait_for(r.s_in, ago(bank->find(p)->ev_fwd, k_bank_depth))); }
        }
        T* const slot      = r.xring.template as<T>() + (step % r.slots) * r.slot_elems;
        size_t const mine  = (r.info.in_first - r.gather_first) * pitch;  // offset of the rank's own rows inside a slot
        size_t const bytes = r.info.in_count * pitch * sizeof(T);
        NEO_CUDA_TRY(cudaMemcpyAsync(slot + mine, in_rows[l], bytes, kin, r.s_in));
        if (gather.size() > 1) {
            if (bank->nccl && r.dma_in) {
                // copy engines push the rows into the other ranks' rings (all ranks of a gather domain hold the same rows per slot)
                size_t me = 0;
                for (size_t i = 0; i < gather.size(); ++i) {
                    if (gather[i] == size_t(r.info.rank)) { me = i; }
                }
                for (size_t i = 0; i < gather.size(); ++i) {
                    if (i == me) { continue; }
                    T* const dst = static_cast<T*>(r.xring_of[i]) + (step % r.xslots_of[i]) * r.slot_elems + mine;
                    NEO_CUDA_TRY(cudaMemcpyAsync(dst, slot + mine, bytes, cudaMemcpyDeviceToDevice, r.s_in));
                }
                // gate of the input side: completes here when every rank of the domain has reached it -- its rows of this step have
                // landed and, because each rank first waits for its own forward of two steps ago, the slots step i+1 overwrites
                // (last read by the forwards of step i-2) are free
                NEO_TRY(wait_for(r.s_in, ago(r.ev_fwd, 2)));
                float* const words = r.gate_in.as<float>();
                NEO_NCCL_TRY(bank->api, bank->api->AllGather(words + me, words, 1, nccl_api::k_float32, r.comm_in, r.s_in));
            } else if (bank->nccl) {
                NEO_NCCL_TRY(bank->api, bank->api->AllGather(slot + mine, slot, r.info.in_count * pitch,
                                                             sizeof(T) == 4 ? nccl_api::k_float32 : nccl_api::k_float64, r.comm_in, r.s_in));
            } else {
                for (size_t p : gather) {  // push the rows over NVLink into the peers' slots
                    bank_rank* const peer = bank->find(p);
                    if (peer == &r) { continue; }
                    T* const dst = peer->xring.template as<T>() + (step % peer->slots) * peer->slot_elems + (r.info.in_first - peer->gather_first) * pitch;
                    NEO_CUDA_TRY(cudaMemcpyPeerAsync(dst, peer->info.device, slot + mine, r.info.device, bytes, r.s_in));
                }
            }
        }
        NEO_CUDA_TRY(cudaEventRecord(r.ev_in[e0], r.s_in));
    }

    // kernel-push form: the gate behind this step's forward waits for the previous step's c2r, so that c2r goes first
    bool any_push = false;
    for (auto& r : bank->ranks) { any_push = any_push || r.push; }
    if (any_push) { NEO_TRY(bank_finish_older(bank)); }

    // ---- 2. forward: window + r2c + delay line + MAC of the rank's partitions -> partial spectra ----
    for (auto& r : bank->ranks) {
        NEO_CUDA_TRY(cudaSetDevice(r.info.device));
        std::vector<size_t> gather, reduce;
        bank_domains(bank, r, &gather, &reduce);
        if (bank->nccl) {
            NEO_CUDA_TRY(cudaStreamWaitEvent(r.s_cmp, r.ev_in[e0], 0));
            // the reduce-scatter / copy-out of two steps ago read this buffer (kernel push: the gate of the previous step orders it)
            if (gp_n > 1 && !r.push) { NEO_TRY(wait_for(r.s_cmp, ago(r.ev_red, 2))); }
            if (r.dma) { NEO_TRY(wait_for(r.s_cmp, ago(r.ev_c2r, 2))); }  // ... and the c2r of two steps ago read the rank's own rows of it
        } else {
            for (size_t p : gather) { NEO_CUDA_TRY(cudaStreamWaitEvent(r.s_cmp, bank->find(p)->ev_in[e0], 0)); }
            // the partial spectra buffer / inbox slot of this parity was last read by the c2r of two steps ago on every rank of the group
            if (gp_n > 1) {
                for (size_t p : reduce) { NEO_TRY(wait_for(r.s_cmp, ago(bank->find(p)->ev_c2r, 2))); }
            }
            if (r.dma) { NEO_TRY(wait_for(r.s_cmp, ago(r.ev_red, 2))); }  // the copy-out of two steps ago read this buffer
        }
        // an unsharded handle has a single spectra buffer: the c2r of the previous step must have read it
        if (gp_n == 1) { NEO_TRY(wait_for(r.s_cmp, ago(r.ev_c2r, 1))); }
        size_t const delay_slots = c.frame_blocks > 0 ? r.info.delay_blocks / c.frame_blocks : 0;
        size_t const read_slot   = (step + r.slots - delay_slots) % r.slots;  // zeros until the delayed step exists
        T const* const x         = r.xring.template as<T>() + read_slot * r.slot_elems;
        NEO_TRY(with_engine(r.conv, [&](auto& e) -> int {
            using E = std::remove_reference_t<decltype(e)>;
            if constexpr (std::is_same_v<E, conv_engine<T>>) {
                NEO_TRY(e.forward_r2c(x, pitch, blocks, 0, r.conv->cfg.inputs, r.s_cmp));
                e.push_owners = 0;
                if (r.push) {  // result rows of owner o's channels go into o's inbox, slot (parity, my shard)
                    e.push_owners    = int(gp_n);
                    e.push_own_count = int(r.info.out_count);
                    for (size_t o = 0; o < gp_n; ++o) {
                        e.push_dst[o] = static_cast<cx<T>*>(r.inbox_of[o]) + (size_t(b) * gp_n + r.info.partition_shard) * r.inbox_slot;
                    }
                }
                NEO_TRY(e.forward_mac(blocks, 0, r.conv->cfg.outputs, r.s_cmp));
                r.partial[b] = e.acc_w();
                e.advance(blocks);
            }
            return NEO_B200_OK;
        }));
        if (r.push && bank->nccl) {
            // gate of step i: a tiny all-gather on the compute stream. It completes on this rank only after every shard of the group has
            // reached it, i.e. finished its forward of step i (its stores into my inbox are done) and -- because each rank waits for
            // its own c2r of step i-1 first -- finished reading the inbox slots that the forwards of step i+1 will overwrite.
            NEO_TRY(wait_for(r.s_cmp, ago(r.ev_c2r, 1)));
            float* const words = r.gate.as<float>();
            NEO_NCCL_TRY(bank->api, bank->api->AllGather(words + r.info.partition_shard, words, 1, nccl_api::k_float32, r.comm_out, r.s_cmp));
        }
        NEO_CUDA_TRY(cudaEventRecord(r.ev_fwd[e0], r.s_cmp));
    }

    // the previous step's inverse side goes behind this step's forward on the compute stream (its exchange had the forward to finish)
    NEO_TRY(bank_finish_older(bank));

    // ---- 3a. copy-engine exchange: each rank hands every other shard of its group the partial spectra of THAT shard's channels ----
    for (auto& r : bank->ranks) {
        if (!r.dma) { continue; }
        NEO_CUDA_TRY(cudaSetDevice(r.info.device));
        size_t const base      = r.info.channel_group * gp_n;
        size_t const own_elems = r.info.out_count * blocks * c.block;
        NEO_CUDA_TRY(cudaStreamWaitEvent(r.s_red, r.ev_fwd[e0], 0));
        for (size_t o = 0; o < gp_n; ++o) {
            if (o == r.info.partition_shard) { continue; }
            // the owner's c2r of two steps ago read this inbox slot (rank-per-process: the gate of the previous step orders it)
            if (!bank->nccl) { NEO_TRY(wait_for(r.s_red, ago(bank->find(base + o)->ev_c2r, 2))); }
            cx<T>* const dst       = static_cast<cx<T>*>(r.inbox_of[o]) + (size_t(b) * gp_n + r.info.partition_shard) * r.inbox_slot;
            cx<T> const* const src = static_cast<cx<T> const*>(r.partial[b]) + o * own_elems;
            NEO_CUDA_TRY(cudaMemcpyAsync(dst, src, own_elems * sizeof(cx<T>), cudaMemcpyDeviceToDevice, r.s_red));
        }
        if (bank->nccl) {
            // gate of step i: completes here only when every shard of the group has reached it -- its copies of step i have landed
            // and, because each rank first waits for its own c2r of step i-1, the inbox slots that step i+1 overwrites are free
            NEO_TRY(wait_for(r.s_red, ago(r.ev_c2r, 1)));
            float* const words = r.gate.as<float>();
            NEO_NCCL_TRY(bank->api, bank->api->AllGather(words + r.info.partition_shard, words, 1, nccl_api::k_float32, r.comm_out, r.s_red));
        }
        NEO_CUDA_TRY(cudaEventRecord(r.ev_red[e0], r.s_red));
    }

    // the reduce-scatter of the collective form is this step's exchange too
    for (auto& r : bank->ranks) {
        if (gp_n == 1 || r.dma || r.push || !bank->nccl) { continue; }
        NEO_CUDA_TRY(cudaSetDevice(r.info.device));
        size_t const own_elems = r.info.out_count * blocks * c.block;
        NEO_CUDA_TRY(cudaStreamWaitEvent(r.s_red, r.ev_fwd[e0], 0));
        NEO_TRY(wait_for(r.s_red, ago(r.ev_c2r, 2)));  // the c2r of two steps ago read red[b]
        NEO_TRY(r.red[b].reserve(own_elems * sizeof(cx<T>)));
        NEO_NCCL_TRY(bank->api, bank->api->ReduceScatter(r.partial[b], r.red[b].ptr, own_elems * 2,
                                                         sizeof(T) == 4 ? nccl_api::k_float32 : nccl_api::k_float64, nccl_api::k_sum, r.comm_out,
                                                         r.s_red));
        NEO_CUDA_TRY(cudaEventRecord(r.ev_red[e0], r.s_red));
    }

    neo_b200_bank_step st;
    st.step     = step;
    st.blocks   = blocks;
    st.memspace = memspace;
    st.out_rows.assign(out_rows, out_rows + bank->ranks.size());
    bank->pending.push_back(std::move(st));
    ++bank->step;
    // without partition shards nothing is exchanged: the inverse side follows at once. With shards and DEVICE buffers it is enqueued
    // behind the NEXT step's forward (or by wait), so the exchange of this step has a whole forward to complete and the compute stream
    // never idles. HOST calls are bound by the host link, not by the kernels: there the copy-out must start as early as possible
    // (deferring it would put a forward and an input copy between a step's c2r and the submit that its completion unblocks).
    if (gp_n == 1 || host) { NEO_TRY(bank_finish(bank, bank->pending.back())); }
    return NEO_B200_OK;
}

// ---- 3b. sum over the partition shards + c2r for the rank's own channels; 4. output rows. On the compute stream: the transforms are
// issue-bound, running them beside the next forward only slows both (measured), what overlaps them is the copy engines' work ----
template<typename T>
int bank_finish_impl(neo_b200_bank* bank, neo_b200_bank_step& st)
{
    neo_b200_conv_config const& c = bank->cfg;
    size_t const blocks = st.blocks;
    size_t const pitch  = blocks * c.block;
    int const b         = int(st.step & 1U);
    int const e0        = int(st.step & 3U);
    size_t const gp_n   = bank->layout.partition_shards;
    bool const host     = st.memspace == NEO_B200_HOST;
    for (size_t l = 0; l < bank->ranks.size(); ++l) {
        bank_rank& r = bank->ranks[l];
        NEO_CUDA_TRY(cudaSetDevice(r.info.device));
        std::vector<size_t> reduce;
        bank_domains(bank, r, nullptr, &reduce);
        size_t const own_in_group = r.info.out_first - r.info.group_first;  // first own channel, relative to the group
        cx<T> const* srcs[k_bank_max_shards];
        int nsrc = 1;
        if (gp_n == 1) {
            srcs[0] = static_cast<cx<T> const*>(r.partial[b]) + own_in_group * blocks * c.block;  // same stream as the forward
        } else if (r.dma) {
            // own rows straight from the rank's partial spectra, the other shards' rows from the inbox: a LOCAL sum, in shard order
            if (bank->nccl) {
                NEO_CUDA_TRY(cudaStreamWaitEvent(r.s_cmp, r.ev_red[e0], 0));  // recorded behind the gate
            } else {
                for (size_t p : reduce) { NEO_CUDA_TRY(cudaStreamWaitEvent(r.s_cmp, bank->find(p)->ev_red[e0], 0)); }
            }
            nsrc = int(gp_n);
            for (size_t s = 0; s < gp_n; ++s) {
                srcs[s] = s == r.info.partition_shard ? static_cast<cx<T> const*>(r.partial[b]) + own_in_group * blocks * c.block
                                                      : r.inbox.template as<cx<T>>() + (size_t(b) * gp_n + s) * r.inbox_slot;
            }
        } else if (r.push) {
            // the shards have pushed their partial spectra of my channels into my inbox: a LOCAL sum, in shard order
            // (rank-per-process: the gate sits on this stream behind the forward)
            if (!bank->nccl) {
                for (size_t p : reduce) { NEO_CUDA_TRY(cudaStreamWaitEvent(r.s_cmp, bank->find(p)->ev_fwd[e0], 0)); }
            }
            nsrc = int(gp_n);
            for (size_t s = 0; s < gp_n; ++s) { srcs[s] = r.inbox.template as<cx<T>>() + (size_t(b) * gp_n + s) * r.inbox_slot; }
        } else if (bank->nccl) {
            NEO_CUDA_TRY(cudaStreamWaitEvent(r.s_cmp, r.ev_red[e0], 0));
            srcs[0] = r.red[b].template as<cx<T>>();
        } else {
            nsrc = 0;
            for (size_t p : reduce) {  // shard order: every rank sums in the same order
                bank_rank* const peer = bank->find(p);
                NEO_CUDA_TRY(cudaStreamWaitEvent(r.s_cmp, peer->ev_fwd[e0], 0));
                srcs[nsrc++] = static_cast<cx<T> const*>(peer->partial[b]) + own_in_group * blocks * c.block;
            }
        }
        T* dst = static_cast<T*>(st.out_rows[l]);
        if (host) {
            device_buffer& stage = r.yout[st.step % k_bank_depth];
            NEO_TRY(stage.reserve(r.info.out_count * c.max_blocks * c.block * sizeof(T)));
            dst = stage.template as<T>();
            if (st.step >= k_bank_depth) {  // its previous copy-out (on the output stream) has left
                NEO_CUDA_TRY(cudaStreamWaitEvent(r.s_cmp, r.ev_out[(st.step - k_bank_depth) & 3U], 0));
            }
        }
        NEO_TRY(with_engine(r.conv, [&](auto& e) -> int {
            using E = std::remove_reference_t<decltype(e)>;
            if constexpr (std::is_same_v<E, conv_engine<T>>) {
                return e.inverse(srcs, nsrc, dst, pitch, own_in_group, r.info.out_count, blocks, r.s_cmp);
            }
            return NEO_B200_OK;
        }));
        NEO_CUDA_TRY(cudaEventRecord(r.ev_c2r[e0], r.s_cmp));
        NEO_CUDA_TRY(cudaStreamWaitEvent(r.s_out, r.ev_c2r[e0], 0));
        if (host) {
            NEO_CUDA_TRY(cudaMemcpyAsync(st.out_rows[l], dst, r.info.out_count * pitch * sizeof(T), cudaMemcpyDeviceToHost, r.s_out));
        }
        NEO_CUDA_TRY(cudaEventRecord(r.ev_out[e0], r.s_out));
    }
    st.finished = true;
    return NEO_B200_OK;
}

int bank_finish(neo_b200_bank* bank, neo_b200_bank_step& st)
{
    if (st.finished) { return NEO_B200_OK; }
    return bank->cfg.dtype == NEO_B200_F32 ? bank_finish_impl<float>(bank, st) : bank_finish_impl<double>(bank, st);
}

// enqueue the inverse side of every step submitted before the current one
int bank_finish_older(neo_b200_bank* bank)
{
    for (auto& st : bank->pending) { NEO_TRY(bank_finish(bank, st)); }
    return NEO_B200_OK;
}

int bank_check_call(neo_b200_bank* bank, void const* const* in_rows, void* const* out_rows, size_t blocks)
{
    if (bank == nullptr || in_rows == nullptr || out_rows == nullptr) { return fail(NEO_B200_ERR_INVALID, "null argument"); }
    if (!bank->has_filter) { return fail(NEO_B200_ERR_INVALID, "no filter set"); }
    if (blocks == 0 || blocks > bank->cfg.max_blocks) {
        return fail(NEO_B200_ERR_INVALID, "blocks=%zu outside [1, max_blocks=%zu]", blocks, bank->cfg.max_blocks);
    }
    if (bank->cfg.frame_blocks != 0 && blocks != bank->cfg.frame_blocks) {
        return fail(NEO_B200_ERR_INVALID, "frame mode: every call processes exactly frame_blocks=%zu blocks, got %zu", bank->cfg.frame_blocks, blocks);
    }
    for (size_t l = 0; l < bank->ranks.size(); ++l) {
        if (in_rows[l] == nullptr || out_rows[l] == nullptr) { return fail(NEO_B200_ERR_INVALID, "null row pointer for local rank %zu", l); }
    }
    return NEO_B200_OK;
}

}  // namespace
}  // namespace neo_b200

extern "C" {

int neo_b200_bank_unique_id(void* id)
{
    if (id == nullptr) { return fail(NEO_B200_ERR_INVALID, "null argument"); }
    nccl_api* const api = nccl_api::get();
    if (api == nullptr) { return fail(NEO_B200_ERR_UNSUPPORTED, "NCCL (libnccl.so.2 or $NEO_B200_NCCL_LIB) could not be loaded"); }
    nccl_api::unique_id uid{};
    NEO_NCCL_TRY(api, api->GetUniqueId(&uid));
    std::memcpy(id, &uid, sizeof(uid));
    return NEO_B200_OK;
}

int neo_b200_bank_create(neo_b200_bank** out, neo_b200_conv_config const* config, neo_b200_bank_layout const* layout, int const* devices,
                         size_t n_devices)
{
    if (devices == nullptr || n_devices == 0) { return fail(NEO_B200_ERR_INVALID, "no devices"); }
    std::unique_ptr<neo_b200_bank> bank;
    NEO_TRY(bank_common_create(out, config, layout, n_devices, bank));
    int const ndev = neo_b200_device_count();
    int before     = 0;
    cudaGetDevice(&before);
    bank->ranks.resize(n_devices);
    for (size_t r = 0; r < n_devices; ++r) {
        if (devices[r] < 0 || devices[r] >= ndev) { return fail(NEO_B200_ERR_INVALID, "device %d does not exist (%d devices)", devices[r], ndev); }
        bank_fill_info(bank->cfg, bank->layout, n_devices, r, devices[r], &bank->ranks[r].info);
    }
    // peer transport: rows are pushed into, and partial spectra read from, the memory of the other devices
    for (size_t a = 0; a < n_devices; ++a) {
        for (size_t b = 0; b < n_devices; ++b) {
            if (devices[a] == devices[b]) { continue; }
            int can = 0;
            NEO_CUDA_TRY(cudaDeviceCanAccessPeer(&can, devices[a], devices[b]));
            if (can == 0) { return fail(NEO_B200_ERR_UNSUPPORTED, "device %d cannot map the memory of device %d (no peer access)", devices[a], devices[b]); }
            NEO_CUDA_TRY(cudaSetDevice(devices[a]));
            cudaError_t const err = cudaDeviceEnablePeerAccess(devices[b], 0);
            if (err != cudaSuccess && err != cudaErrorPeerAccessAlreadyEnabled) {
                return fail(NEO_B200_ERR_CUDA, "cudaDeviceEnablePeerAccess(%d -> %d): %s", devices[a], devices[b], cudaGetErrorString(err));
            }
            (void)cudaGetLastError();
        }
    }
    for (auto& r : bank->ranks) { NEO_TRY(bank_build_rank(bank.get(), r)); }
    NEO_TRY(bank_connect_inboxes(bank.get()));
    cudaSetDevice(before);
    *out = bank.release();
    return NEO_B200_OK;
}

int neo_b200_bank_create_rank(neo_b200_bank** out, neo_b200_conv_config const* config, neo_b200_bank_layout const* layout, int device,
                              int rank, int world, void const* unique_id)
{
    if (world < 1 || rank < 0 || rank >= world) { return fail(NEO_B200_ERR_INVALID, "bad rank %d of %d", rank, world); }
    std::unique_ptr<neo_b200_bank> bank;
    NEO_TRY(bank_common_create(out, config, layout, size_t(world), bank));
    bank->nccl = true;
    bank->ranks.resize(1);
    bank_rank& r = bank->ranks[0];
    bank_fill_info(bank->cfg, bank->layout, size_t(world), size_t(rank), device, &r.info);
    NEO_CUDA_TRY(cudaSetDevice(device));
    size_t const gp_n    = bank->layout.partition_shards;
    bool const matrix    = bank->cfg.topology == NEO_B200_MATRIX;
    bool const need_in   = matrix ? world > 1 : gp_n > 1;
    bool const need_out  = gp_n > 1;
    if (need_in || need_out) {
        if (unique_id == nullptr) { return fail(NEO_B200_ERR_INVALID, "this layout exchanges data between ranks: pass the id of neo_b200_bank_unique_id"); }
        bank->api = nccl_api::get();
        if (bank->api == nullptr) { return fail(NEO_B200_ERR_UNSUPPORTED, "NCCL (libnccl.so.2) could not be loaded"); }
        nccl_api::unique_id uid{};
        std::memcpy(&uid, unique_id, sizeof(uid));
        NEO_NCCL_TRY(bank->api, bank->api->CommInitRank(&r.comm_world, world, uid, rank));
        // separate communicators for the two collectives: they run on different streams and overlap across steps
        int const color = int(r.info.channel_group), key = int(r.info.partition_shard);
        if (need_in) {
            if (matrix) { r.comm_in = r.comm_world; }
            else { NEO_NCCL_TRY(bank->api, bank->api->CommSplit(r.comm_world, color, key, &r.comm_in, nullptr)); }
        }
        if (need_out) { NEO_NCCL_TRY(bank->api, bank->api->CommSplit(r.comm_world, color, key, &r.comm_out, nullptr)); }
    }
    NEO_TRY(bank_build_rank(bank.get(), r));
    NEO_TRY(bank_connect_inboxes(bank.get()));
    NEO_TRY(bank_connect_inputs(bank.get()));
    *out = bank.release();
    return NEO_B200_OK;
}

void neo_b200_bank_destroy(neo_b200_bank* bank)
{
    if (bank == nullptr) { return; }
    int before = 0;
    cudaGetDevice(&before);
    delete bank;
    cudaSetDevice(before);
}

int neo_b200_bank_local_ranks(neo_b200_bank const* bank, size_t* count)
{
    if (bank == nullptr || count == nullptr) { return fail(NEO_B200_ERR_INVALID, "null argument"); }
    *count = bank->ranks.size();
    return NEO_B200_OK;
}

int neo_b200_bank_local_rank(neo_b200_bank const* bank, size_t local_index, neo_b200_bank_rank_info* info)
{
    if (bank == nullptr || info == nullptr) { return fail(NEO_B200_ERR_INVALID, "null argument"); }
    if (local_index >= bank->ranks.size()) { return fail(NEO_B200_ERR_INVALID, "local rank %zu of %zu", local_index, bank->ranks.size()); }
    *info = bank->ranks[local_index].info;
    return NEO_B200_OK;
}

int neo_b200_bank_layout_info(neo_b200_conv_config const* config, neo_b200_bank_layout const* layout, size_t rank, neo_b200_bank_rank_info* info)
{
    if (config == nullptr || layout == nullptr || info == nullptr) { return fail(NEO_B200_ERR_INVALID, "null argument"); }
    neo_b200_conv_config c = *config;
    size_t const world     = layout->channel_groups * layout->partition_shards;
    NEO_TRY(bank_validate(c, *layout, world));
    if (rank >= world) { return fail(NEO_B200_ERR_INVALID, "rank %zu of %zu", rank, world); }
    bank_fill_info(c, *layout, world, rank, -1, info);
    return NEO_B200_OK;
}

static int bank_set_filters(neo_b200_bank* bank, void const* const* per_rank, size_t taps, int memspace, bool impulse)
{
    if (bank == nullptr || per_rank == nullptr) { return fail(NEO_B200_ERR_INVALID, "null argument"); }
    while (!bank->pending.empty()) { NEO_TRY(bank_wait_oldest(bank)); }
    int before = 0;
    cudaGetDevice(&before);
    for (size_t l = 0; l < bank->ranks.size(); ++l) {
        bank_rank& r = bank->ranks[l];
        if (per_rank[l] == nullptr) { return fail(NEO_B200_ERR_INVALID, "null filter pointer for local rank %zu", l); }
        NEO_CUDA_TRY(cudaSetDevice(r.info.device));
        if (impulse) { NEO_TRY(neo_b200_conv_set_impulse(r.conv, per_rank[l], taps, memspace)); }
        else { NEO_TRY(neo_b200_conv_set_filter(r.conv, per_rank[l], memspace)); }
    }
    cudaSetDevice(before);
    bank->has_filter = true;
    return neo_b200_bank_reset(bank);
}

int neo_b200_bank_set_impulse(neo_b200_bank* bank, void const* const* ir_per_rank, size_t taps, int memspace)
{
    return bank_set_filters(bank, ir_per_rank, taps, memspace, true);
}

int neo_b200_bank_set_filter(neo_b200_bank* bank, void const* const* h_per_rank, int memspace)
{
    return bank_set_filters(bank, h_per_rank, 0, memspace, false);
}

int neo_b200_bank_reset(neo_b200_bank* bank)
{
    if (bank == nullptr) { return fail(NEO_B200_ERR_INVALID, "null argument"); }
    while (!bank->pending.empty()) { NEO_TRY(bank_wait_oldest(bank)); }
    int before = 0;
    cudaGetDevice(&before);
    for (auto& r : bank->ranks) {
        NEO_CUDA_TRY(cudaSetDevice(r.info.device));
        for (cudaStream_t s : {r.s_in, r.s_cmp, r.s_red, r.s_out}) { NEO_CUDA_TRY(cudaStreamSynchronize(s)); }
        NEO_TRY(neo_b200_conv_reset(r.conv));
        NEO_TRY(neo_b200_conv_synchronize(r.conv));
        NEO_CUDA_TRY(cudaMemsetAsync(r.xring.ptr, 0, r.xring.bytes, r.s_in));
        // rank-per-process: nobody may push rows of the next step into this ring before it has been cleared -- every rank of the
        // gather domain passes this gate only after all of them have cleared theirs
        if (r.dma_in) {
            float* const words = r.gate_in.as<float>();
            size_t me          = 0;
            std::vector<size_t> gather;
            bank_domains(bank, r, &gather, nullptr);
            for (size_t i = 0; i < gather.size(); ++i) {
                if (gather[i] == size_t(r.info.rank)) { me = i; }
            }
            NEO_NCCL_TRY(bank->api, bank->api->AllGather(words + me, words, 1, nccl_api::k_float32, r.comm_in, r.s_in));
        }
        NEO_CUDA_TRY(cudaStreamSynchronize(r.s_in));
    }
    cudaSetDevice(before);
    bank->step = 0;
    return NEO_B200_OK;
}

int neo_b200_bank_submit(neo_b200_bank* bank, void const* const* in_rows, void* const* out_rows, size_t blocks, int memspace)
{
    NEO_TRY(bank_check_call(bank, in_rows, out_rows, blocks));
    while (bank->pending.size() >= size_t(k_bank_depth)) { NEO_TRY(bank_wait_oldest(bank)); }  // input ring and output staging are k_bank_depth deep
    int before = 0;
    cudaGetDevice(&before);
    int const status = bank->cfg.dtype == NEO_B200_F32 ? bank_submit_impl<float>(bank, in_rows, out_rows, blocks, memspace)
                                                       : bank_submit_impl<double>(bank, in_rows, out_rows, blocks, memspace);
    cudaSetDevice(before);
    return status;
}

int neo_b200_bank_wait(neo_b200_bank* bank)
{
    if (bank == nullptr) { return fail(NEO_B200_ERR_INVALID, "null argument"); }
    int before = 0;
    cudaGetDevice(&before);
    int const status = bank_wait_oldest(bank);
    cudaSetDevice(before);
    return status;
}

int neo_b200_bank_process(neo_b200_bank* bank, void const* const* in_rows, void* const* out_rows, size_t blocks, int memspace)
{
    NEO_TRY(neo_b200_bank_submit(bank, in_rows, out_rows, blocks, memspace));
    while (!bank->pending.empty()) { NEO_TRY(neo_b200_bank_wait(bank)); }
    return NEO_B200_OK;
}

int neo_b200_bank_timer_start(neo_b200_bank* bank)
{
    if (bank == nullptr) { return fail(NEO_B200_ERR_INVALID, "null argument"); }
    while (!bank->pending.empty()) { NEO_TRY(bank_wait_oldest(bank)); }
    int before = 0;
    cudaGetDevice(&before);
    for (auto& r : bank->ranks) {
        NEO_CUDA_TRY(cudaSetDevice(r.info.device));
        for (cudaStream_t s : {r.s_in, r.s_cmp, r.s_red, r.s_out}) { NEO_CUDA_TRY(cudaStreamSynchronize(s)); }
        NEO_CUDA_TRY(cudaEventRecord(r.t_begin, r.s_in));  // every step starts on the input stream
    }
    cudaSetDevice(before);
    return NEO_B200_OK;
}

int neo_b200_bank_timer_stop(neo_b200_bank* bank, double* ms)
{
    if (bank == nullptr || ms == nullptr) { return fail(NEO_B200_ERR_INVALID, "null argument"); }
    int before = 0;
    cudaGetDevice(&before);
    NEO_TRY(bank_finish_older(bank));  // the inverse side of the last step may still be waiting for a next submit
    for (auto& r : bank->ranks) {  // every step ends on the output stream: the event follows the last submitted step there
        NEO_CUDA_TRY(cudaSetDevice(r.info.device));
        NEO_CUDA_TRY(cudaEventRecord(r.t_end, r.s_out));
    }
    while (!bank->pending.empty()) { NEO_TRY(bank_wait_oldest(bank)); }
    *ms = 0.0;
    for (auto& r : bank->ranks) {
        NEO_CUDA_TRY(cudaSetDevice(r.info.device));
        NEO_CUDA_TRY(cudaEventSynchronize(r.t_end));
        float t = 0.f;
        NEO_CUDA_TRY(cudaEventElapsedTime(&t, r.t_begin, r.t_end));
        *ms = std::max(*ms, double(t));
    }
    cudaSetDevice(before);
    return NEO_B200_OK;
}

int neo_b200_bank_profile_enable(neo_b200_bank* bank, int enable)
{
    if (bank == nullptr) { return fail(NEO_B200_ERR_INVALID, "null argument"); }
    for (auto& r : bank->ranks) { NEO_TRY(neo_b200_conv_profile_enable(r.conv, enable)); }
    return NEO_B200_OK;
}

int neo_b200_bank_profile_read(neo_b200_bank* bank, size_t local_index, double* phase_ms, uint64_t* mac_launches)
{
    if (bank == nullptr || phase_ms == nullptr || mac_launches == nullptr) { return fail(NEO_B200_ERR_INVALID, "null argument"); }
    if (local_index >= bank->ranks.size()) { return fail(NEO_B200_ERR_INVALID, "local rank %zu of %zu", local_index, bank->ranks.size()); }
    while (!bank->pending.empty()) { NEO_TRY(bank_wait_oldest(bank)); }
    bank_rank& r = bank->ranks[local_index];
    int before   = 0;
    cudaGetDevice(&before);
    NEO_CUDA_TRY(cudaSetDevice(r.info.device));
    for (cudaStream_t s : {r.s_in, r.s_cmp, r.s_red, r.s_out}) { NEO_CUDA_TRY(cudaStreamSynchronize(s)); }
    int const status = with_engine(r.conv, [&](auto& e) { return e.read_profile(phase_ms, mac_launches, r.s_cmp); });
    cudaSetDevice(before);
    return status;
}

size_t neo_b200_bank_device_bytes(neo_b200_bank const* bank, size_t local_index)
{
    if (bank == nullptr || local_index >= bank->ranks.size()) { return 0; }
    bank_rank const& r = bank->ranks[local_index];
    return neo_b200_conv_device_bytes(r.conv) + r.xring.bytes + r.red[0].bytes + r.red[1].bytes + r.yout[0].bytes + r.yout[1].bytes + r.yout[2].bytes + r.inbox.bytes;
}

}  // extern "C"
