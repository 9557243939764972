// Launch plans: the whole raw-stream pass replayed from a file written by libs/modeling/plan.py (include/avdf.h,
// "the whole model"). The parser validates everything before it returns and makes no CUDA call; a session rebuilds every
// launch's arguments with relocated pointers and calls the same avdf_* entry point the Python path calls, so tensor maps
// and SM-count-dependent choices are made the same way.
//
// File format (little-endian, 64-bit sizes):
//   "AVDFPLAN" u32 format_version u32 abi_version
//   i32 cc_major cc_minor sm_count max_batch max_seg_num t_out in_dtype; i32 channels[3]; i64 stream_rows[3]; u64 batch_mask
//   u64 n, char description[n]
//   u64 n_allocs, per allocation: u32 kind u32 role u64 bytes u64 data_offset (constants: offset into the blob, 256-aligned)
//   u64 blob_bytes, blob (the constants' bytes, uploaded as one block: device offset = data_offset)
//   u64 n_lists, per list: u64 batch u64 n_launches, per launch: u32 name_len char name[] u32 n_args, per argument:
//     u32 tag u32 0, then by tag: I32 / I64: i64 | F32: u32 bits u32 0 | PTR: u64 alloc (NULL: ~0) u64 byte offset |
//     HOST_I32 / HOST_F32: u64 count, count * 4 bytes | STRUCT: u64 size, bytes, u64 n_relocs, per relocation:
//     u64 field_offset u64 alloc u64 offset (alloc HOST_REF: offset = byte count of a host array that follows) | STREAM
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <new>
#include <string>
#include <vector>

#include "common.cuh"

namespace {

constexpr char kMagic[8] = {'A', 'V', 'D', 'F', 'P', 'L', 'A', 'N'};
constexpr uint32_t kFormatVersion = 1;
constexpr uint64_t kNull = ~0ull, kHostRef = ~0ull - 1;
constexpr size_t kAlign = 256;
constexpr int kMaxBatch = 64;

enum Kind : uint32_t { KIND_CONST = 0, KIND_SCRATCH, KIND_INPUT, KIND_OUTPUT, KIND_WORKSPACE, KIND_N };
enum Role : uint32_t { ROLE_NONE = 0, ROLE_VIDEO, ROLE_BYOLA, ROLE_EMO, ROLE_OFFSETS, ROLE_META, ROLE_SEGS, ROLE_SCORES,
                       ROLE_COUNTS, ROLE_VCLS, ROLE_N };
enum Tag : uint32_t { TAG_I32 = 1, TAG_I64, TAG_F32, TAG_PTR, TAG_HOST_I32, TAG_HOST_F32, TAG_STRUCT, TAG_STREAM };
const char kTagChar[] = "?ILFPABST";

enum Op { OP_INTERP, OP_CONV_GEMM, OP_MLP_FUSED, OP_LN_DWCONV_LN, OP_ATTENTION, OP_LN_ROWS, OP_INSTNORM, OP_FPN_FUSE,
          OP_HEAD_FINAL, OP_HEAD_COMBINE, OP_VCLS12, OP_VCLS13, OP_POSTPROCESS, OP_N };

// Entry points a plan may call. sig: one character per argument (I int32, L int64, F float, P device pointer,
// A host int32 array, B host float array, S the entry point's args struct, T the stream). Host arrays hold exactly as
// many elements as the int32 argument `count_arg` says.
struct OpInfo {
  const char* name;
  const char* sig;
  size_t struct_size;
  int arrays[2][2];   // (array argument, count argument), -1 = none
};
const OpInfo kOps[OP_N] = {
    {"avdf_interp_concat_in", "PPPIPPPIIIIIPIT", 0, {{-1, -1}, {-1, -1}}},
    {"avdf_conv_gemm", "ST", sizeof(avdf_conv_gemm_args), {{-1, -1}, {-1, -1}}},
    {"avdf_mlp_fused", "ST", sizeof(avdf_mlp_fused_args), {{-1, -1}, {-1, -1}}},
    {"avdf_ln_dwconv_ln", "ST", sizeof(avdf_ln_dwconv_ln_args), {{-1, -1}, {-1, -1}}},
    {"avdf_attention", "PPPPPIIIIIIIIT", 0, {{-1, -1}, {-1, -1}}},
    {"avdf_ln_rows", "PPPPILIT", 0, {{-1, -1}, {-1, -1}}},
    {"avdf_instnorm_lrelu", "PPIIIIFT", 0, {{-1, -1}, {-1, -1}}},
    {"avdf_fpn_fuse", "PPPPPPIIIIAT", 0, {{10, 9}, {-1, -1}}},
    {"avdf_head_final", "PPIPPPPPBPPIIIAT", 0, {{8, 13}, {14, 13}}},
    {"avdf_head_combine", "PPPPPBPPIIAT", 0, {{5, 9}, {10, 9}}},
    {"avdf_vcls_exp12", "PIPPPPPPPIIIT", 0, {{-1, -1}, {-1, -1}}},
    {"avdf_vcls_exp13", "PIPPPPPPIIIT", 0, {{-1, -1}, {-1, -1}}},
    {"avdf_postprocess", "ST", sizeof(avdf_postprocess_args), {{-1, -1}, {-1, -1}}},
};

struct Reloc {
  uint64_t field, alloc, offset;
  std::vector<uint8_t> host;   // alloc == kHostRef
};
struct Arg {
  uint32_t tag = 0;
  int64_t i = 0;
  float f = 0.f;
  uint64_t alloc = kNull, offset = 0;
  std::vector<uint8_t> bytes;  // host array / struct
  std::vector<Reloc> relocs;
};
struct Launch {
  int op = -1;
  std::vector<Arg> args;
};
struct Alloc {
  uint32_t kind, role;
  uint64_t bytes, data_offset;
  uint64_t session_offset = 0;  // non-constants: offset inside a session arena
};

struct Reader {
  const uint8_t* p;
  size_t n, pos = 0;
  bool take(void* dst, size_t k) {
    if (k > n - pos) return false;
    memcpy(dst, p + pos, k);
    pos += k;
    return true;
  }
  bool u32(uint32_t& v) { return take(&v, 4); }
  bool u64(uint64_t& v) { return take(&v, 8); }
  bool i32(int32_t& v) { return take(&v, 4); }
  bool i64(int64_t& v) { return take(&v, 8); }
  bool bytes(std::vector<uint8_t>& v, uint64_t k) {
    if (k > n - pos) return false;
    v.assign(p + pos, p + pos + k);
    pos += k;
    return true;
  }
};

size_t align_up(size_t v) { return (v + kAlign - 1) / kAlign * kAlign; }

}  // namespace

struct avdf_plan {
  avdf_plan_info info{};
  std::vector<Alloc> allocs;
  std::vector<uint8_t> blob;
  std::vector<Launch> lists[kMaxBatch];
  int io[ROLE_N];                 // allocation of every io role, -1 if absent
  uint8_t* consts = nullptr;      // device copy of the blob (avdf_plan_upload)
  int device = -1;
};

struct avdf_session {
  const avdf_plan* plan;
  uint8_t* arena;
  int device;
  std::vector<std::vector<uint8_t>> structs[kMaxBatch];   // per launch: its args struct with relocated pointers
  cudaGraphExec_t graph[kMaxBatch] = {};
  // sliding windows (avdf_session_attach_windows): the caller's device block, the windowed graphs (first launch =
  // avdf_interp_concat_ranges on the fixed start / count arrays), the pinned parameter buffer and its copy's event
  uint8_t* win = nullptr;
  int32_t max_windows = 0, max_per_rec = 0;
  cudaGraphExec_t win_graph[kMaxBatch] = {};
  uint8_t* pinned = nullptr;
  cudaEvent_t copied = nullptr;
  float iou_threshold = 0.f, min_score = 0.f, sigma = 0.f, voting_thresh = 0.f;   // of the recorded avdf_postprocess
  int32_t use_soft_nms = 0;
};

namespace {

#define PLAN_FAIL(...)              \
  do {                              \
    avdf::set_error(__VA_ARGS__);   \
    return AVDF_ERR_INVALID;        \
  } while (0)
#define PLAN_READ(expr) \
  do {                  \
    if (!(expr)) PLAN_FAIL("avdf_plan_open: truncated file (%zu bytes, needed more at byte %zu)", rd.n, rd.pos); \
  } while (0)

int check_ref(const avdf_plan& p, uint64_t alloc, uint64_t offset, const char* op, const char* what, int index) {
  if (alloc == kNull) return AVDF_OK;
  if (alloc >= p.allocs.size())
    PLAN_FAIL("avdf_plan_open: %s %s %d: allocation %llu does not exist (%zu allocations)", op, what, index,
              (unsigned long long)alloc, p.allocs.size());
  if (offset >= p.allocs[alloc].bytes)
    PLAN_FAIL("avdf_plan_open: %s %s %d: relocation outside its allocation (offset %llu, allocation %llu of %llu bytes)",
              op, what, index, (unsigned long long)offset, (unsigned long long)alloc,
              (unsigned long long)p.allocs[alloc].bytes);
  return AVDF_OK;
}

// The only host pointer inside an args struct a plan carries: avdf_conv_gemm_args.tap_rows, `taps` int32 values.
int check_host_reloc(int op, const Arg& a, const Reloc& r) {
  if (op == OP_CONV_GEMM && r.field == offsetof(avdf_conv_gemm_args, tap_rows)) {
    avdf_conv_gemm_args g;
    memcpy(&g, a.bytes.data(), sizeof(g));
    if (g.taps >= 1 && g.taps <= AVDF_MAX_TAPS && r.host.size() == (size_t)g.taps * 4) return AVDF_OK;
    PLAN_FAIL("avdf_plan_open: avdf_conv_gemm tap_rows: %zu bytes for %d taps", r.host.size(), g.taps);
  }
  PLAN_FAIL("avdf_plan_open: %s: host array at struct offset %llu has no length rule", kOps[op].name,
            (unsigned long long)r.field);
}

int parse_launch(Reader& rd, avdf_plan& p, Launch& l) {
  uint32_t name_len = 0;
  PLAN_READ(rd.u32(name_len));
  std::vector<uint8_t> nm;
  PLAN_READ(name_len <= 128 && rd.bytes(nm, name_len));
  const std::string name(nm.begin(), nm.end());
  for (int o = 0; o < OP_N; ++o)
    if (name == kOps[o].name) l.op = o;
  if (l.op < 0) PLAN_FAIL("avdf_plan_open: unknown entry point '%s'", name.c_str());
  const OpInfo& op = kOps[l.op];
  uint32_t n_args = 0;
  PLAN_READ(rd.u32(n_args));
  if (n_args != strlen(op.sig)) PLAN_FAIL("avdf_plan_open: %s: %u arguments, expected %zu", op.name, n_args, strlen(op.sig));
  l.args.resize(n_args);
  for (uint32_t k = 0; k < n_args; ++k) {
    Arg& a = l.args[k];
    uint32_t pad = 0;
    PLAN_READ(rd.u32(a.tag) && rd.u32(pad));
    if (a.tag < TAG_I32 || a.tag > TAG_STREAM || kTagChar[a.tag] != op.sig[k])
      PLAN_FAIL("avdf_plan_open: %s argument %u: type tag %u, expected '%c'", op.name, k, a.tag, op.sig[k]);
    switch (a.tag) {
      case TAG_I32:
        PLAN_READ(rd.i64(a.i));
        if (a.i < INT32_MIN || a.i > INT32_MAX) PLAN_FAIL("avdf_plan_open: %s argument %u: int32 out of range", op.name, k);
        break;
      case TAG_I64: PLAN_READ(rd.i64(a.i)); break;
      case TAG_F32: {
        uint32_t bits = 0;
        PLAN_READ(rd.u32(bits) && rd.u32(pad));
        memcpy(&a.f, &bits, 4);
        break;
      }
      case TAG_PTR:
        PLAN_READ(rd.u64(a.alloc) && rd.u64(a.offset));
        if (int rc = check_ref(p, a.alloc, a.offset, op.name, "argument", (int)k)) return rc;
        break;
      case TAG_HOST_I32:
      case TAG_HOST_F32: {
        uint64_t count = 0;
        PLAN_READ(rd.u64(count));
        PLAN_READ(count <= 4096 && rd.bytes(a.bytes, count * 4));
        break;
      }
      case TAG_STRUCT: {
        uint64_t size = 0, n_rel = 0;
        PLAN_READ(rd.u64(size));
        if (size != op.struct_size)
          PLAN_FAIL("avdf_plan_open: %s: struct size %llu, sizeof its args struct is %zu", op.name, (unsigned long long)size,
                    op.struct_size);
        PLAN_READ(rd.bytes(a.bytes, size) && rd.u64(n_rel));
        PLAN_READ(n_rel <= size / 8);
        a.relocs.resize(n_rel);
        for (uint64_t r = 0; r < n_rel; ++r) {
          Reloc& rl = a.relocs[r];
          PLAN_READ(rd.u64(rl.field) && rd.u64(rl.alloc) && rd.u64(rl.offset));
          if (rl.field % 8 != 0 || rl.field + 8 > size)
            PLAN_FAIL("avdf_plan_open: %s relocation %llu: field offset %llu is not a pointer field", op.name,
                      (unsigned long long)r, (unsigned long long)rl.field);
          if (rl.alloc == kHostRef) {
            PLAN_READ(rl.offset <= 4096 && rd.bytes(rl.host, rl.offset));
            if (int rc = check_host_reloc(l.op, a, rl)) return rc;
          } else if (rl.alloc == kNull) {
            PLAN_FAIL("avdf_plan_open: %s relocation %llu: NULL", op.name, (unsigned long long)r);
          } else if (int rc = check_ref(p, rl.alloc, rl.offset, op.name, "relocation", (int)r)) {
            return rc;
          }
        }
        break;
      }
      default: break;   // TAG_STREAM: no payload
    }
  }
  for (const auto& ar : op.arrays) {
    if (ar[0] < 0) continue;
    const int64_t want = l.args[ar[1]].i;
    if (want < 1 || want > AVDF_MAX_LEVELS || (int64_t)l.args[ar[0]].bytes.size() != want * 4)
      PLAN_FAIL("avdf_plan_open: %s argument %d: host array of %zu elements, argument %d says %lld", op.name, ar[0],
                l.args[ar[0]].bytes.size() / 4, ar[1], (long long)want);
  }
  return AVDF_OK;
}

int parse(Reader& rd, avdf_plan& p) {
  char magic[8];
  PLAN_READ(rd.take(magic, 8));
  if (memcmp(magic, kMagic, 8) != 0) PLAN_FAIL("avdf_plan_open: bad magic (not a plan file)");
  uint32_t version = 0, abi = 0;
  PLAN_READ(rd.u32(version) && rd.u32(abi));
  if (version != kFormatVersion) PLAN_FAIL("avdf_plan_open: unsupported format version %u (this library reads %u)", version, kFormatVersion);
  if (abi != AVDF_ABI_VERSION) PLAN_FAIL("avdf_plan_open: plan recorded against ABI version %u, library is %d", abi, AVDF_ABI_VERSION);
  avdf_plan_info& in = p.info;
  in.abi_version = (int32_t)abi;
  PLAN_READ(rd.i32(in.cc_major) && rd.i32(in.cc_minor) && rd.i32(in.sm_count) && rd.i32(in.max_batch) &&
            rd.i32(in.max_seg_num) && rd.i32(in.t_out) && rd.i32(in.in_dtype));
  for (int s = 0; s < 3; ++s) PLAN_READ(rd.i32(in.channels[s]));
  for (int s = 0; s < 3; ++s) PLAN_READ(rd.i64(in.stream_rows[s]));
  PLAN_READ(rd.u64(in.batch_mask));
  if (in.max_batch < 1 || in.max_batch > kMaxBatch || in.max_seg_num < 1 || in.max_seg_num > AVDF_MAX_SEGS || in.t_out < 1 ||
      (in.in_dtype != AVDF_DTYPE_F32 && in.in_dtype != AVDF_DTYPE_BF16))
    PLAN_FAIL("avdf_plan_open: header out of range (max_batch %d, max_seg_num %d, t_out %d, in_dtype %d)", in.max_batch,
              in.max_seg_num, in.t_out, in.in_dtype);
  for (int s = 0; s < 3; ++s)
    if (in.channels[s] < 0 || in.stream_rows[s] < 0 || (in.channels[s] > 0) != (in.stream_rows[s] > 0) ||
        in.stream_rows[s] > INT32_MAX)
      PLAN_FAIL("avdf_plan_open: stream %d: %d channels, %lld rows", s, in.channels[s], (long long)in.stream_rows[s]);
  uint64_t desc_len = 0;
  std::vector<uint8_t> desc;
  PLAN_READ(rd.u64(desc_len));
  if (desc_len >= sizeof(in.description)) PLAN_FAIL("avdf_plan_open: description of %llu bytes", (unsigned long long)desc_len);
  PLAN_READ(rd.bytes(desc, desc_len));
  memcpy(in.description, desc.data(), desc_len);
  in.description[desc_len] = 0;

  uint64_t n_allocs = 0;
  PLAN_READ(rd.u64(n_allocs));
  PLAN_READ(n_allocs <= (rd.n - rd.pos) / 24);
  p.allocs.resize(n_allocs);
  for (auto& r : p.io) r = -1;
  for (uint64_t i = 0; i < n_allocs; ++i) {
    Alloc& a = p.allocs[i];
    PLAN_READ(rd.u32(a.kind) && rd.u32(a.role) && rd.u64(a.bytes) && rd.u64(a.data_offset));
    if (a.kind >= KIND_N || a.role >= ROLE_N || a.bytes == 0 || a.bytes > (1ull << 40))
      PLAN_FAIL("avdf_plan_open: allocation %llu: kind %u, role %u, %llu bytes", (unsigned long long)i, a.kind, a.role,
                (unsigned long long)a.bytes);
    if (a.role != ROLE_NONE) {
      const bool input = a.role <= ROLE_META;
      if (p.io[a.role] >= 0 || a.kind != (input ? KIND_INPUT : KIND_OUTPUT))
        PLAN_FAIL("avdf_plan_open: allocation %llu: role %u twice or with kind %u", (unsigned long long)i, a.role, a.kind);
      p.io[a.role] = (int)i;
    }
  }
  uint64_t blob_bytes = 0;
  PLAN_READ(rd.u64(blob_bytes));
  PLAN_READ(rd.bytes(p.blob, blob_bytes));
  size_t session = 0;
  for (uint64_t i = 0; i < n_allocs; ++i) {
    Alloc& a = p.allocs[i];
    if (a.kind == KIND_CONST) {
      if (a.data_offset % kAlign != 0 || a.data_offset > blob_bytes || a.bytes > blob_bytes - a.data_offset)
        PLAN_FAIL("avdf_plan_open: constant %llu: [%llu, +%llu) is outside the %llu-byte blob", (unsigned long long)i,
                  (unsigned long long)a.data_offset, (unsigned long long)a.bytes, (unsigned long long)blob_bytes);
    } else {
      a.session_offset = session;
      session += align_up(a.bytes);
    }
  }
  in.const_bytes = align_up(blob_bytes);
  in.session_bytes = session;

  // io allocations: present exactly where the header says, large enough for max_batch
  const int64_t B = in.max_batch, K = in.max_seg_num, es = in.in_dtype == AVDF_DTYPE_F32 ? 4 : 2;
  const int64_t need[ROLE_N] = {0, in.stream_rows[0] * in.channels[0] * es, in.stream_rows[1] * in.channels[1] * es,
                                in.stream_rows[2] * in.channels[2] * es, 3 * (B + 1) * 4, 4 * B * 4, B * K * 8, B * K * 4,
                                B * 4, B * 4};
  for (int r = ROLE_VIDEO; r < ROLE_N; ++r) {
    const bool want = r > ROLE_EMO || in.channels[r - ROLE_VIDEO] > 0;
    if (want != (p.io[r] >= 0) || (want && p.allocs[p.io[r]].bytes < (uint64_t)need[r]))
      PLAN_FAIL("avdf_plan_open: io role %d: %s (needs %lld bytes)", r, p.io[r] >= 0 ? "allocation too small or unexpected" : "missing",
                (long long)need[r]);
  }

  uint64_t n_lists = 0, mask = 0;
  PLAN_READ(rd.u64(n_lists));
  if (n_lists > (uint64_t)in.max_batch) PLAN_FAIL("avdf_plan_open: %llu launch lists for max_batch %d", (unsigned long long)n_lists, in.max_batch);
  for (uint64_t li = 0; li < n_lists; ++li) {
    uint64_t b = 0, n_launch = 0;
    PLAN_READ(rd.u64(b) && rd.u64(n_launch));
    if (b < 1 || b > (uint64_t)in.max_batch || (mask >> (b - 1) & 1))
      PLAN_FAIL("avdf_plan_open: launch list for batch %llu (max_batch %d, or listed twice)", (unsigned long long)b, in.max_batch);
    mask |= 1ull << (b - 1);
    PLAN_READ(n_launch <= (rd.n - rd.pos) / 8);
    auto& list = p.lists[b - 1];
    list.resize(n_launch);
    for (auto& l : list)
      if (int rc = parse_launch(rd, p, l)) return rc;
  }
  if (mask != in.batch_mask)
    PLAN_FAIL("avdf_plan_open: batch mask %#llx, launch lists for %#llx", (unsigned long long)in.batch_mask, (unsigned long long)mask);
  if (rd.pos != rd.n) PLAN_FAIL("avdf_plan_open: %zu trailing bytes", rd.n - rd.pos);
  return AVDF_OK;
}

void* resolve(const avdf_plan& p, const uint8_t* arena, uint64_t alloc, uint64_t offset) {
  if (alloc == kNull) return nullptr;
  const Alloc& a = p.allocs[alloc];
  return (void*)((a.kind == KIND_CONST ? p.consts + a.data_offset : arena + a.session_offset) + offset);
}

// One launch: the arguments rebuilt with this session's pointers, then the entry point Python's ops.py calls.
int call(const avdf_session& s, const Launch& l, const std::vector<uint8_t>& st_buf, cudaStream_t st) {
  const avdf_plan& p = *s.plan;
  void* P[16] = {};
  for (size_t k = 0; k < l.args.size(); ++k) {
    const Arg& a = l.args[k];
    if (a.tag == TAG_PTR) P[k] = resolve(p, s.arena, a.alloc, a.offset);
    else if (a.tag == TAG_HOST_I32 || a.tag == TAG_HOST_F32) P[k] = (void*)a.bytes.data();
    else if (a.tag == TAG_STRUCT) P[k] = (void*)st_buf.data();
  }
  auto I = [&](int k) { return (int32_t)l.args[k].i; };
  auto F = [&](int k) { return l.args[k].f; };
  auto fp = [&](int k) { return (float*)P[k]; };
  auto u8 = [&](int k) { return (uint8_t*)P[k]; };
  auto i32 = [&](int k) { return (int32_t*)P[k]; };
  switch (l.op) {
    case OP_INTERP:
      return avdf_interp_concat_in(P[0], P[1], P[2], I(3), i32(4), i32(5), i32(6), I(7), I(8), I(9), I(10), I(11), P[12], I(13), st);
    case OP_CONV_GEMM: return avdf_conv_gemm((const avdf_conv_gemm_args*)P[0], st);
    case OP_MLP_FUSED: return avdf_mlp_fused((const avdf_mlp_fused_args*)P[0], st);
    case OP_LN_DWCONV_LN: return avdf_ln_dwconv_ln((const avdf_ln_dwconv_ln_args*)P[0], st);
    case OP_ATTENTION:
      return avdf_attention(P[0], P[1], P[2], u8(3), P[4], I(5), I(6), I(7), I(8), I(9), I(10), I(11), I(12), st);
    case OP_LN_ROWS: return avdf_ln_rows(fp(0), fp(1), fp(2), P[3], I(4), l.args[5].i, I(6), st);
    case OP_INSTNORM: return avdf_instnorm_lrelu(fp(0), P[1], I(2), I(3), I(4), I(5), F(6), st);
    case OP_FPN_FUSE: return avdf_fpn_fuse(fp(0), u8(1), fp(2), fp(3), fp(4), P[5], I(6), I(7), I(8), I(9), i32(10), st);
    case OP_HEAD_FINAL:
      return avdf_head_final(P[0], P[1], I(2), u8(3), fp(4), fp(5), fp(6), fp(7), fp(8), fp(9), fp(10), I(11), I(12), I(13), i32(14), st);
    case OP_HEAD_COMBINE:
      return avdf_head_combine(fp(0), fp(1), u8(2), fp(3), fp(4), fp(5), fp(6), fp(7), I(8), I(9), i32(10), st);
    case OP_VCLS12: return avdf_vcls_exp12(P[0], I(1), fp(2), fp(3), fp(4), fp(5), fp(6), fp(7), fp(8), I(9), I(10), I(11), st);
    case OP_VCLS13: return avdf_vcls_exp13(P[0], I(1), fp(2), fp(3), fp(4), fp(5), fp(6), fp(7), I(8), I(9), I(10), st);
    case OP_POSTPROCESS: return avdf_postprocess((const avdf_postprocess_args*)P[0], st);
    default: break;
  }
  avdf::set_error("avdf_session_run: launch of unknown entry point %d", l.op);
  return AVDF_ERR_INVALID;
}

int run_list(const avdf_session& s, int batch, cudaStream_t st) {
  const auto& list = s.plan->lists[batch - 1];
  const auto& structs = s.structs[batch - 1];
  for (size_t i = 0; i < list.size(); ++i)
    if (int rc = call(s, list[i], structs[i], st)) return rc;
  return AVDF_OK;
}

// The first call for a list runs it eagerly on `st` (lazy per-device setup happens outside the capture), then captures it
// in thread-local mode; every call launches the graph.
template <class Run>
int launch_graph(cudaGraphExec_t& exec, Run run, cudaStream_t st, const char* who) {
  if (!exec) {
    if (int rc = run()) return rc;
    AVDF_CUDA(cudaStreamBeginCapture(st, cudaStreamCaptureModeThreadLocal));
    const int rc = run();
    cudaGraph_t g = nullptr;
    const cudaError_t e = cudaStreamEndCapture(st, &g);
    if (rc) {
      if (g) cudaGraphDestroy(g);
      return rc;
    }
    AVDF_CUDA(e);
    const cudaError_t ei = cudaGraphInstantiate(&exec, g, 0);
    cudaGraphDestroy(g);
    if (ei != cudaSuccess) {
      exec = nullptr;
      avdf::set_error("%s: cudaGraphInstantiate -> %s", who, cudaGetErrorString(ei));
      return AVDF_ERR_CUDA;
    }
  }
  AVDF_CUDA(cudaGraphLaunch(exec, st));
  return AVDF_OK;
}

// ---- sliding windows (libs/modeling/windows.py, the same double operations) ----
#define WIN_FAIL(code, ...)         \
  do {                              \
    avdf::set_error(__VA_ARGS__);   \
    return code;                    \
  } while (0)

// First stream of a window's meta: video if present, else byola, else emo.
int first_stream(const avdf_plan& p) { return p.info.channels[0] > 0 ? 0 : p.info.channels[1] > 0 ? 1 : 2; }

int check_window(const char* who, double W, double H) {
  if (!(W > 0)) WIN_FAIL(AVDF_ERR_INVALID, "%s: window must be > 0 seconds, got %g", who, W);
  if (!(H > 0 && H <= W)) WIN_FAIL(AVDF_ERR_INVALID, "%s: hop must satisfy 0 < hop <= window, got hop %g, window %g", who, H, W);
  return AVDF_OK;
}

// Number of windows of one recording (window_plan), after every check of its inputs.
int window_count(const avdf_plan& p, const char* who, double D, const int64_t rows[3], double W, double H, int64_t* n) {
  if (int rc = check_window(who, W, H)) return rc;
  if (!(D > 0) || !(D <= 1e300)) WIN_FAIL(AVDF_ERR_INVALID, "%s: duration must be a positive finite number of seconds, got %g", who, D);
  for (int s = 0; s < 3; ++s) {
    if (p.info.channels[s] == 0 && rows[s] != 0)
      WIN_FAIL(AVDF_ERR_INVALID, "%s: stream %d is absent from the plan but has %lld rows", who, s, (long long)rows[s]);
    if (p.info.channels[s] > 0 && (rows[s] < 1 || rows[s] > INT32_MAX))
      WIN_FAIL(AVDF_ERR_INVALID, "%s: stream %d is present in the plan but has %lld rows", who, s, (long long)rows[s]);
  }
  if (D <= W) {
    *n = 1;
    return AVDF_OK;
  }
  for (int s = 0; s < 3; ++s)
    if (p.info.channels[s] > 0 && floor(W * (double)rows[s] / D) < 1)
      WIN_FAIL(AVDF_ERR_INVALID, "%s: a %.3f s window of a %.3f s recording holds no row of stream %d (%lld rows)", who, W, D,
               s, (long long)rows[s]);
  const double k = ceil((D - W) / H);
  if (!(k < (double)(1 << 30)))
    WIN_FAIL(AVDF_ERR_INVALID, "%s: %.3f s in %g s hops of a %g s window is more than 2^30 windows", who, D, H, W);
  *n = (int64_t)k + 1;
  return AVDF_OK;
}

// The meta formula of avdf_session_run (streaming.video_meta with feat_stride = num_frames = 1).
void window_meta(const avdf_plan& p, int64_t T, double duration, float* m) {
  const double fs = (double)T / p.info.t_out;
  m[0] = (float)fs;
  m[1] = (float)(0.5 * fs);
  m[2] = (float)((double)T / duration);
  m[3] = (float)duration;
}

// Window k of n (window_count's n) of one recording: rows relative to the recording, meta, fp32 start.
void window_at(const avdf_plan& p, double D, const int64_t rows[3], double W, double H, int64_t n, int64_t k,
               int32_t start[3], int32_t count[3], float meta[4], float* win_start) {
  const int first = first_stream(p);
  if (D <= W) {
    for (int s = 0; s < 3; ++s) start[s] = 0, count[s] = (int32_t)rows[s];
    window_meta(p, rows[first], D, meta);
    *win_start = 0.f;
    return;
  }
  const double sk = std::min((double)k * H, D - W);
  for (int s = 0; s < 3; ++s) {
    const bool on = p.info.channels[s] > 0;
    start[s] = on ? (int32_t)floor(sk * (double)rows[s] / D) : 0;
    count[s] = on ? (int32_t)floor(W * (double)rows[s] / D) : 0;
  }
  window_meta(p, count[first], W, meta);
  *win_start = (float)sk;
}

// Can every launch list run windows? Its first launch is the CSR resampling reading the io offsets for its own batch size
// (replaced by the range form in the windowed list), and it has one postprocess writing the io outputs without records.
// Fills the NMS settings of the merge when `s` is given.
int check_windowable(const avdf_plan& p, const char* who, avdf_session* s) {
  const uint64_t off = (uint64_t)p.io[ROLE_OFFSETS];
  for (int b = 1; b <= p.info.max_batch; ++b) {
    if (!(p.info.batch_mask >> (b - 1) & 1)) continue;
    const auto& list = p.lists[b - 1];
    if (list.empty() || list[0].op != OP_INTERP)
      WIN_FAIL(AVDF_ERR_UNSUPPORTED, "%s: the launch list for batch %d does not start with avdf_interp_concat_in (it starts "
               "with %s)", who, b, list.empty() ? "nothing" : kOps[list[0].op].name);
    const Launch& in = list[0];
    for (int k = 0; k < 3; ++k) {
      const Arg& a = in.args[4 + k];
      if (p.info.channels[k] > 0 ? (a.alloc != off) : (a.alloc != kNull))
        WIN_FAIL(AVDF_ERR_UNSUPPORTED, "%s: batch %d: the resampling's stream %d offsets are not the io offsets", who, b, k);
    }
    if (in.args[7].i != b)
      WIN_FAIL(AVDF_ERR_UNSUPPORTED, "%s: batch %d: the resampling runs %lld recordings", who, b, (long long)in.args[7].i);
    const Launch* post = nullptr;
    for (const Launch& l : list)
      if (l.op == OP_POSTPROCESS) {
        if (post) WIN_FAIL(AVDF_ERR_UNSUPPORTED, "%s: batch %d: more than one avdf_postprocess", who, b);
        post = &l;
      }
    if (!post) WIN_FAIL(AVDF_ERR_UNSUPPORTED, "%s: batch %d: no avdf_postprocess", who, b);
    const Arg& a = post->args[0];
    avdf_postprocess_args pa;
    memcpy(&pa, a.bytes.data(), sizeof(pa));
    const struct { size_t field; int role; } outs[3] = {{offsetof(avdf_postprocess_args, out_segs), ROLE_SEGS},
                                                        {offsetof(avdf_postprocess_args, out_scores), ROLE_SCORES},
                                                        {offsetof(avdf_postprocess_args, out_count), ROLE_COUNTS}};
    for (const auto& o : outs) {
      bool ok = false;
      for (const Reloc& r : a.relocs) ok |= r.field == o.field && r.alloc == (uint64_t)p.io[o.role] && r.offset == 0;
      if (!ok) WIN_FAIL(AVDF_ERR_UNSUPPORTED, "%s: batch %d: avdf_postprocess does not write the io outputs", who, b);
    }
    for (const Reloc& r : a.relocs)
      if (r.field == offsetof(avdf_postprocess_args, rec_ring))
        WIN_FAIL(AVDF_ERR_UNSUPPORTED, "%s: batch %d: avdf_postprocess keeps result records", who, b);
    if (pa.use_soft_nms != 0 && !(pa.use_soft_nms == 1 && pa.soft_method == 2))
      WIN_FAIL(AVDF_ERR_UNSUPPORTED, "%s: batch %d: avdf_postprocess runs use_soft_nms %d (method %d); windows merge with hard "
               "or soft (method 2) NMS", who, b, pa.use_soft_nms, pa.soft_method);
    if (s) {
      s->iou_threshold = pa.iou_threshold, s->min_score = pa.min_score, s->sigma = pa.sigma;
      s->voting_thresh = pa.voting_thresh, s->use_soft_nms = pa.use_soft_nms;
    }
  }
  return AVDF_OK;
}

// The window block: byte offsets of its parts (avdf_session_window_bytes documents the sum).
struct WinBlock {
  size_t table, fixed, segs, scores, count, cls, ws, ws_bytes, total;
};
size_t table_bytes(const avdf_plan& p, int64_t W) { return 4 * (12 * W + 10 * (int64_t)p.info.max_batch); }
WinBlock win_block(const avdf_plan& p, int64_t W, int64_t per_rec) {
  const int64_t B = p.info.max_batch, K = p.info.max_seg_num;
  WinBlock w{};
  size_t o = 0;
  w.table = o, o += align_up(table_bytes(p, W));
  w.fixed = o, o += align_up(24 * B);
  w.segs = o, o += align_up(8 * K * W);
  w.scores = o, o += align_up(4 * K * W);
  w.count = o, o += align_up(4 * W);
  w.cls = o, o += align_up(4 * W);
  w.ws = o, w.ws_bytes = avdf_window_merge_workspace_bytes((int32_t)W, (int32_t)(K * per_rec));
  w.total = o + w.ws_bytes;
  return w;
}

int check_limits(const avdf_plan& p, const char* who, int32_t max_windows, int32_t per_rec) {
  if (max_windows < 1 || max_windows > (1 << 24) || per_rec < 1 || per_rec > max_windows)
    WIN_FAIL(AVDF_ERR_INVALID, "%s: need 1 <= max_windows_per_recording (%d) <= max_windows (%d) <= 2^24", who, per_rec,
             max_windows);
  if ((int64_t)per_rec * p.info.max_seg_num > INT32_MAX)
    WIN_FAIL(AVDF_ERR_INVALID, "%s: max_windows_per_recording %d * max_seg_num %d overflows int32", who, per_rec,
             p.info.max_seg_num);
  return AVDF_OK;
}

// Batch size whose list runs `b` windows: b itself when recorded, else the smallest recorded size above it.
int run_size(const avdf_plan& p, int b) {
  for (int r = b; r <= p.info.max_batch; ++r)
    if (p.info.batch_mask >> (r - 1) & 1) return r;
  return 0;
}

// The windowed list for batch B: the recorded list with its first launch as the range form, reading the fixed arrays.
int run_windowed_list(const avdf_session& s, int batch, cudaStream_t st) {
  const avdf_plan& p = *s.plan;
  const auto& list = p.lists[batch - 1];
  const Launch& l = list[0];
  void* P[3];
  for (int k = 0; k < 3; ++k) P[k] = resolve(p, s.arena, l.args[k].alloc, l.args[k].offset);
  const int32_t* start = (const int32_t*)(s.win + win_block(p, s.max_windows, s.max_per_rec).fixed);
  auto I = [&](int k) { return (int32_t)l.args[k].i; };
  if (int rc = avdf_interp_concat_ranges(P[0], P[1], P[2], I(3), start, start + 3 * batch, I(7), I(8), I(9), I(10), I(11),
                                         resolve(p, s.arena, l.args[12].alloc, l.args[12].offset), I(13), st))
    return rc;
  const auto& structs = s.structs[batch - 1];
  for (size_t i = 1; i < list.size(); ++i)
    if (int rc = call(s, list[i], structs[i], st)) return rc;
  return AVDF_OK;
}

}  // namespace

extern "C" int avdf_plan_open(const char* path, avdf_plan** out) {
  AVDF_CHECK_ARG(path != nullptr && out != nullptr, "path / out is NULL");
  *out = nullptr;
  FILE* f = fopen(path, "rb");
  if (!f) {
    avdf::set_error("avdf_plan_open: cannot open %s", path);
    return AVDF_ERR_INVALID;
  }
  std::vector<uint8_t> data;
  uint8_t chunk[1 << 16];
  size_t got;
  while ((got = fread(chunk, 1, sizeof(chunk), f)) > 0) data.insert(data.end(), chunk, chunk + got);
  const bool err = ferror(f) != 0;
  fclose(f);
  if (err) {
    avdf::set_error("avdf_plan_open: read error on %s", path);
    return AVDF_ERR_INVALID;
  }
  avdf_plan* p = new (std::nothrow) avdf_plan();
  if (!p) {
    avdf::set_error("avdf_plan_open: out of host memory");
    return AVDF_ERR_INVALID;
  }
  Reader rd{data.data(), data.size()};
  if (int rc = parse(rd, *p)) {
    delete p;
    return rc;
  }
  *out = p;
  return AVDF_OK;
}

extern "C" int avdf_plan_get_info(const avdf_plan* p, avdf_plan_info* info) {
  AVDF_CHECK_ARG(p != nullptr && info != nullptr, "plan / info is NULL");
  *info = p->info;
  return AVDF_OK;
}

extern "C" int avdf_plan_upload(avdf_plan* p, void* dev, size_t bytes, void* stream) {
  AVDF_CHECK_ARG(p != nullptr, "plan is NULL");
  AVDF_CHECK_ARG(p->consts == nullptr, "the plan's constants are already uploaded");
  AVDF_CHECK_ARG(bytes >= p->info.const_bytes && (p->info.const_bytes == 0 || dev != nullptr), "device block smaller than const_bytes");
  AVDF_CHECK_ARG((uintptr_t)dev % kAlign == 0, "device block is not 256-byte aligned");
  int32_t sms = 0, ccma = 0, ccmi = 0;
  if (int rc = avdf_device_info(&sms, &ccma, &ccmi)) return rc;
  if (sms != p->info.sm_count || ccma != p->info.cc_major || ccmi != p->info.cc_minor) {
    avdf::set_error("avdf_plan_upload: the plan was recorded on a device with compute capability %d.%d and %d SMs, this one "
                    "has %d.%d and %d SMs", p->info.cc_major, p->info.cc_minor, p->info.sm_count, ccma, ccmi, sms);
    return AVDF_ERR_UNSUPPORTED;
  }
  if (!p->blob.empty())
    AVDF_CUDA(cudaMemcpyAsync(dev, p->blob.data(), p->blob.size(), cudaMemcpyHostToDevice, (cudaStream_t)stream));
  p->consts = (uint8_t*)dev;
  p->device = avdf::current_device();
  return AVDF_OK;
}

extern "C" void avdf_plan_close(avdf_plan* p) { delete p; }

extern "C" int avdf_session_create(const avdf_plan* p, void* dev, size_t bytes, avdf_session** out) {
  AVDF_CHECK_ARG(p != nullptr && out != nullptr, "plan / out is NULL");
  *out = nullptr;
  AVDF_CHECK_ARG(p->consts != nullptr || p->info.const_bytes == 0, "the plan's constants are not uploaded (avdf_plan_upload)");
  AVDF_CHECK_ARG(dev != nullptr && bytes >= p->info.session_bytes, "device block smaller than session_bytes");
  AVDF_CHECK_ARG((uintptr_t)dev % kAlign == 0, "device block is not 256-byte aligned");
  AVDF_CHECK_ARG(avdf::current_device() == p->device, "the current device is not the one the constants were uploaded to");
  AVDF_CUDA(cudaMemset(dev, 0, p->info.session_bytes));
  AVDF_CUDA(cudaDeviceSynchronize());
  avdf_session* s = new (std::nothrow) avdf_session();
  if (!s) {
    avdf::set_error("avdf_session_create: out of host memory");
    return AVDF_ERR_INVALID;
  }
  s->plan = p;
  s->arena = (uint8_t*)dev;
  s->device = p->device;
  for (int b = 0; b < kMaxBatch; ++b) {
    for (const Launch& l : p->lists[b]) {
      std::vector<uint8_t> st;
      for (const Arg& a : l.args) {
        if (a.tag != TAG_STRUCT) continue;
        st = a.bytes;
        for (const Reloc& r : a.relocs) {
          const void* v = r.alloc == kHostRef ? (const void*)r.host.data() : resolve(*p, s->arena, r.alloc, r.offset);
          memcpy(st.data() + r.field, &v, 8);
        }
      }
      s->structs[b].push_back(std::move(st));
    }
  }
  *out = s;
  return AVDF_OK;
}

extern "C" int avdf_session_get_io(const avdf_session* s, avdf_session_io* io) {
  AVDF_CHECK_ARG(s != nullptr && io != nullptr, "session / io is NULL");
  const avdf_plan& p = *s->plan;
  auto at = [&](int role) { return p.io[role] < 0 ? nullptr : resolve(p, s->arena, (uint64_t)p.io[role], 0); };
  for (int k = 0; k < 3; ++k) io->streams[k] = at(ROLE_VIDEO + k);
  io->offsets = (int32_t*)at(ROLE_OFFSETS);
  io->meta = (float*)at(ROLE_META);
  io->segs = (float*)at(ROLE_SEGS);
  io->scores = (float*)at(ROLE_SCORES);
  io->counts = (int32_t*)at(ROLE_COUNTS);
  io->video_cls = (float*)at(ROLE_VCLS);
  return AVDF_OK;
}

extern "C" int avdf_session_run(avdf_session* s, int32_t batch, const int64_t rows[3], void* stream) {
  AVDF_CHECK_ARG(s != nullptr && rows != nullptr, "session / rows is NULL");
  const avdf_plan& p = *s->plan;
  if (batch < 1 || batch > p.info.max_batch || !(p.info.batch_mask >> (batch - 1) & 1)) {
    avdf::set_error("avdf_session_run: the plan has no launch list for batch size %d (batch mask %#llx)", batch,
                    (unsigned long long)p.info.batch_mask);
    return AVDF_ERR_INVALID;
  }
  for (int k = 0; k < 3; ++k)
    if (rows[k] < 0 || rows[k] > p.info.stream_rows[k]) {
      avdf::set_error("avdf_session_run: stream %d: %lld rows, the staging holds %lld", k, (long long)rows[k],
                      (long long)p.info.stream_rows[k]);
      return AVDF_ERR_INVALID;
    }
  AVDF_CHECK_ARG(stream != nullptr, "stream is the legacy default stream (graph capture needs a created stream)");
  AVDF_CHECK_ARG(avdf::current_device() == s->device, "the current device is not the plan's");
  cudaStream_t st = (cudaStream_t)stream;
  return launch_graph(s->graph[batch - 1], [&] { return run_list(*s, batch, st); }, st, "avdf_session_run");
}

extern "C" void avdf_session_destroy(avdf_session* s) {
  if (!s) return;
  for (auto& g : s->graph)
    if (g) cudaGraphExecDestroy(g);
  for (auto& g : s->win_graph)
    if (g) cudaGraphExecDestroy(g);
  if (s->copied) {
    cudaEventSynchronize(s->copied);         // the last call's parameter copy still reads the pinned buffer
    cudaEventDestroy(s->copied);
  }
  if (s->pinned) cudaFreeHost(s->pinned);
  delete s;
}

// ---- sliding windows ----
extern "C" int32_t avdf_plan_window_layout(const avdf_plan* p, double duration, const int64_t rows[3], double window,
                                           double hop, int32_t cap, int32_t* start, int32_t* count, float* meta,
                                           float* win_start) {
  AVDF_CHECK_ARG(p != nullptr && rows != nullptr, "plan / rows is NULL");
  int64_t n = 0;
  if (int rc = window_count(*p, "avdf_plan_window_layout", duration, rows, window, hop, &n)) return rc;
  if (n > INT32_MAX) WIN_FAIL(AVDF_ERR_INVALID, "avdf_plan_window_layout: %lld windows", (long long)n);
  if (cap >= n && start && count && meta && win_start)
    for (int64_t k = 0; k < n; ++k)
      window_at(*p, duration, rows, window, hop, n, k, start + 3 * k, count + 3 * k, meta + 4 * k, win_start + k);
  return (int32_t)n;
}

extern "C" size_t avdf_session_window_bytes(const avdf_plan* p, int32_t max_windows, int32_t max_windows_per_recording) {
  if (!p) {
    avdf::set_error("avdf_session_window_bytes: plan is NULL");
    return 0;
  }
  if (check_limits(*p, "avdf_session_window_bytes", max_windows, max_windows_per_recording) ||
      check_windowable(*p, "avdf_session_window_bytes", nullptr))
    return 0;
  return win_block(*p, max_windows, max_windows_per_recording).total;
}

extern "C" int avdf_session_attach_windows(avdf_session* s, void* dev, size_t bytes, int32_t max_windows,
                                           int32_t max_windows_per_recording) {
  AVDF_CHECK_ARG(s != nullptr, "session is NULL");
  AVDF_CHECK_ARG(s->win == nullptr, "the session already has a window block");
  const avdf_plan& p = *s->plan;
  const char* who = "avdf_session_attach_windows";
  if (int rc = check_limits(p, who, max_windows, max_windows_per_recording)) return rc;
  if (int rc = check_windowable(p, who, s)) return rc;
  AVDF_CHECK_ARG(dev != nullptr && bytes >= win_block(p, max_windows, max_windows_per_recording).total,
                 "device block smaller than avdf_session_window_bytes");
  AVDF_CHECK_ARG((uintptr_t)dev % kAlign == 0, "device block is not 256-byte aligned");
  AVDF_CHECK_ARG(avdf::current_device() == s->device, "the current device is not the plan's");
  AVDF_CUDA(cudaHostAlloc((void**)&s->pinned, table_bytes(p, max_windows), cudaHostAllocDefault));
  const cudaError_t e = cudaEventCreateWithFlags(&s->copied, cudaEventDisableTiming);
  if (e != cudaSuccess) {
    cudaFreeHost(s->pinned);
    s->pinned = nullptr, s->copied = nullptr;
    WIN_FAIL(AVDF_ERR_CUDA, "%s: cudaEventCreateWithFlags -> %s", who, cudaGetErrorString(e));
  }
  s->win = (uint8_t*)dev;
  s->max_windows = max_windows, s->max_per_rec = max_windows_per_recording;
  return AVDF_OK;
}

extern "C" int avdf_session_run_windows(avdf_session* s, const avdf_window_run_args* a, void* stream) {
  AVDF_CHECK_ARG(s != nullptr && a != nullptr, "session / args is NULL");
  const char* who = "avdf_session_run_windows";
  if (!s->win) WIN_FAIL(AVDF_ERR_INVALID, "%s: the session has no window block (avdf_session_attach_windows)", who);
  if (a->n_rec < 1) WIN_FAIL(AVDF_ERR_INVALID, "%s: n_rec is %d, needs >= 1 recording", who, a->n_rec);
  AVDF_CHECK_ARG(a->duration && a->rows && a->out_segs && a->out_scores && a->out_count && a->out_cls,
                 "duration / rows / an output is NULL");
  const avdf_plan& p = *s->plan;
  const int R = a->n_rec;
  std::vector<int64_t> n_win(R);
  int64_t total_win = 0, most = 0, total_rows[3] = {0, 0, 0};
  for (int r = 0; r < R; ++r) {
    const int64_t* rows = a->rows + 3 * r;
    if (int rc = window_count(p, who, a->duration[r], rows, a->window, a->hop, &n_win[r])) return rc;
    if (n_win[r] > s->max_per_rec)
      WIN_FAIL(AVDF_ERR_INVALID, "%s: recording %d has %lld windows, the window block holds %d per recording", who, r,
               (long long)n_win[r], s->max_per_rec);
    total_win += n_win[r], most = std::max(most, n_win[r]);
    for (int k = 0; k < 3; ++k) total_rows[k] += rows[k];
  }
  if (total_win > s->max_windows)
    WIN_FAIL(AVDF_ERR_INVALID, "%s: %lld windows, the window block holds %d", who, (long long)total_win, s->max_windows);
  for (int k = 0; k < 3; ++k)
    if (total_rows[k] > p.info.stream_rows[k])
      WIN_FAIL(AVDF_ERR_INVALID, "%s: stream %d: %lld rows, the staging holds %lld", who, k, (long long)total_rows[k],
               (long long)p.info.stream_rows[k]);
  AVDF_CHECK_ARG(stream != nullptr, "stream is the legacy default stream (graph capture needs a created stream)");
  AVDF_CHECK_ARG(avdf::current_device() == s->device, "the current device is not the plan's");
  cudaStream_t st = (cudaStream_t)stream;

  // ---- the table: per batch [start 3B | count 3B | meta 4B] (B = the size its list runs), then win_start, rec_win
  int step = 0;
  for (int b = p.info.max_batch; b >= 1 && !step; --b)
    if (p.info.batch_mask >> (b - 1) & 1) step = b;
  struct Batch { int64_t u0; int b, run; size_t word; };
  std::vector<Batch> batches;
  size_t words = 0;
  for (int64_t u0 = 0; u0 < total_win; u0 += step) {
    const int b = (int)std::min<int64_t>(step, total_win - u0);
    const int run = run_size(p, b);
    batches.push_back({u0, b, run, words});
    words += 10 * (size_t)run;
  }
  const size_t ws_word = words, rw_word = words + total_win, used = 4 * (rw_word + R + 1);
  AVDF_CUDA(cudaEventSynchronize(s->copied));       // the previous call's copy has read the buffer
  int32_t* wi = (int32_t*)s->pinned;
  float* wf = (float*)s->pinned;
  int64_t u = 0, row0[3] = {0, 0, 0};          // window index; first row of the recording in each stream's staging
  for (int r = 0; r < R; ++r) {
    const int64_t* rows = a->rows + 3 * r;
    wi[rw_word + r] = (int32_t)u;
    for (int64_t k = 0; k < n_win[r]; ++k, ++u) {
      const Batch& bt = batches[u / step];
      int32_t sa[3], ca[3];
      float m[4];
      window_at(p, a->duration[r], rows, a->window, a->hop, n_win[r], k, sa, ca, m, &wf[ws_word + u]);
      const int j0 = (int)(u - bt.u0), j1 = j0 + 1 == bt.b ? bt.run : j0 + 1;   // the batch's last window fills its unused slots
      for (int j = j0; j < j1; ++j) {
        for (int q = 0; q < 3; ++q) {
          wi[bt.word + q * bt.run + j] = (int32_t)(row0[q] + sa[q]);
          wi[bt.word + (3 + q) * bt.run + j] = ca[q];
        }
        for (int q = 0; q < 4; ++q) wf[bt.word + (6 + q) * bt.run + j] = m[q];
      }
    }
    for (int q = 0; q < 3; ++q) row0[q] += rows[q];
  }
  wi[rw_word + R] = (int32_t)u;
  const WinBlock wb = win_block(p, s->max_windows, s->max_per_rec);
  uint8_t* table = s->win + wb.table;
  AVDF_CUDA(cudaMemcpyAsync(table, s->pinned, used, cudaMemcpyHostToDevice, st));
  AVDF_CUDA(cudaEventRecord(s->copied, st));

  // ---- the windows, batch by batch; every window's results set aside
  avdf_session_io io;
  avdf_session_get_io(s, &io);
  const int64_t K = p.info.max_seg_num;
  float* w_segs = (float*)(s->win + wb.segs);
  float* w_scores = (float*)(s->win + wb.scores);
  int32_t* w_count = (int32_t*)(s->win + wb.count);
  float* w_cls = (float*)(s->win + wb.cls);
  for (const Batch& bt : batches) {
    const uint8_t* blk = table + 4 * bt.word;
    AVDF_CUDA(cudaMemcpyAsync(s->win + wb.fixed, blk, 24 * (size_t)bt.run, cudaMemcpyDeviceToDevice, st));
    AVDF_CUDA(cudaMemcpyAsync(io.meta, blk + 24 * (size_t)bt.run, 16 * (size_t)bt.run, cudaMemcpyDeviceToDevice, st));
    const int run = bt.run;
    if (int rc = launch_graph(s->win_graph[run - 1], [&] { return run_windowed_list(*s, run, st); }, st, who)) return rc;
    AVDF_CUDA(cudaMemcpyAsync(w_segs + bt.u0 * K * 2, io.segs, 8 * K * bt.b, cudaMemcpyDeviceToDevice, st));
    AVDF_CUDA(cudaMemcpyAsync(w_scores + bt.u0 * K, io.scores, 4 * K * bt.b, cudaMemcpyDeviceToDevice, st));
    AVDF_CUDA(cudaMemcpyAsync(w_count + bt.u0, io.counts, 4 * (size_t)bt.b, cudaMemcpyDeviceToDevice, st));
    AVDF_CUDA(cudaMemcpyAsync(w_cls + bt.u0, io.video_cls, 4 * (size_t)bt.b, cudaMemcpyDeviceToDevice, st));
  }

  // ---- one result per recording
  avdf_window_merge_args m{};
  m.n_rec = R;
  m.rec_win = (const int32_t*)(table + 4 * rw_word);
  m.win_start = (const float*)(table + 4 * ws_word);
  m.win_segs = w_segs, m.win_scores = w_scores, m.win_count = w_count, m.win_cls = w_cls;
  m.cand_cap = (int32_t)(K * most);
  m.iou_threshold = s->iou_threshold, m.min_score = s->min_score, m.sigma = s->sigma, m.voting_thresh = s->voting_thresh;
  m.max_seg_num = (int32_t)K, m.use_soft_nms = s->use_soft_nms;
  m.out_segs = a->out_segs, m.out_scores = a->out_scores, m.out_count = a->out_count, m.out_cls = a->out_cls;
  m.workspace = s->win + wb.ws, m.workspace_bytes = avdf_window_merge_workspace_bytes(R, m.cand_cap);
  return avdf_window_merge(&m, stream);
}
