// hcj_api.cu — the C ABI of libhcjpeg (include/hcjpeg.h): contexts, batches, orchestration.
//
// Host work per image is what the model does before its block loop (Header.decode + init); everything
// else is queued on the context's CUDA stream.  No CPU fallback exists: if CUDA is unavailable every
// compute entry point fails with HCJ_ERR_CUDA - cudaError.
#include <cuda_runtime.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <chrono>
#include <map>
#include <new>
#include <string>
#include <thread>
#include <vector>

#include "../../include/hcjpeg.h"
#include "hcj_host.h"
#include "hcj_internal.h"
#include "hcj_kernels.cuh"


using hcj::align_up;

struct hcj_batch {
  int n = 0, mode = 0;
  unsigned flags = 0;
  std::vector<HcjImageDesc> descs;
  std::vector<int> host_status;
  std::vector<size_t> out_bytes;
  std::vector<void *> owned;  // device allocations
  hcjk::DecodeBatchDev dev;
  size_t coef_bytes = 0;
  int kernels = 0;
  std::vector<uint32_t> list_restart, list_spec;  // host copies (sorted by image index) for chunked launches
  std::vector<uint32_t> tile_base;                // [n + 1] first IDCT tile of every image in the batch tile plan
};

// output modes produced by the Planar_444 kernel from the padded planes
static inline bool post_444(int mode) { return mode == HCJ_OUT_RGB24 || mode == HCJ_OUT_YUV444; }

extern "C" {

int hcj_version(void) { return HCJ_VERSION; }

const char *hcj_strerror(int status) {
  switch (status) {
    case HCJ_OK: return "ok";
    case HCJ_ERR_UNSUPPORTED_MARKER: return "unsupported marker code";
    case HCJ_ERR_NO_DC_CODE: return "Can't find dc code";
    case HCJ_ERR_NO_AC_CODE: return "Can't find ac code";
    case HCJ_ERR_COEF_INDEX: return "coefficient index out of range:";
    case HCJ_ERR_NO_COMPONENT: return "unable to find component identifier";
    case HCJ_ERR_NO_QUANT_TABLE: return "unable to find quantisation table";
    case HCJ_ERR_NO_HUFFMAN_TABLE: return "unable to find huffman table";
    case HCJ_ERR_NO_FRAME_OR_SCAN: return "From start of frame or start of scan marker";
    case HCJ_ERR_BITS_OUT_OF_BOUNDS: return "Bitstream_reader out of bounds";
    case HCJ_ERR_PLANE_BOUNDS: return "[Plane.get/set] out of bounds";
    case HCJ_ERR_FRAME_INFER: return "Could not infer chroma subsampling";
    case HCJ_ERR_NEED_3_COMPONENTS: return "index out of bounds (get_yuv_frame needs 3 components)";
    case HCJ_ERR_ENCODER_PARAMS: return "invalid encoder parameters";
    case HCJ_ERR_NO_TERMINATOR: return "no marker terminates the entropy-coded segment (the model would not return)";
    case HCJ_ERR_RESTART_COUNT: return "restart marker count does not match the restart interval";
    case HCJ_ERR_UNSUPPORTED_GEOMETRY: return "outside the supported domain (components / sampling factors / DC category / Pq)";
    case HCJ_ERR_DC_RANGE: return "resolved DC does not fit int16";
    case HCJ_ERR_TRUNCATED: return "truncated header (the model would not return)";
    case HCJ_ERR_BAD_HUFFMAN_TABLE: return "index out of bounds (over-subscribed Huffman table)";
    case HCJ_ERR_BUFFER_TOO_SMALL: return "output buffer too small";
    case HCJ_ERR_INVALID_ARG: return "invalid argument";
    case HCJ_ERR_OUT_OF_MEMORY: return "out of device memory";
    default: break;
  }
  if (status <= HCJ_ERR_CUDA) return cudaGetErrorString((cudaError_t)(HCJ_ERR_CUDA - status));
  return "unknown status";
}

int hcj_header_decode(const uint8_t *jpeg, size_t len, hcj_header *out) { return hcj_header_decode_ex(jpeg, len, 0u, out); }

int hcj_header_decode_ex(const uint8_t *jpeg, size_t len, unsigned flags, hcj_header *out) {
  if (!jpeg || !out) return HCJ_ERR_INVALID_ARG;
  return hcj::header_decode(jpeg, len, out, flags);
}

int hcj_frame_info_get(const uint8_t *jpeg, size_t len, hcj_frame_info *out) {
  return hcj_frame_info_get_ex(jpeg, len, HCJ_FLAG_DEFAULT, out);
}

int hcj_frame_info_get_ex(const uint8_t *jpeg, size_t len, unsigned flags, hcj_frame_info *out) {
  if (!jpeg || !out) return HCJ_ERR_INVALID_ARG;
  hcj_header *h = new (std::nothrow) hcj_header;
  if (!h) return HCJ_ERR_OUT_OF_MEMORY;
  int st = hcj::header_decode(jpeg, len, h, flags);
  hcj::ImagePlan plan;
  if (st == HCJ_OK) st = hcj::plan_image(*h, flags, &plan);
  if (st == HCJ_OK) *out = plan.info;
  delete h;
  return st;
}

int hcj_ctx_create(int device, void *cuda_stream, hcj_ctx **out) {
  if (!out) return HCJ_ERR_INVALID_ARG;
  *out = nullptr;
  CU_TRY(cudaSetDevice(device));
  hcj_ctx *c = new (std::nothrow) hcj_ctx;
  if (!c) return HCJ_ERR_OUT_OF_MEMORY;
  c->device = device;
  {
    const int ce = hcjk::configure_device(&c->sm_count);
    if (ce != 0) {
      delete c;
      return HCJ_ERR_CUDA - ce;
    }
  }
  if (cuda_stream) {
    c->stream = (cudaStream_t)cuda_stream;
  } else {
    cudaError_t e = cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking);
    if (e != cudaSuccess) {
      delete c;
      return HCJ_ERR_CUDA - (int)e;
    }
    c->own_stream = true;
  }
  cudaEventCreate(&c->ev0);
  cudaEventCreate(&c->ev1);
  cudaEventCreate(&c->enc0);
  cudaEventCreate(&c->enc1);
  cudaStreamCreateWithFlags(&c->copy_stream, cudaStreamNonBlocking);
  cudaStreamCreateWithFlags(&c->up_stream, cudaStreamNonBlocking);
  *out = c;
  return HCJ_OK;
}

void hcj_ctx_destroy(hcj_ctx *c) {
  if (!c) return;
  cudaSetDevice(c->device);
  cudaStreamSynchronize(c->stream);
  for (auto &f : c->pool) cudaFree(f.p);
  if (c->ev0) cudaEventDestroy(c->ev0);
  if (c->ev1) cudaEventDestroy(c->ev1);
  if (c->enc0) cudaEventDestroy(c->enc0);
  if (c->enc1) cudaEventDestroy(c->enc1);
  for (cudaEvent_t e : c->chunk_events) cudaEventDestroy(e);
  if (c->copy_stream) cudaStreamDestroy(c->copy_stream);
  if (c->up_stream) cudaStreamDestroy(c->up_stream);
  free(c->hdr_buf);
  for (cudaEvent_t ev : c->up_events) cudaEventDestroy(ev);
  if (c->own_stream) cudaStreamDestroy(c->stream);
  delete c;
}

int hcj_ctx_synchronize(hcj_ctx *c) {
  if (!c) return HCJ_ERR_INVALID_ARG;
  CU_TRY(cudaStreamSynchronize(c->stream));
  return HCJ_OK;
}

void *hcj_host_alloc(size_t bytes) {
  void *p = nullptr;
  if (cudaHostAlloc(&p, bytes ? bytes : 1, cudaHostAllocDefault) != cudaSuccess) {
    (void)cudaGetLastError();
    return nullptr;
  }
  return p;
}
void hcj_host_free(void *p) {
  if (p) cudaFreeHost(p);
}

int hcj_timer_start(hcj_ctx *c) {
  if (!c) return HCJ_ERR_INVALID_ARG;
  CU_TRY(cudaEventRecord(c->ev0, c->stream));
  return HCJ_OK;
}
int hcj_timer_stop(hcj_ctx *c, float *ms) {
  if (!c || !ms) return HCJ_ERR_INVALID_ARG;
  CU_TRY(cudaEventRecord(c->ev1, c->stream));
  CU_TRY(cudaEventSynchronize(c->ev1));
  CU_TRY(cudaEventElapsedTime(ms, c->ev0, c->ev1));
  return HCJ_OK;
}

// ------------------------------------------------------------------------------------------------
// decode
// ------------------------------------------------------------------------------------------------
static int batch_alloc(hcj_ctx *c, hcj_batch *b, void **p, size_t bytes) {
  int st = c->alloc(p, bytes);
  if (st == HCJ_OK) b->owned.push_back(*p);
  return st;
}

void hcj_batch_destroy(hcj_ctx *c, hcj_batch *b) {
  if (!b) return;
  if (c) {
    cudaSetDevice(c->device);
    cudaStreamSynchronize(c->stream);
    for (void *p : b->owned) c->release(p);
  }
  delete b;
}

// Copies the compressed files of images [lo, hi) to the device on `s`, merging images that are adjacent in
// host memory with matching padding into one copy.
static cudaError_t upload_files(const hcj_batch *b, const uint8_t *const *jpeg, const size_t *len, int lo, int hi,
                                cudaStream_t s) {
  cudaError_t e = cudaSuccess;
  uint8_t *d_files = const_cast<uint8_t *>(b->dev.files);
  for (int i = lo; i < hi && e == cudaSuccess;) {
    if (!b->descs[i].valid) {
      i++;
      continue;
    }
    int j = i;
    size_t bytes = len[i];
    while (j + 1 < hi && b->descs[j + 1].valid && jpeg[j + 1] == jpeg[i] + (b->descs[j + 1].file_off - b->descs[i].file_off)) {
      j++;
      bytes = (size_t)(b->descs[j].file_off - b->descs[i].file_off) + len[j];
    }
    e = cudaMemcpyAsync(d_files + b->descs[i].file_off, jpeg[i], bytes, cudaMemcpyHostToDevice, s);
    i = j + 1;
  }
  return e;
}

static int batch_create(hcj_ctx *c, const uint8_t *const *jpeg, const size_t *len, int n, int mode, unsigned flags,
                        int *status, hcj_batch **out, bool with_files) {
  if (!c || !out || n < 0 || n > HCJ_MAX_BATCH || (n > 0 && (!jpeg || !len)) || mode < 0 || mode > HCJ_OUT_YUV444 ||
      ((flags & HCJ_FLAG_LIBJPEG) && (flags & HCJ_FLAG_SCALE_MASK)))
    return HCJ_ERR_INVALID_ARG;
  *out = nullptr;
  CU_TRY(cudaSetDevice(c->device));
  hcj_batch *b = new (std::nothrow) hcj_batch;
  if (!b) return HCJ_ERR_OUT_OF_MEMORY;
  const bool trace = getenv("HCJ_TRACE") != nullptr;
  const auto t0 = std::chrono::steady_clock::now();
  auto mark = [&](const char *what) {
    if (trace)
      fprintf(stderr, "[batch_create]     %-28s %8.3f ms\n", what,
              std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count());
  };
  b->n = n;
  b->mode = mode;
  b->flags = flags;
  b->descs.assign(n, HcjImageDesc());
  b->host_status.assign(n, HCJ_OK);
  b->out_bytes.assign(n, 0);
  memset(&b->dev, 0, sizeof(b->dev));

  std::vector<HcjTableSet> table_sets;
  std::vector<uint16_t> prim_pool, full_pool;
  std::vector<int32_t> qt_pool;
  std::map<std::string, uint32_t> set_index;
  std::vector<uint32_t> list_restart, list_spec;
  size_t file_bytes = 0, ent_bytes = 0, nsegs = 0, out_total = 0, plane_total = 0;
  uint64_t total_blocks = 0;
  uint32_t total_tiles = 0;
  uint32_t max_segments = 0, max_tiles = 0, max_rows = 0, max_width = 0, max_sub_chunks = 0;
  size_t total_sub = 0, total_ds_tiles = 0;
  uint32_t max_ds_tiles = 0, max_blocks = 0, max_deferred = 0;
  uint32_t sub_log2 = 12;  // measured on 1080p q75: 1024 -> 11.0 ms, 2048 -> 9.4 ms, 4096 -> 8.9 ms for the four K3 kernels
  bool sub_log2_env = false, spec_has_units = false;
  uint64_t long_ri_blocks = 128;  // 4:2:0: intervals of 22 MCUs and more
  if (const char *e = getenv("HCJ_LONG_RI_BLOCKS")) long_ri_blocks = (uint64_t)std::max(1, atoi(e));  // tuning / test knob
  uint32_t guess_bits = 2048;
  if (const char *e = getenv("HCJ_GUESS_BITS")) guess_bits = (uint32_t)std::max(64, atoi(e));
  if (const char *e = getenv("HCJ_SUB_LOG2")) {  // tuning knob: preferred subsequence length, log2 of bits
    sub_log2 = (uint32_t)std::min(15, std::max(8, atoi(e)));
    sub_log2_env = true;
  }
  const int tile_mcus = HCJ_IDCT_THREADS;  // upper bound on MCUs per IDCT tile (one thread per block)
  const int scale_log = hcj::scale_log2(flags);  // every image of the batch is decoded at 1 / 2^scale_log (plan_image sizes it)
  const bool libjpeg = (flags & HCJ_FLAG_LIBJPEG) != 0;  // every image of the batch is reconstructed as libjpeg does
  // Decoder.Header.decode + the geometry of Decoder.init for every image: independent per image, so spread over
  // a few host threads (it is the serial prologue of every batch: 6 ms single-threaded for 1024 files)
  if (c->hdr_cap < (size_t)std::max(n, 1) * sizeof(hcj_header)) {
    free(c->hdr_buf);
    c->hdr_cap = (size_t)std::max(n, 1) * sizeof(hcj_header);
    c->hdr_buf = malloc(c->hdr_cap);
    if (!c->hdr_buf) {
      c->hdr_cap = 0;
      delete b;
      return HCJ_ERR_OUT_OF_MEMORY;
    }
  }
  hcj_header *hdrs = static_cast<hcj_header *>(c->hdr_buf);
  std::vector<hcj::ImagePlan> plans;
  std::vector<int> parse_st;
  try {
    plans.resize(std::max(n, 1));
    parse_st.assign(std::max(n, 1), HCJ_OK);
  } catch (const std::bad_alloc &) {
    delete b;
    return HCJ_ERR_OUT_OF_MEMORY;
  }
  {
    auto work = [&](int lo, int hi) {
      for (int i = lo; i < hi; i++) {
        int st = (jpeg[i] && len[i] < 0xfffffff0u) ? hcj::header_decode(jpeg[i], len[i], &hdrs[i], flags, false) : HCJ_ERR_INVALID_ARG;
        if (st == HCJ_OK) st = hcj::plan_image(hdrs[i], flags, &plans[i]);
        // bit positions inside a scan are 32-bit on the device: scans of 512 MiB and more are outside the domain
        if (st == HCJ_OK && len[i] - std::min<size_t>(len[i], (size_t)hdrs[i].scan_byte_pos) >= ((size_t)1 << 29)) st = HCJ_ERR_UNSUPPORTED_GEOMETRY;
        parse_st[i] = st;
      }
    };
    const int nthreads = std::max(1, std::min({(int)std::thread::hardware_concurrency(), 8, n / 64}));
    if (nthreads <= 1) {
      work(0, n);
    } else {
      std::vector<std::thread> pool;
      const int per = (n + nthreads - 1) / nthreads;
      for (int t = 1; t < nthreads; t++) pool.emplace_back(work, std::min(n, t * per), std::min(n, (t + 1) * per));
      work(0, std::min(n, per));
      for (auto &th : pool) th.join();
    }
  }
  mark("headers parsed");
  try {
    qt_pool.reserve((size_t)n * 3 * 128);
  } catch (const std::bad_alloc &) {
    delete b;
    return HCJ_ERR_OUT_OF_MEMORY;
  }
  int prev_pairs = -1, prev_pair_dc[HCJ_MAX_COMPONENTS], prev_pair_ac[HCJ_MAX_COMPONENTS], prev_img = -1;

  for (int i = 0; i < n; i++) {
    HcjImageDesc &d = b->descs[i];
    memset(&d, 0, sizeof(d));
    const hcj_header *h = &hdrs[i];
    const hcj::ImagePlan &plan = plans[i];
    int st = parse_st[i];
    const hcj_frame_info &f = plan.info;
    // table set of this image: one (dc, ac) pair per distinct binding among its scan components
    int pair_of[HCJ_MAX_COMPONENTS] = {0, 0, 0, 0}, npairs = 0, pair_dc[HCJ_MAX_COMPONENTS], pair_ac[HCJ_MAX_COMPONENTS];
    std::string key;
    if (st == HCJ_OK) {
      for (int k = 0; k < f.ncomp; k++) {
        int p = -1;
        for (int j = 0; j < npairs; j++)
          if (pair_dc[j] == plan.dc_index[k] && pair_ac[j] == plan.ac_index[k]) p = j;
        if (p < 0) {
          p = npairs++;
          pair_dc[p] = plan.dc_index[k];
          pair_ac[p] = plan.ac_index[k];
        }
        pair_of[k] = p;
      }
      // same tables as the previous image (the usual case in a batch): same table set, no key to build
      bool same_as_prev = prev_img >= 0 && prev_pairs == npairs;
      for (int p = 0; same_as_prev && p < npairs; p++)
        same_as_prev = memcmp(&h->huffman_tables[pair_dc[p]], &hdrs[prev_img].huffman_tables[prev_pair_dc[p]], sizeof(hcj_dht)) == 0 &&
                       memcmp(&h->huffman_tables[pair_ac[p]], &hdrs[prev_img].huffman_tables[prev_pair_ac[p]], sizeof(hcj_dht)) == 0;
      if (!same_as_prev)
        for (int p = 0; p < npairs; p++)
          for (int which = 0; which < 2; which++) {
            const hcj_dht &t = h->huffman_tables[which ? pair_ac[p] : pair_dc[p]];
            key.push_back((char)t.table_class);
            for (int q = 0; q < 16; q++) key.push_back((char)t.lengths[q]);
            key.append(reinterpret_cast<const char *>(t.values), (size_t)t.nvalues);
          }
      auto it = same_as_prev ? set_index.end() : set_index.find(key);
      if (same_as_prev) {
        d.table_set = b->descs[prev_img].table_set;
      } else if (it != set_index.end()) {
        d.table_set = it->second;
      } else {
        HcjTableSet ts;
        memset(&ts, 0, sizeof(ts));
        ts.npairs = (uint32_t)npairs;
        ts.primary_off = (uint32_t)prim_pool.size();
        std::vector<uint16_t> prim_local, full_local;
        for (int p = 0; p < npairs && st == HCJ_OK; p++)
          for (int which = 0; which < 2 && st == HCJ_OK; which++) {
            hcj::HuffLut lut;
            st = hcj::build_lut(h->huffman_tables[which ? pair_ac[p] : pair_dc[p]], &lut);
            if (st != HCJ_OK) break;
            ts.meta[p][which].max_bits = (uint32_t)lut.max_bits;
            ts.meta[p][which].full_off = (uint32_t)(full_pool.size() + full_local.size());
            prim_local.insert(prim_local.end(), lut.primary.begin(), lut.primary.end());
            full_local.insert(full_local.end(), lut.full.begin(), lut.full.end());
            while (full_local.size() % 8) full_local.push_back(0);
          }
        if (st == HCJ_OK) {
          prim_pool.insert(prim_pool.end(), prim_local.begin(), prim_local.end());
          full_pool.insert(full_pool.end(), full_local.begin(), full_local.end());
          d.table_set = (uint32_t)table_sets.size();
          set_index[key] = d.table_set;
          table_sets.push_back(ts);
        }
      }
      if (st == HCJ_OK) {
        prev_img = i;
        prev_pairs = npairs;
        for (int p = 0; p < npairs; p++) prev_pair_dc[p] = pair_dc[p], prev_pair_ac[p] = pair_ac[p];
      }
    }
    if (st == HCJ_OK && (mode == HCJ_OUT_YUV || post_444(mode))) {
      if (f.ncomp < 3) st = HCJ_ERR_NEED_3_COMPONENTS;  // decoder.ml:415-420
      // jdsample.c: integral ratios of 3-component frames (4-component ones would be CMYK / YCCK to libjpeg)
      else if (libjpeg && post_444(mode)) st = f.ncomp == 3 && plan.up_integral ? HCJ_OK : HCJ_ERR_UNSUPPORTED_GEOMETRY;
      else if (f.chroma == 0) st = HCJ_ERR_FRAME_INFER;  // frame.ml:44,55
    }
    b->host_status[i] = st;
    if (st != HCJ_OK) continue;

    d.valid = 1;
    d.file_off = file_bytes;
    d.file_len = (uint32_t)len[i];
    d.scan_start = (uint32_t)h->scan_byte_pos;
    if (d.scan_start > d.file_len) d.scan_start = d.file_len;
    file_bytes += align_up(len[i] + 16, 16);
    d.ds_off = (uint32_t)total_ds_tiles;
    {
      const uint32_t base0 = d.scan_start & ~15u;
      const uint32_t nt = d.file_len > base0 ? (d.file_len - base0 + 4095) / 4096 : 0;
      total_ds_tiles += nt;
      max_ds_tiles = std::max(max_ds_tiles, nt);
    }
    d.ent_off = ent_bytes;
    d.ent_cap = (uint32_t)align_up(len[i] - d.scan_start + 32, 16);
    ent_bytes += d.ent_cap;
    d.ncomp = f.ncomp;
    d.bpm = f.blocks_per_mcu;
    d.mcus_wide = f.mcus_wide;
    d.mcus_high = f.mcus_high;
    d.nmcu = (uint32_t)(f.mcus_wide * f.mcus_high);
    d.nblocks = (uint32_t)f.nblocks;
    d.ri = (uint32_t)f.restart_interval;
    d.nseg_expected = d.ri ? (d.nmcu + d.ri - 1) / d.ri : 1;
    d.seg_off = (uint32_t)nsegs;
    nsegs += d.nseg_expected + 1;
    d.coef_off = total_blocks;
    total_blocks += d.nblocks;
    d.chroma = f.chroma;
    d.width = f.width;
    d.height = f.height;
    d.qt_off = (uint32_t)qt_pool.size();
    size_t out_i = mode == HCJ_OUT_YUV ? f.yuv_bytes : mode == HCJ_OUT_PLANES ? f.planes_bytes : f.rgb_bytes;
    d.out_off = out_total;
    d.out_bytes = out_i;
    b->out_bytes[i] = out_i;
    out_total += align_up(out_i, 256);
    size_t plane_acc = 0, yuv_acc = 0;
    int first_blk = 0;
    for (int k = 0; k < f.ncomp; k++) {
      HcjCompGeom &g = d.comp[k];
      g.hs = f.hs[k];
      g.vs = f.vs[k];
      // The colour kernels read the scratch planes of RGB24 / YUV444 output in 8-byte words: their rows start 8-byte aligned.
      // Full-size planes are multiples of 8 wide already; scaled ones (8 / s samples per block) get a wider pitch there.
      g.decoded_w = post_444(mode) ? (int32_t)align_up((size_t)f.decoded_width[k], 8) : f.decoded_width[k];
      g.decoded_h = f.decoded_height[k];
      g.actual_w = f.actual_width[k];
      g.actual_h = f.actual_height[k];
      g.pair = pair_of[k];
      g.qt = k;
      g.first_blk = first_blk;
      if (libjpeg && post_444(mode)) g.up_h = (uint8_t)plan.up_h[k], g.up_v = (uint8_t)plan.up_v[k];
      first_blk += g.hs * g.vs;
      g.plane_off = (post_444(mode) ? plane_total : 0) + plane_acc;
      plane_acc += (size_t)g.decoded_w * g.decoded_h;
      g.out_off = yuv_acc;
      yuv_acc += (size_t)g.actual_w * g.actual_h;
      const hcj_dqt &q = h->quant_tables[plan.qt_index[k]];
      const size_t q0 = qt_pool.size();
      qt_pool.resize(q0 + 128);
      int32_t *qp = qt_pool.data() + q0;
      for (int e = 0; e < 64; e++) {
        qp[e] = (int32_t)q.elements[e];  // plain values, used by the 64-bit path
        if (q.elements[e] > 255) d.wide_idct = 1;
        // "dp2a form" used by the 32-bit path (see HCJ_QD in hcj_device.cuh)
        qp[64 + e] = (e & 1) ? (int32_t)(q.elements[e] & 0xff) << 8 : (int32_t)(q.elements[e] & 0xff);
      }
    }
    if (post_444(mode)) plane_total += align_up(plane_acc, 256);
    for (int k = 0; k < f.blocks_per_mcu && k < HCJ_MAX_BPM; k++) {
      d.blk_comp[k] = (uint8_t)plan.blk_comp[k];
      d.blk_bx[k] = (uint8_t)plan.blk_bx[k];
      d.blk_by[k] = (uint8_t)plan.blk_by[k];
    }
    // Restart intervals of at least `long_ri_blocks` blocks (two or more subsequences each) are decoded like scans
    // without markers, every interval a unit of the speculative decoder; shorter ones by one thread each (K2).
    if (d.ri && (uint64_t)d.ri * (uint64_t)d.bpm < long_ri_blocks) {
      list_restart.push_back((uint32_t)i);
      max_segments = std::max(max_segments, d.nseg_expected);
    } else {
      list_spec.push_back((uint32_t)i);
      if (d.ri) spec_has_units = true;
      // subsequences of 2^sub_log2 bits: long enough for the decoder to resynchronise inside one almost always
      // (a couple of MCUs), short enough for one thread each to fill the GPU
      // measured: 4096 bits for 65-bit blocks (1080p q75: 7.8 ms vs 8.0 ms at 8192), 8192 bits for 175-bit blocks
      // (4k 4:4:4 q95: 11.5 ms vs 12.9 ms at 4096): the per-subsequence work is per block, not per bit
      const uint64_t est_bits = (uint64_t)(d.file_len - d.scan_start) * 8;  // upper bound of the destuffed length
      // round 2 (one synchronisation pass with a 2048-bit warm-up in front of every subsequence, exact pass on whole MCUs):
      // longer subsequences pay less warm-up per bit and leave the lanes of the exact pass more alike: 1080p q75 K3
      // 5.80 / 5.25 / 4.88 / 5.73 ms at 2048 / 4096 / 8192 / 16384 bits (profiles/r02_experiments/r03f_*), so 8192 from 2 Mbit up
      const uint32_t s0 = sub_log2_env ? 1u << sub_log2 : ((est_bits > (uint64_t)d.nblocks * 120 || est_bits >= (1ull << 21)) ? 8192u : 4096u);
      // ... and cut so that the subsequences fill whole CTAs of the exact pass (512 threads): 1080p q75 has ~800
      // subsequences of 4096 bits, i.e. a second CTA with 44 % of its lanes idle; 1024 of ~3150 bits keep all busy.
      // (The count is bounded from above here: one subsequence beyond the last full CTA would cost a CTA of its own.)
      const uint64_t ctas = std::max<uint64_t>(1, (est_bits + 256ull * s0) / (512ull * s0));
      const uint64_t extra = d.nseg_expected > 1 ? d.nseg_expected : 0;  // every unit ends with a partial subsequence
      const uint64_t slots = 512 * ctas > 2 * extra ? 512 * ctas - extra : 512 * ctas;
      uint64_t sb = (est_bits + slots - 1) / slots;
      sb = (sb + 31) & ~31ull;
      d.sub_bits = (uint32_t)std::min<uint64_t>(32768, std::max<uint64_t>(sb, s0 / 2));
      d.sub_off = (uint32_t)total_sub;
      const size_t nsub_max = (size_t)((est_bits + d.sub_bits - 1) / d.sub_bits) + (size_t)extra + 1;
      total_sub += nsub_max + 1;
      max_sub_chunks = std::max(max_sub_chunks, (uint32_t)((nsub_max - 1 + 255) / 256));
    }
    int tm_max = std::max(1, std::min(tile_mcus, HCJ_IDCT_THREADS / d.bpm));
    uint32_t tiles = (uint32_t)((d.mcus_wide + tm_max - 1) / tm_max) * (uint32_t)d.mcus_high;
    max_tiles = std::max(max_tiles, tiles);
    d.idct_tile_off = total_tiles;
    d.idct_tiles = tiles;
    total_tiles += tiles;
    max_rows = std::max(max_rows, (uint32_t)f.height);
    {
      bool unit_sampling = f.ncomp == 3;
      for (int k = 0; k < f.ncomp; k++) unit_sampling = unit_sampling && f.hs[k] == 1 && f.vs[k] == 1;
      // scaled images (HCJ_FLAG_SCALE_*) are never fused: their tiles hold k x k samples per block, K9 converts their planes
      // nor are libjpeg reconstructions (HCJ_FLAG_LIBJPEG): the fused tiles hold the model's transform
      const bool fusable = mode == HCJ_OUT_RGB24 && f.ncomp == 3 && !d.wide_idct && !scale_log && !libjpeg && !getenv("HCJ_NO_FUSED_RGB");
      // sub-sampled: luma 2x2 or 2x1, chroma 1x1, even size (the chroma planes are exactly half)
      const bool sub = f.ncomp == 3 && f.hs[0] == 2 && f.hs[1] == 1 && f.hs[2] == 1 && f.vs[1] == 1 && f.vs[2] == 1 &&
                       ((f.chroma == 420 && f.vs[0] == 2 && f.height % 2 == 0) || (f.chroma == 422 && f.vs[0] == 1)) && f.width % 2 == 0;
      // Measured on 1024 x 1080p 4:2:0 (profiles/r02s_*): fused 4.89 ms + 0.64 ms for the deferred units against
      // 2.20 + 2.39 ms for k_idct_persistent + k_rgb_sub_pairs.  Both forms are bound by the instructions of the
      // conversion (about 24 per pixel: interpolation, four multiply-adds, shifts, saturating packs), which fusing does
      // not remove, and the deferred units cost more than the plane round trip saves: the two-kernel form stays the
      // default for sub-sampled images; HCJ_FUSED_SUB=1 selects the fused one.
      d.fused_rgb = !fusable ? 0 : (f.chroma == 444 && unit_sampling) ? 1 : (sub && getenv("HCJ_FUSED_SUB")) ? 2 : 0;
    }
    if (d.fused_rgb == 1) b->dev.has_fused = 1;
    else if (d.fused_rgb == 2) {
      b->dev.has_fused_sub = 1;
      // what k_rgb_deferred enumerates: a pixel row per MCU row with a chroma row below it, 16 pixels per row and tile boundary
      const uint32_t tm_max_i = (uint32_t)std::max(1, std::min(tile_mcus, HCJ_IDCT_THREADS / d.bpm));
      const uint32_t tpr = ((uint32_t)d.mcus_wide + tm_max_i - 1) / tm_max_i;
      const uint32_t def_rows = f.vs[0] == 2 ? (uint32_t)(f.actual_height[1] - 1) / 8 : 0;
      max_deferred = std::max(max_deferred, def_rows * (((uint32_t)f.width + 15) / 16) + (tpr - 1) * (uint32_t)f.height);
    }
    else if (f.chroma == 444) b->dev.has_444 = 1;  // 4:4:4 needs no up-sampling: libjpeg's copy is Planar_444's
    else if (libjpeg && post_444(mode)) d.libjpeg = 1, b->dev.has_libjpeg = 1;
    else b->dev.has_subsampled |= ((f.width & 1) || (f.chroma == 420 && (f.height & 1))) ? 2 : 1;
    max_blocks = std::max(max_blocks, d.nblocks);
    max_width = std::max(max_width, (uint32_t)f.width);
  }
  if (status)
    for (int i = 0; i < n; i++) status[i] = b->host_status[i];

  mark("descriptors and tables built");
  // ---- device buffers
  hcjk::DecodeBatchDev &dv = b->dev;
  int st = HCJ_OK;
  void *p = nullptr;
#define BALLOC(field, type, bytes)                          \
  if (st == HCJ_OK) {                                       \
    st = batch_alloc(c, b, &p, (bytes));                    \
    dv.field = reinterpret_cast<type>(p);                   \
  }
  HcjImageDesc *d_descs = nullptr;
  uint8_t *d_files = nullptr;
  HcjTableSet *d_sets = nullptr;
  uint16_t *d_prim = nullptr, *d_full = nullptr;
  int32_t *d_qt = nullptr;
  uint32_t *d_lr = nullptr, *d_ls = nullptr;
  if (st == HCJ_OK) st = batch_alloc(c, b, (void **)&d_descs, sizeof(HcjImageDesc) * std::max(n, 1));
  if (st == HCJ_OK) st = batch_alloc(c, b, (void **)&d_files, file_bytes + 16);
  if (st == HCJ_OK) st = batch_alloc(c, b, (void **)&d_sets, sizeof(HcjTableSet) * std::max<size_t>(table_sets.size(), 1));
  if (st == HCJ_OK) st = batch_alloc(c, b, (void **)&d_prim, 2 * std::max<size_t>(prim_pool.size(), 8));
  if (st == HCJ_OK) st = batch_alloc(c, b, (void **)&d_full, 2 * std::max<size_t>(full_pool.size(), 8));
  if (st == HCJ_OK) st = batch_alloc(c, b, (void **)&d_qt, 4 * std::max<size_t>(qt_pool.size(), 8));
  if (st == HCJ_OK) st = batch_alloc(c, b, (void **)&d_lr, 4 * std::max<size_t>(list_restart.size(), 1));
  if (st == HCJ_OK) st = batch_alloc(c, b, (void **)&d_ls, 4 * std::max<size_t>(list_spec.size(), 1));
  BALLOC(states, HcjImageState *, sizeof(HcjImageState) * std::max(n, 1));
  BALLOC(entropy, uint8_t *, ent_bytes + 64);  // + slack: the fast readers prefetch up to 16 bytes past the data
  BALLOC(seg_offs, uint32_t *, 4 * (nsegs + 1));
  BALLOC(ds_tiles, hcjk::DsTile *, 8 * (total_ds_tiles + 1));
  if (!list_spec.empty()) {
    BALLOC(sub_start, uint16_t *, 2 * total_sub + 16);
    BALLOC(seg_sub, uint32_t *, 4 * (nsegs + 1));
    BALLOC(sub_end2, uint16_t *, 2 * total_sub + 16);
    BALLOC(sub_first, uint32_t *, 4 * total_sub + 16);
    BALLOC(sub_nstart, int32_t *, 4 * total_sub + 16);
    BALLOC(sub_blk, int32_t *, 4 * total_sub + 16);
    BALLOC(sub_dc, int4 *, 16 * total_sub + 16);
    BALLOC(sub_dpre, int4 *, 16 * total_sub + 16);
    BALLOC(sub_list, uint32_t *, 4 * total_sub + 16);
  }
  b->coef_bytes = (size_t)total_blocks * 128;
  BALLOC(coefs, int16_t *, b->coef_bytes + 16);
  BALLOC(wide_flags, uint32_t *, (size_t)(total_blocks / 32 + 2) * 4 + 64);  // + slack: k_idct stages 48 bytes per tile
  BALLOC(out, uint8_t *, out_total + 16);
  BALLOC(idct_plan, hcjk::IdctTile *, hcjk::idct_plan_bytes(total_tiles));
  if (post_444(mode)) BALLOC(planes, uint8_t *, plane_total + 16);
#undef BALLOC
  mark("device buffers");
  if (st != HCJ_OK) {
    hcj_batch_destroy(c, b);
    return st;
  }
  dv.total_blocks = total_blocks;
  {
    int tm = hcjk::make_coef_tensor_map(&dv);
    if (tm != 0) {
      hcj_batch_destroy(c, b);
      return HCJ_ERR_CUDA - tm;
    }
  }
  dv.n = n;
  dv.sm_count = c->sm_count;
  dv.descs = d_descs;
  dv.files = d_files;
  dv.table_sets = d_sets;
  dv.lut_primary = d_prim;
  dv.lut_full = d_full;
  dv.qtables = d_qt;
  dv.list_restart = d_lr;
  dv.n_restart = (int)list_restart.size();
  dv.max_segments = max_segments;
  dv.max_pairs = 1;
  for (const HcjTableSet &ts : table_sets) dv.max_pairs = std::max(dv.max_pairs, ts.npairs);
  dv.list_spec = d_ls;
  dv.n_spec = (int)list_spec.size();
  dv.max_sub_chunks = max_sub_chunks;
  dv.spec_guess_bits = guess_bits;
  dv.spec_has_units = spec_has_units ? 1 : 0;
  dv.max_ds_tiles = max_ds_tiles;
  dv.total_ds_tiles = (uint32_t)total_ds_tiles;
  dv.max_idct_tiles = max_tiles;
  dv.total_idct_tiles = total_tiles;
  dv.tile_lo = 0;
  dv.tile_hi = total_tiles;
  b->tile_base.assign((size_t)n + 1, 0);
  for (int i = 0; i < n; i++) b->tile_base[i + 1] = b->tile_base[i] + b->descs[i].idct_tiles;
  dv.tile_mcus = tile_mcus;
  dv.block_k = 8 >> scale_log;
  dv.islow = libjpeg ? 1 : 0;
  dv.max_rgb_rows = max_rows;
  dv.max_blocks = max_blocks;
  dv.max_deferred_groups = max_deferred;
  dv.max_width = max_width;
  dv.total_blocks = total_blocks;
  dv.img_lo = 0;
  dv.img_hi = (uint32_t)n;
  dv.lr_lo = 0;
  dv.lr_hi = (uint32_t)list_restart.size();
  dv.ls_lo = 0;
  dv.ls_hi = (uint32_t)list_spec.size();
  b->list_restart = list_restart;
  b->list_spec = list_spec;
  b->kernels = hcjk::destuff_kernel_count() + (dv.n_restart ? 1 : 0) + (dv.n_spec ? hcjk::huff_spec_kernel_count(dv) : 0) + hcjk::idct_kernel_count() + (post_444(mode) ? dv.has_444 + (mode == HCJ_OUT_RGB24 ? (dv.has_subsampled & 1) + (dv.has_subsampled >> 1) + dv.has_fused + dv.has_fused_sub : (dv.has_subsampled ? 1 : 0)) + dv.has_libjpeg : 0);

  // ---- upload
  cudaStream_t s = c->stream;
  cudaError_t e = cudaSuccess;
  auto up = [&](void *dst, const void *src, size_t bytes) {
    if (e == cudaSuccess && bytes) e = cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, s);
  };
  up(d_descs, b->descs.data(), sizeof(HcjImageDesc) * n);
  up(d_sets, table_sets.data(), sizeof(HcjTableSet) * table_sets.size());
  up(d_prim, prim_pool.data(), 2 * prim_pool.size());
  up(d_full, full_pool.data(), 2 * full_pool.size());
  up(d_qt, qt_pool.data(), 4 * qt_pool.size());
  up(d_lr, list_restart.data(), 4 * list_restart.size());
  up(d_ls, list_spec.data(), 4 * list_spec.size());
  if (e == cudaSuccess && with_files) e = upload_files(b, jpeg, len, 0, n, s);
  if (e == cudaSuccess) e = cudaStreamSynchronize(s);  // host staging vectors go out of scope
  mark("tables on the device");
  if (e != cudaSuccess) {
    hcj_batch_destroy(c, b);
    return HCJ_ERR_CUDA - (int)e;
  }
  *out = b;
  return HCJ_OK;
}

int hcj_batch_create(hcj_ctx *c, const uint8_t *const *jpeg, const size_t *len, int n, int mode, unsigned flags,
                     int *status, hcj_batch **out) {
  return batch_create(c, jpeg, len, n, mode, flags, status, out, true);
}

int hcj_batch_count_kernels(const hcj_batch *b) { return b ? b->kernels : 0; }

int hcj_batch_decode(hcj_ctx *c, hcj_batch *b) {
  if (!c || !b) return HCJ_ERR_INVALID_ARG;
  CU_TRY(cudaSetDevice(c->device));
  cudaStream_t s = c->stream;
  if (b->n == 0) return HCJ_OK;
  CU_TRY((cudaError_t)hcjk::decode_prologue(b->dev, s));
  hcjk::launch_destuff(b->dev, s);
  hcjk::launch_huff_restart(b->dev, s);
  hcjk::launch_huff_spec(b->dev, s);
  hcjk::launch_idct(b->dev, b->mode == HCJ_OUT_YUV ? 0 : b->mode == HCJ_OUT_PLANES ? 1 : 2, s);
  if (post_444(b->mode)) hcjk::launch_rgb(b->dev, b->mode == HCJ_OUT_YUV444, s);
  CU_TRY(cudaGetLastError());
  return HCJ_OK;
}

static const char *kStageNames[] = {"clear_flags", "destuff", "huffman_restart", "huffman_speculative", "idct", "rgb"};
const char *hcj_decode_stage_name(int i) { return i >= 0 && i < 6 ? kStageNames[i] : ""; }

int hcj_batch_decode_stages(hcj_ctx *c, hcj_batch *b, float *ms, int capacity, int *nstages) {
  if (!c || !b || !ms || !nstages || capacity < 6) return HCJ_ERR_INVALID_ARG;
  CU_TRY(cudaSetDevice(c->device));
  cudaStream_t s = c->stream;
  cudaEvent_t ev[7];
  for (auto &e : ev) CU_TRY(cudaEventCreate(&e));
  const int mode = b->mode == HCJ_OUT_YUV ? 0 : b->mode == HCJ_OUT_PLANES ? 1 : 2;
  cudaEventRecord(ev[0], s);
  hcjk::decode_prologue(b->dev, s);
  cudaEventRecord(ev[1], s);
  hcjk::launch_destuff(b->dev, s);
  cudaEventRecord(ev[2], s);
  hcjk::launch_huff_restart(b->dev, s);
  cudaEventRecord(ev[3], s);
  hcjk::launch_huff_spec(b->dev, s);
  cudaEventRecord(ev[4], s);
  hcjk::launch_idct(b->dev, mode, s);
  cudaEventRecord(ev[5], s);
  if (post_444(b->mode)) hcjk::launch_rgb(b->dev, b->mode == HCJ_OUT_YUV444, s);
  cudaEventRecord(ev[6], s);
  cudaError_t e = cudaEventSynchronize(ev[6]);
  if (e == cudaSuccess) e = cudaGetLastError();
  for (int i = 0; i < 6 && e == cudaSuccess; i++) e = cudaEventElapsedTime(&ms[i], ev[i], ev[i + 1]);
  for (auto &x : ev) cudaEventDestroy(x);
  if (e == cudaSuccess && getenv("HCJ_SPEC_STATS") && !b->list_spec.empty()) {
    // fix-point statistics of the speculative decoder: rounds and subsequences decoded again per image
    std::vector<HcjImageState> states(b->n);
    e = cudaMemcpy(states.data(), b->dev.states, sizeof(HcjImageState) * b->n, cudaMemcpyDeviceToHost);
    unsigned long long redo = 0, rounds = 0;
    unsigned max_rounds = 0, with_redo = 0;
    for (uint32_t i : b->list_spec) {
      const unsigned r = states[i].pad_ & 255u, n = states[i].pad_ >> 8;
      redo += n, rounds += r;
      max_rounds = std::max(max_rounds, r);
      with_redo += r != 0;
    }
    fprintf(stderr, "[spec] images %zu  with redo %u  rounds total %llu max %u  subsequences redone %llu\n", b->list_spec.size(), with_redo,
            rounds, max_rounds, redo);
  }
  *nstages = 6;
  return e == cudaSuccess ? HCJ_OK : HCJ_ERR_CUDA - (int)e;
}

static int fetch_states(hcj_ctx *c, hcj_batch *b, std::vector<HcjImageState> *states) {
  states->assign(std::max(b->n, 1), HcjImageState());
  if (b->n)
    CU_TRY(cudaMemcpyAsync(states->data(), b->dev.states, sizeof(HcjImageState) * b->n, cudaMemcpyDeviceToHost, c->stream));
  CU_TRY(cudaStreamSynchronize(c->stream));
  for (int i = 0; i < b->n; i++) {
    HcjImageState &st = (*states)[i];
    if (b->host_status[i] != HCJ_OK) st.status = b->host_status[i];
    else if (st.status == 0 && st.err_key != HCJ_NO_ERR_KEY) st.status = -(int)(st.err_key & 0xff);
  }
  return HCJ_OK;
}

int hcj_batch_fetch(hcj_ctx *c, hcj_batch *b, uint8_t *const *out, const size_t *out_capacity, int *status) {
  if (!c || !b || (b->n > 0 && (!out || !out_capacity))) return HCJ_ERR_INVALID_ARG;
  CU_TRY(cudaSetDevice(c->device));
  std::vector<int> st(b->host_status);
  for (int i = 0; i < b->n; i++) {
    if (st[i] != HCJ_OK) continue;
    if (!out[i] || out_capacity[i] < b->out_bytes[i]) {
      st[i] = HCJ_ERR_BUFFER_TOO_SMALL;
      continue;
    }
    CU_TRY(cudaMemcpyAsync(out[i], b->dev.out + b->descs[i].out_off, b->out_bytes[i], cudaMemcpyDeviceToHost, c->stream));
  }
  std::vector<HcjImageState> states;
  int r = fetch_states(c, b, &states);
  if (r != HCJ_OK) return r;
  for (int i = 0; i < b->n; i++)
    if (st[i] == HCJ_OK && states[i].status != 0) st[i] = states[i].status;
  if (status)
    for (int i = 0; i < b->n; i++) status[i] = st[i];
  return HCJ_OK;
}

int hcj_batch_device_output(hcj_batch *b, int i, void **dptr, size_t *bytes) {
  if (!b || i < 0 || i >= b->n || !dptr || !bytes) return HCJ_ERR_INVALID_ARG;
  if (b->host_status[i] != HCJ_OK) return b->host_status[i];
  *dptr = b->dev.out + b->descs[i].out_off;
  *bytes = b->out_bytes[i];
  return HCJ_OK;
}

// One-call form.  The batch is decoded in chunks of images: while the kernels of chunk k+1 run on the
// context's stream, the frames of chunk k travel to the host on a second stream (D2H dominates the
// end-to-end time: 3 MB out per 0.4 MB in for 1080p 4:2:0).
int hcj_decode_batch(hcj_ctx *c, const uint8_t *const *jpeg, const size_t *len, int n, int mode, unsigned flags,
                     uint8_t *const *out, const size_t *out_capacity, int *status) {
  // Three streams: the files of chunk k + 1 go up while the kernels of chunk k run and the frames of chunk
  // k - 1 come down; PCIe is full duplex and the kernels are a small fraction of either transfer.
  const bool trace = getenv("HCJ_TRACE") != nullptr;  // host-side milestones of one call, to stderr
  const auto t0 = std::chrono::steady_clock::now();
  auto mark = [&](const char *what) {
    if (trace)
      fprintf(stderr, "[hcj_decode_batch] %-28s %8.3f ms\n", what,
              std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count());
  };
  hcj_batch *b = nullptr;
  int st = batch_create(c, jpeg, len, n, mode, flags, status, &b, false);
  mark("headers parsed, tables up");
  if (st != HCJ_OK) return st;
  if (n > 0 && (!out || !out_capacity)) {
    hcj_batch_destroy(c, b);
    return HCJ_ERR_INVALID_ARG;
  }
  cudaStream_t s = c->stream, cs = c->copy_stream, us = c->up_stream;
  cudaError_t e = cudaSuccess;
  // Chunk boundaries: the first chunks are small (a quarter, then half of the regular size) so that the first frames
  // start down the link as early as possible; the regular chunk keeps the per-launch overhead small.
  const int chunk = std::max(16, std::min(128, (n + 7) / 8));
  std::vector<int> bound(1, 0);
  for (int sz = std::max(8, chunk / 4); bound.back() < n; sz = std::min(chunk, sz * 2)) bound.push_back(std::min(n, bound.back() + sz));
  const int nchunks = (int)bound.size() - 1;
  while ((int)c->chunk_events.size() < nchunks + 1) {
    cudaEvent_t ev;
    if (cudaEventCreateWithFlags(&ev, cudaEventDisableTiming) != cudaSuccess) break;
    c->chunk_events.push_back(ev);
  }
  while ((int)c->up_events.size() < nchunks + 1) {
    cudaEvent_t ev;
    if (cudaEventCreateWithFlags(&ev, cudaEventDisableTiming) != cudaSuccess) break;
    c->up_events.push_back(ev);
  }
  std::vector<int> host_st(b->host_status);
  if (n > 0 && (int)c->chunk_events.size() >= nchunks + 1 && (int)c->up_events.size() >= nchunks + 1) {
    for (int k = 0; k < nchunks && e == cudaSuccess; k++) {
      e = upload_files(b, jpeg, len, bound[k], bound[k + 1], us);
      if (e == cudaSuccess) e = cudaEventRecord(c->up_events[k], us);
    }
    if (e == cudaSuccess) e = (cudaError_t)hcjk::decode_prologue(b->dev, s);
    const int kmode = mode == HCJ_OUT_YUV ? 0 : mode == HCJ_OUT_PLANES ? 1 : 2;
    size_t lr = 0, ls = 0;
    for (int k = 0; k < nchunks && e == cudaSuccess; k++) {
      hcjk::DecodeBatchDev dv = b->dev;
      dv.img_lo = (uint32_t)bound[k];
      dv.img_hi = (uint32_t)bound[k + 1];
      dv.tile_lo = b->tile_base[dv.img_lo];
      dv.tile_hi = b->tile_base[dv.img_hi];
      dv.lr_lo = (uint32_t)lr;
      while (lr < b->list_restart.size() && b->list_restart[lr] < dv.img_hi) lr++;
      dv.lr_hi = (uint32_t)lr;
      dv.ls_lo = (uint32_t)ls;
      while (ls < b->list_spec.size() && b->list_spec[ls] < dv.img_hi) ls++;
      dv.ls_hi = (uint32_t)ls;
      e = cudaStreamWaitEvent(s, c->up_events[k], 0);
      if (e != cudaSuccess) break;
      hcjk::launch_destuff(dv, s);
      hcjk::launch_huff_restart(dv, s);
      hcjk::launch_huff_spec(dv, s);
      hcjk::launch_idct(dv, kmode, s);
      if (post_444(mode)) hcjk::launch_rgb(dv, mode == HCJ_OUT_YUV444, s);
      e = cudaGetLastError();
      if (e == cudaSuccess) e = cudaEventRecord(c->chunk_events[k], s);
      if (e == cudaSuccess) e = cudaStreamWaitEvent(cs, c->chunk_events[k], 0);
      for (uint32_t i = dv.img_lo; i < dv.img_hi; i++)
        if (host_st[i] == HCJ_OK && (!out[i] || out_capacity[i] < b->out_bytes[i])) host_st[i] = HCJ_ERR_BUFFER_TOO_SMALL;
      for (uint32_t i = dv.img_lo; i < dv.img_hi && e == cudaSuccess;) {
        if (host_st[i] != HCJ_OK) {
          i++;
          continue;
        }
        // frames that are laid out in the caller's memory like in the device buffer leave in one copy
        uint32_t j = i;
        size_t bytes = b->out_bytes[i];
        while (j + 1 < dv.img_hi && host_st[j + 1] == HCJ_OK &&
               out[j + 1] == out[i] + (b->descs[j + 1].out_off - b->descs[i].out_off) &&
               out_capacity[j] >= (size_t)(b->descs[j + 1].out_off - b->descs[j].out_off)) {
          j++;
          bytes = (size_t)(b->descs[j].out_off - b->descs[i].out_off) + b->out_bytes[j];
        }
        e = cudaMemcpyAsync(out[i], b->dev.out + b->descs[i].out_off, bytes, cudaMemcpyDeviceToHost, cs);
        i = j + 1;
      }
    }
    mark("everything enqueued");
    if (trace && e == cudaSuccess) {
      e = cudaStreamSynchronize(us);
      mark("files on the device");
      if (e == cudaSuccess) e = cudaStreamSynchronize(s);
      mark("kernels done");
    }
    if (e == cudaSuccess) e = cudaStreamSynchronize(cs);
    mark("frames on the host");
    std::vector<HcjImageState> states;
    if (e == cudaSuccess) {
      int r = fetch_states(c, b, &states);
      if (r != HCJ_OK) {
        cudaStreamSynchronize(us);
        cudaStreamSynchronize(cs);
        hcj_batch_destroy(c, b);
        return r;
      }
      for (int i = 0; i < n; i++)
        if (host_st[i] == HCJ_OK && states[i].status != 0) host_st[i] = states[i].status;
    }
  } else if (n > 0) {
    e = cudaErrorMemoryAllocation;
  }
  if (status)
    for (int i = 0; i < n; i++) status[i] = host_st[i];
  if (e != cudaSuccess) {  // copies may still be reading the caller's files / writing the caller's frames
    cudaStreamSynchronize(us);
    cudaStreamSynchronize(cs);
  }
  hcj_batch_destroy(c, b);
  mark("batch released");
  return e == cudaSuccess ? HCJ_OK : HCJ_ERR_CUDA - (int)e;
}

int hcj_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) {
    (void)cudaGetLastError();
    return 0;
  }
  return n;
}

void hcj_shard_range(int n, int part, int nparts, int *lo, int *hi) {
  if (nparts < 1) nparts = 1;
  part = std::min(std::max(part, 0), nparts - 1);
  if (lo) *lo = (int)((int64_t)n * part / nparts);
  if (hi) *hi = (int)((int64_t)n * (part + 1) / nparts);
}

// One process, several GPUs (SURVEY 8e: one hcj_ctx + host thread + CUDA stream set per device): images are
// independent, so context k decodes the contiguous index range hcj_shard_range(n, k, nctx) with its own pipelined
// hcj_decode_batch on its own host thread; nothing is exchanged between devices.
int hcj_decode_batch_multi(hcj_ctx *const *ctx, int nctx, const uint8_t *const *jpeg, const size_t *len, int n, int mode,
                           unsigned flags, uint8_t *const *out, const size_t *out_capacity, int *status) {
  if (!ctx || nctx < 1 || n < 0 || (n > 0 && (!jpeg || !len || !out || !out_capacity))) return HCJ_ERR_INVALID_ARG;
  for (int k = 0; k < nctx; k++)
    if (!ctx[k]) return HCJ_ERR_INVALID_ARG;
  for (int k = 0; k < nctx; k++)
    for (int j = 0; j < k; j++)
      if (ctx[k] == ctx[j]) return HCJ_ERR_INVALID_ARG;  // a context is not thread-safe
  std::vector<int> rc((size_t)nctx, HCJ_OK);
  auto work = [&](int k) {
    int lo, hi;
    hcj_shard_range(n, k, nctx, &lo, &hi);
    rc[k] = hcj_decode_batch(ctx[k], jpeg + lo, len + lo, hi - lo, mode, flags, out + lo, out_capacity + lo, status ? status + lo : nullptr);
  };
  std::vector<std::thread> pool;
  try {
    for (int k = 1; k < nctx; k++) pool.emplace_back(work, k);
  } catch (...) {
    for (auto &t : pool) t.join();
    return HCJ_ERR_OUT_OF_MEMORY;
  }
  work(0);
  for (auto &t : pool) t.join();
  for (int k = 0; k < nctx; k++)
    if (rc[k] != HCJ_OK) return rc[k];
  return HCJ_OK;
}

int hcj_batch_fetch_coefficients(hcj_ctx *c, hcj_batch *b, int i, int16_t *coefs, size_t capacity_blocks) {
  if (!c || !b || i < 0 || i >= b->n || !coefs) return HCJ_ERR_INVALID_ARG;
  if (b->host_status[i] != HCJ_OK) return b->host_status[i];
  const HcjImageDesc &d = b->descs[i];
  if (capacity_blocks < d.nblocks) return HCJ_ERR_BUFFER_TOO_SMALL;
  CU_TRY(cudaSetDevice(c->device));
  CU_TRY(cudaMemcpyAsync(coefs, b->dev.coefs + d.coef_off * 64, (size_t)d.nblocks * 128, cudaMemcpyDeviceToHost, c->stream));
  std::vector<HcjImageState> states;
  int r = fetch_states(c, b, &states);
  return r != HCJ_OK ? r : states[i].status;
}

int hcj_batch_fetch_entropy(hcj_ctx *c, hcj_batch *b, int i, uint8_t *out, size_t capacity, size_t *len) {
  if (!c || !b || i < 0 || i >= b->n || !out || !len) return HCJ_ERR_INVALID_ARG;
  if (b->host_status[i] != HCJ_OK) return b->host_status[i];
  CU_TRY(cudaSetDevice(c->device));
  std::vector<HcjImageState> states;
  int r = fetch_states(c, b, &states);
  if (r != HCJ_OK) return r;
  *len = states[i].ent_len;
  if (states[i].status == HCJ_ERR_NO_TERMINATOR) return states[i].status;
  if (capacity < states[i].ent_len) return HCJ_ERR_BUFFER_TOO_SMALL;
  CU_TRY(cudaMemcpy(out, b->dev.entropy + b->descs[i].ent_off, states[i].ent_len, cudaMemcpyDeviceToHost));
  return HCJ_OK;
}

int hcj_idct_blocks(hcj_ctx *c, const int16_t *coefs, size_t nblocks, const uint16_t quant_table[64], uint8_t *out) {
  if (!c || !coefs || !quant_table || !out) return HCJ_ERR_INVALID_ARG;
  CU_TRY(cudaSetDevice(c->device));
  void *d_c = nullptr, *d_q = nullptr, *d_o = nullptr;
  int st = c->alloc(&d_c, nblocks * 128 + 16);
  if (st == HCJ_OK) st = c->alloc(&d_q, 256);
  if (st == HCJ_OK) st = c->alloc(&d_o, nblocks * 64 + 16);
  cudaError_t e = cudaSuccess;
  if (st == HCJ_OK) {
    bool wide = false;
    for (int i = 0; i < 64; i++) wide |= quant_table[i] > 255;
    e = cudaMemcpyAsync(d_c, coefs, nblocks * 128, cudaMemcpyHostToDevice, c->stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(d_q, quant_table, 128, cudaMemcpyHostToDevice, c->stream);
    if (e == cudaSuccess) {
      hcjk::launch_idct_blocks((const int16_t *)d_c, nblocks, (const uint16_t *)d_q, wide, (uint8_t *)d_o, c->stream);
      e = cudaGetLastError();
    }
    if (e == cudaSuccess) e = cudaMemcpyAsync(out, d_o, nblocks * 64, cudaMemcpyDeviceToHost, c->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
  }
  c->release(d_c);
  c->release(d_q);
  c->release(d_o);
  if (st != HCJ_OK) return st;
  return e == cudaSuccess ? HCJ_OK : HCJ_ERR_CUDA - (int)e;
}

int hcj_batch_fetch_block_log(hcj_ctx *c, hcj_batch *b, int i, size_t first_block, size_t count, hcj_block_log *out) {
  static_assert(sizeof(hcj_block_log) == sizeof(hcjk::BlockLog), "hcj_block_log layout");
  if (!c || !b || i < 0 || i >= b->n || !out) return HCJ_ERR_INVALID_ARG;
  if (b->host_status[i] != HCJ_OK) return b->host_status[i];
  const HcjImageDesc &d = b->descs[i];
  if (first_block > d.nblocks || count > d.nblocks - first_block) return HCJ_ERR_INVALID_ARG;
  CU_TRY(cudaSetDevice(c->device));
  std::vector<HcjImageState> states;
  int r = fetch_states(c, b, &states);
  if (r != HCJ_OK) return r;
  if (states[i].status != 0) return states[i].status;
  if (count == 0) return HCJ_OK;
  void *d_out = nullptr;
  int st = c->alloc(&d_out, count * sizeof(hcj_block_log));
  if (st != HCJ_OK) return st;
  hcjk::launch_block_log(b->dev, (uint32_t)i, (uint32_t)first_block, (uint32_t)count, (hcjk::BlockLog *)d_out, c->stream);
  cudaError_t e = cudaGetLastError();
  if (e == cudaSuccess) e = cudaMemcpyAsync(out, d_out, count * sizeof(hcj_block_log), cudaMemcpyDeviceToHost, c->stream);
  if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
  c->release(d_out);
  return e == cudaSuccess ? HCJ_OK : HCJ_ERR_CUDA - (int)e;
}

int hcj_decode_a_frame(hcj_ctx *c, const uint8_t *jpeg, size_t len, int mode, unsigned flags, uint8_t *out, size_t out_capacity) {
  int status = HCJ_OK;
  const uint8_t *in[1] = {jpeg};
  uint8_t *o[1] = {out};
  int st = hcj_decode_batch(c, in, &len, 1, mode, flags, o, &out_capacity, &status);
  return st != HCJ_OK ? st : status;
}

int hcj_mjpeg_split(const uint8_t *stream, size_t len, size_t *offsets, size_t *lengths, int capacity, int *nframes) {
  if (!stream || !nframes || capacity < 0) return HCJ_ERR_INVALID_ARG;
  return hcj::mjpeg_split(stream, len, offsets, lengths, capacity, nframes);
}

int hcj_decode_stream(hcj_ctx *c, const uint8_t *stream, size_t len, int mode, unsigned flags, uint8_t *out, size_t out_capacity,
                      size_t *out_offsets, int *status, int capacity, int *nframes) {
  if (!c || !stream || !nframes || capacity < 0) return HCJ_ERR_INVALID_ARG;
  int n = 0;
  std::vector<size_t> off((size_t)capacity + 1), ln((size_t)capacity + 1);
  int st = hcj::mjpeg_split(stream, len, off.data(), ln.data(), capacity, &n);
  *nframes = n;
  if (st != HCJ_OK) return st;
  if (n == 0) return HCJ_OK;
  if (!out || !out_offsets || !status) return HCJ_ERR_INVALID_ARG;
  // frames are laid out back to back, each at a 256-byte boundary like in the device buffer: consecutive good
  // frames then leave in one device-to-host copy
  std::vector<const uint8_t *> jp((size_t)n);
  std::vector<uint8_t *> op((size_t)n);
  std::vector<size_t> cap((size_t)n);
  size_t acc = 0;
  for (int i = 0; i < n; i++) {
    jp[i] = stream + off[i];
    hcj_frame_info f;
    size_t bytes = 0;
    if (hcj_frame_info_get_ex(jp[i], ln[i], flags, &f) == HCJ_OK)
      bytes = mode == HCJ_OUT_YUV ? f.yuv_bytes : mode == HCJ_OUT_PLANES ? f.planes_bytes : f.rgb_bytes;
    out_offsets[i] = acc;
    cap[i] = bytes;
    acc += (bytes + 255) & ~(size_t)255;
  }
  out_offsets[n] = acc;
  if (acc > out_capacity) return HCJ_ERR_BUFFER_TOO_SMALL;
  // the slot of every frame but the last reaches to the next frame: hcj_decode_batch then merges consecutive frames
  // into one device-to-host copy (it needs capacity >= the distance to the next frame in the device buffer)
  for (int i = 0; i + 1 < n; i++)
    if (cap[i]) cap[i] = out_offsets[i + 1] - out_offsets[i];
  for (int i = 0; i < n; i++) op[i] = out + out_offsets[i];
  return hcj_decode_batch(c, jp.data(), ln.data(), n, mode, flags, op.data(), cap.data(), status);
}

int hcj_yuv_convert(hcj_ctx *c, const uint8_t *src, int width, int height, int chroma, int x_off, int y_off, uint8_t *dst, int dst_width,
                    int dst_height, int dst_chroma, size_t dst_capacity) {
  auto ok = [](int ch) { return ch == 420 || ch == 422 || ch == 444; };
  if (!c || !src || !dst || width < 1 || height < 1 || dst_width < 1 || dst_height < 1 || !ok(chroma) || !ok(dst_chroma))
    return HCJ_ERR_INVALID_ARG;
  const size_t nin = hcjk::yuv_frame_bytes(width, height, chroma), nout = hcjk::yuv_frame_bytes(dst_width, dst_height, dst_chroma);
  if (dst_capacity < nout) return HCJ_ERR_BUFFER_TOO_SMALL;
  CU_TRY(cudaSetDevice(c->device));
  void *d_in = nullptr, *d_out = nullptr;
  int st = c->alloc(&d_in, nin + 16);
  if (st == HCJ_OK) st = c->alloc(&d_out, nout + 16);
  cudaError_t e = cudaSuccess;
  if (st == HCJ_OK) {
    e = cudaMemcpyAsync(d_in, src, nin, cudaMemcpyHostToDevice, c->stream);
    if (e == cudaSuccess) {
      hcjk::launch_yuv_convert((const uint8_t *)d_in, width, height, chroma, x_off, y_off, (uint8_t *)d_out, dst_width, dst_height, dst_chroma,
                               c->stream);
      e = cudaGetLastError();
    }
    if (e == cudaSuccess) e = cudaMemcpyAsync(dst, d_out, nout, cudaMemcpyDeviceToHost, c->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
  }
  c->release(d_in);
  c->release(d_out);
  if (st != HCJ_OK) return st;
  return e == cudaSuccess ? HCJ_OK : HCJ_ERR_CUDA - (int)e;
}

int hcj_batch_compare(hcj_ctx *c, hcj_batch *b, const uint8_t *const *ref, const size_t *ref_len, hcj_plane_metrics *out) {
  if (!c || !b || !ref || !ref_len || !out) return HCJ_ERR_INVALID_ARG;
  CU_TRY(cudaSetDevice(c->device));
  const int n = b->n;
  if (n == 0) return HCJ_OK;
  // planes of every image in its output and in the reference buffer
  std::vector<hcjk::ComparePlane> planes((size_t)n * 4);
  std::vector<uint64_t> ref_off((size_t)n, 0);
  uint64_t ref_total = 0;
  for (int i = 0; i < n; i++) {
    memset(&out[i], 0, sizeof(out[i]));
    const HcjImageDesc &d = b->descs[i];
    out[i].status = b->host_status[i];
    if (out[i].status == HCJ_OK && (!ref[i] || ref_len[i] != b->out_bytes[i])) out[i].status = HCJ_ERR_INVALID_ARG;
    if (out[i].status != HCJ_OK) continue;
    ref_off[i] = ref_total;
    ref_total += (b->out_bytes[i] + 15) & ~(uint64_t)15;
    uint64_t acc = 0;
    const int np = b->mode == HCJ_OUT_RGB24 ? 1 : b->mode == HCJ_OUT_PLANES ? d.ncomp : 3;
    for (int k = 0; k < np; k++) {
      uint64_t bytes;
      if (b->mode == HCJ_OUT_RGB24) bytes = (uint64_t)d.width * d.height * 3;
      else if (b->mode == HCJ_OUT_YUV444) bytes = (uint64_t)d.width * d.height;
      else if (b->mode == HCJ_OUT_PLANES) bytes = (uint64_t)d.comp[k].decoded_w * d.comp[k].decoded_h;
      else bytes = (uint64_t)d.comp[k].actual_w * d.comp[k].actual_h;
      planes[(size_t)i * 4 + k] = hcjk::ComparePlane{d.out_off + acc, ref_off[i] + acc, bytes};
      out[i].samples[k] = (int64_t)bytes;
      acc += bytes;
    }
  }
  void *d_ref = nullptr, *d_pl = nullptr, *d_acc = nullptr;
  const size_t acc_bytes = (size_t)n * 16 * sizeof(unsigned long long);
  std::vector<unsigned long long> res((size_t)n * 16, 0);
  int st = c->alloc(&d_ref, ref_total + 16);
  if (st == HCJ_OK) st = c->alloc(&d_pl, planes.size() * sizeof(hcjk::ComparePlane));
  if (st == HCJ_OK) st = c->alloc(&d_acc, acc_bytes);
  cudaError_t e = cudaSuccess;
  if (st == HCJ_OK) {
    for (int i = 0; i < n && e == cudaSuccess; i++)
      if (out[i].status == HCJ_OK)
        e = cudaMemcpyAsync((uint8_t *)d_ref + ref_off[i], ref[i], b->out_bytes[i], cudaMemcpyHostToDevice, c->stream);
    if (e == cudaSuccess)
      e = cudaMemcpyAsync(d_pl, planes.data(), planes.size() * sizeof(hcjk::ComparePlane), cudaMemcpyHostToDevice, c->stream);
    if (e == cudaSuccess) e = cudaMemsetAsync(d_acc, 0, acc_bytes, c->stream);
    if (e == cudaSuccess) {
      hcjk::launch_compare_planes(b->dev.out, (const uint8_t *)d_ref, (const hcjk::ComparePlane *)d_pl, (unsigned long long *)d_acc, n,
                                  c->stream);
      e = cudaGetLastError();
    }
    if (e == cudaSuccess) e = cudaMemcpyAsync(res.data(), d_acc, acc_bytes, cudaMemcpyDeviceToHost, c->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
  }
  c->release(d_ref);
  c->release(d_pl);
  c->release(d_acc);
  if (st != HCJ_OK) return st;
  if (e != cudaSuccess) return HCJ_ERR_CUDA - (int)e;
  for (int i = 0; i < n; i++)
    for (int k = 0; k < 4; k++) {
      out[i].square_error[k] = (int64_t)res[((size_t)i * 4 + k) * 4 + 0];
      out[i].total_difference[k] = (int64_t)res[((size_t)i * 4 + k) * 4 + 1];
      out[i].max_difference[k] = (int)res[((size_t)i * 4 + k) * 4 + 2];
    }
  return HCJ_OK;
}

int hcj_compare_planes(hcj_ctx *c, const uint8_t *a, const uint8_t *b, size_t n, int64_t *square_error, int *max_difference) {
  int64_t total = 0;
  return hcj_compare_planes_ex(c, a, b, n, square_error, max_difference, &total);
}

int hcj_compare_planes_ex(hcj_ctx *c, const uint8_t *a, const uint8_t *b, size_t n, int64_t *square_error, int *max_difference,
                          int64_t *total_difference) {
  if (!c || !a || !b || !square_error || !max_difference || !total_difference) return HCJ_ERR_INVALID_ARG;
  CU_TRY(cudaSetDevice(c->device));
  void *d_a = nullptr, *d_b = nullptr, *d_r = nullptr;
  int st = c->alloc(&d_a, n + 16);
  if (st == HCJ_OK) st = c->alloc(&d_b, n + 16);
  if (st == HCJ_OK) st = c->alloc(&d_r, 256);
  cudaError_t e = cudaSuccess;
  unsigned long long res[3] = {0, 0, 0};
  if (st == HCJ_OK) {
    e = cudaMemcpyAsync(d_a, a, n, cudaMemcpyHostToDevice, c->stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(d_b, b, n, cudaMemcpyHostToDevice, c->stream);
    if (e == cudaSuccess) e = cudaMemsetAsync(d_r, 0, 24, c->stream);
    if (e == cudaSuccess) {
      hcjk::launch_compare((const uint8_t *)d_a, (const uint8_t *)d_b, n, (unsigned long long *)d_r, c->stream);
      e = cudaGetLastError();
    }
    if (e == cudaSuccess) e = cudaMemcpyAsync(res, d_r, 24, cudaMemcpyDeviceToHost, c->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
  }
  c->release(d_a);
  c->release(d_b);
  c->release(d_r);
  if (st != HCJ_OK) return st;
  if (e != cudaSuccess) return HCJ_ERR_CUDA - (int)e;
  *square_error = (int64_t)res[0];
  *max_difference = (int)(res[1] & 0xffffffffu);
  *total_difference = (int64_t)res[2];
  return HCJ_OK;
}

}  // extern "C"
