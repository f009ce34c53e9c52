// graphblast_b200 backend — Descriptor: per-call flags, CLI knobs and the
// grow-only device scratch every operation borrows from.
//
// Replaces reference graphblas/backend/cuda/descriptor.hpp:14-287.  Same field
// table (desc_[GrB_NDESCFIELD]), same toggle() rule (:141-154), same knob names
// and accessors; loadArgs() (:207-287), setKnob() and getKnob() are three functors
// over one enumeration of the knobs.
// Data members the reference drivers reach through `#define private public`
// keep their names: max_niter_, timing_, lastmxv_, debug_
// (reference algorithm/bfs.hpp:46,54,56).
//
// B200-first differences:
//  * no moderngpu context; scratch is a set of typed arenas sized in size_t
//    (the reference sizes scratch in `int` and overflows at RMAT-24 unless
//    --memusage <= 0.5, reference spmspv.hpp:60-66);
//  * push-direction accumulator + touched-bitmap arenas keep an invariant
//    ("all identity" / "all zero") between calls so no O(n) clear per level.
#ifndef GRAPHBLAS_BACKEND_CUDA_DESCRIPTOR_HPP_
#define GRAPHBLAS_BACKEND_CUDA_DESCRIPTOR_HPP_

#include <vector>
#include <string>

#include "graphblas/backend/cuda/util.hpp"

namespace graphblas {
namespace backend {

// Scratch arenas (each grows independently, never shrinks).
enum ScratchSlot {
  GB_SCRATCH_ACC = 0,     // push: dense accumulator, one value per output vertex
  GB_SCRATCH_BITS,        // push: touched bitmap, one bit per output vertex
  GB_SCRATCH_OFFS,        // push: scanned frontier degrees
  GB_SCRATCH_BLOCKSUM,    // compaction: per-CTA counts / offsets
  GB_SCRATCH_COUNTERS,    // small device counters (64 x 8 bytes)
  GB_SCRATCH_CARRY_ROW,   // pull: per-CTA carry-out row ids
  GB_SCRATCH_CARRY_VAL,   // pull: per-CTA carry-out partials
  GB_SCRATCH_VEC_A,       // generic n-sized temporaries
  GB_SCRATCH_VEC_B,
  GB_SCRATCH_CUB,         // cub temp storage
  GB_SCRATCH_BFS,         // fused BFS: visited x2, frontier, next bitmaps + cells
  GB_SCRATCH_NSLOTS
};

// One visitor enumerates the command-line knobs (name -> member); loading a
// variables_map, setting a knob by name and reading one back are three functors
// over it.  Names and types are the drivers' (reference util.hpp:39-132).
class Descriptor {
 public:
  Descriptor() {
    static const Desc_value kDefaults[GrB_NDESCFIELD] = {
        GrB_DEFAULT, GrB_DEFAULT, GrB_DEFAULT, GrB_DEFAULT,     // mask, outp, inp0, inp1
        GrB_FIXEDROW, GrB_32, GrB_32, GrB_128, GrB_PUSHPULL, GrB_16, GrB_CUDA};
    for (int f = 0; f < GrB_NDESCFIELD; ++f) desc_[f] = kDefaults[f];
    for (int i = 0; i < GB_SCRATCH_NSLOTS; ++i) { slot_ptr_[i] = NULL; slot_size_[i] = 0; }
  }
  ~Descriptor() {
    cudaFree(d_buffer_);                      // cudaFree(NULL) is a no-op
    cudaFree(d_temp_);
    for (int i = 0; i < GB_SCRATCH_NSLOTS; ++i) cudaFree(slot_ptr_[i]);
  }

  // ---- field table -----------------------------------------------------------------
  Info set(Desc_field field, Desc_value value) { desc_[field] = value; return GrB_SUCCESS; }
  Info get(Desc_field field, Desc_value* value) const {
    *value = desc_[field];
    return GrB_SUCCESS;
  }
  // MASK, OUTP, INP0, INP1 flip between GrB_DEFAULT and their one other value
  // (GrB_SCMP, GrB_REPLACE, GrB_TRAN, GrB_TRAN); other fields are left alone
  // (reference :141-154).
  Info toggle(Desc_field field) {
    static const Desc_value kOther[4] = {GrB_SCMP, GrB_REPLACE, GrB_TRAN, GrB_TRAN};
    const int f = static_cast<int>(field);
    if (f < 4) desc_[f] = (desc_[f] == GrB_DEFAULT) ? kOther[f] : GrB_DEFAULT;
    return GrB_SUCCESS;
  }

  // ---- knobs -------------------------------------------------------------------------
  template <typename Visitor>
  void eachKnob(Visitor&& knob) {
    knob("ta", ta_);                   knob("tb", tb_);
    knob("mode", mode_);               knob("split", split_);
    knob("niter", niter_);             knob("max_niter", max_niter_);
    knob("directed", directed_);       knob("timing", timing_);
    knob("transpose", transpose_);     knob("mtxinfo", mtxinfo_);
    knob("verbose", verbose_);         knob("mxvmode", mxvmode_);
    knob("switchpoint", switchpoint_); knob("dirinfo", dirinfo_);
    knob("struconly", struconly_);     knob("opreuse", opreuse_);
    knob("memusage", memusage_);       knob("endbit", endbit_);
    knob("sort", sort_);               knob("atomic", atomic_);
    knob("earlyexit", earlyexit_);     knob("fusedmask", fusedmask_);
    knob("nthread", nthread_);         knob("ndevice", ndevice_);
    knob("debug", debug_);             knob("memory", memory_);
  }
  // Fields that follow a knob: GrB_MXVMODE from mxvmode, GrB_NT from nthread.
  Info settleMode() {
    static const Desc_value kModes[3] = {GrB_PUSHPULL, GrB_PUSHONLY, GrB_PULLONLY};
    if (mxvmode_ < 0 || mxvmode_ > 2) {
      std::cout << "Error: incorrect mxvmode selection!\n";
      return GrB_INVALID_VALUE;
    }
    desc_[GrB_MXVMODE] = kModes[mxvmode_];
    return GrB_SUCCESS;
  }
  Info settleThreads() {
    static const struct { int threads; Desc_value value; } kThreads[] = {
        {32, GrB_32}, {64, GrB_64}, {128, GrB_128}, {256, GrB_256}, {512, GrB_512},
        {1024, GrB_1024}};
    for (const auto& t : kThreads)
      if (t.threads == nthread_) { desc_[GrB_NT] = t.value; return GrB_SUCCESS; }
    std::cout << "Error: incorrect nthread selection!\n";
    return GrB_INVALID_VALUE;
  }
  // All knobs from the drivers' command line (reference :207-287); a wrong mode or
  // thread count is reported and otherwise ignored, as there.
  Info loadArgs(const po::variables_map& vm) {
    eachKnob(FromArgs{vm});
    settleMode();
    settleThreads();
    return GrB_SUCCESS;
  }
  // One knob by name (C ABI); numbers arrive as double.
  Info setKnob(const std::string& name, double value) {
    if (name == "mxvmode" && (value < 0 || value > 2)) return GrB_INVALID_VALUE;
    ByName pick{name, value, false, false};
    eachKnob(pick);
    if (!pick.found) return GrB_INVALID_VALUE;
    if (name == "mxvmode") return settleMode();
    if (name == "nthread") settleThreads();
    return GrB_SUCCESS;
  }
  Info getKnob(const std::string& name, double* value) {
    if (name == "lastmxv") { *value = static_cast<int>(lastmxv_); return GrB_SUCCESS; }
    ByName pick{name, 0.0, true, false};
    eachKnob(pick);
    if (!pick.found) return GrB_INVALID_VALUE;
    *value = pick.value;
    return GrB_SUCCESS;
  }

  bool  debug()       { return debug_; }
  bool  memory()      { return memory_; }
  bool  split()       { return split_ && enable_split_; }
  bool  struconly()   { return struconly_; }
  bool  opreuse()     { return opreuse_; }
  bool  earlyexit()   { return earlyexit_; }
  bool  fusedmask()   { return fusedmask_; }
  bool  dirinfo()     { return dirinfo_; }
  bool  endbit()      { return endbit_; }
  bool  sort()        { return sort_; }
  bool  atomic()      { return atomic_; }
  float switchpoint() { return switchpoint_; }
  float memusage()    { return memusage_; }

  // ---- legacy two-buffer scratch (reference :156-192), for callers that name
  // "buffer" / "temp" -------------------------------------------------------------------
  Info resize(size_t target, std::string field) {
    const bool temp = (field == "temp");
    void*&  block = temp ? d_temp_ : d_buffer_;
    size_t& size  = temp ? d_temp_size_ : d_buffer_size_;
    if (target <= size) return GrB_SUCCESS;
    void* grown = NULL;
    CUDA_CALL(cudaMalloc(&grown, target));
    if (block != NULL) {                      // contents survive a resize
      CUDA_CALL(cudaMemcpyAsync(grown, block, size, cudaMemcpyDeviceToDevice, gbStream()));
      CUDA_CALL(cudaStreamSynchronize(gbStream()));
      CUDA_CALL(cudaFree(block));
    }
    block = grown;
    size  = target;
    return GrB_SUCCESS;
  }
  Info clear(std::string field) {
    const bool temp = (field == "temp");
    if (!temp && field != "buffer") return GrB_SUCCESS;
    void* block = temp ? d_temp_ : d_buffer_;
    if (block != NULL)
      CUDA_CALL(cudaMemsetAsync(block, 0, temp ? d_temp_size_ : d_buffer_size_, gbStream()));
    return GrB_SUCCESS;
  }

  // ---- arenas used by this backend's operations --------------------------------------
  void* scratch(ScratchSlot slot, size_t bytes) {
    if (bytes > slot_size_[slot]) {
      if (slot_ptr_[slot] != NULL) {
        // In-flight kernels may still read the old block.
        CUDA_CALL(cudaStreamSynchronize(gbStream()));
        CUDA_CALL(cudaFree(slot_ptr_[slot]));
      }
      size_t want = bytes + bytes/4 + 256;
      CUDA_CALL(cudaMalloc(&slot_ptr_[slot], want));
      slot_size_[slot] = want;
      if (slot == GB_SCRATCH_ACC)  acc_valid_  = false;
      if (slot == GB_SCRATCH_BITS) bits_valid_ = false;
    }
    return slot_ptr_[slot];
  }
  size_t scratchSize(ScratchSlot slot) const { return slot_size_[slot]; }

  // Device counters: 64 x 8-byte cells, zero when first handed out.  Cell 2 is
  // the "finished CTAs" counter of the compaction's count pass, which leaves it
  // at zero again.
  unsigned long long* counters() {
    if (slot_ptr_[GB_SCRATCH_COUNTERS] == NULL) {
      void* p = scratch(GB_SCRATCH_COUNTERS, 64*sizeof(unsigned long long));
      CUDA_CALL(cudaMemsetAsync(p, 0, slot_size_[GB_SCRATCH_COUNTERS], gbStream()));
    }
    return reinterpret_cast<unsigned long long*>(
        slot_ptr_[GB_SCRATCH_COUNTERS]);
  }

  // ---- data (private in the reference; its drivers `#define private public` and
  // reach max_niter_, timing_, lastmxv_, debug_) ----------------------------------------
  Desc_value desc_[GrB_NDESCFIELD];

  void*  d_buffer_ = NULL;   size_t d_buffer_size_ = 0;     // legacy scratch
  void*  d_temp_ = NULL;     size_t d_temp_size_ = 0;       // legacy cub scratch
  void*  slot_ptr_[GB_SCRATCH_NSLOTS];
  size_t slot_size_[GB_SCRATCH_NSLOTS];

  // knobs, in the order of eachKnob
  int ta_ = 0, tb_ = 0;                       // algorithm specific
  std::string mode_;
  bool split_ = false, enable_split_ = false;
  int niter_ = 0, max_niter_ = 0, directed_ = 0, timing_ = 0;      // general
  bool transpose_ = false, mtxinfo_ = false, verbose_ = false;
  int mxvmode_ = 0;                           // mxv
  Desc_value lastmxv_ = GrB_PUSHONLY;         // direction the last mxv took
  float switchpoint_ = 0.f;
  bool dirinfo_ = false, struconly_ = false, opreuse_ = false;
  float memusage_ = 0.f;                      // push
  bool endbit_ = false, sort_ = false, atomic_ = false;
  bool earlyexit_ = false, fusedmask_ = false;                     // pull
  int nthread_ = 0, ndevice_ = 0;             // device
  bool debug_ = false, memory_ = false;

  // State of the push accumulator arena: which identity it is filled with.
  size_t   acc_elems_ = 0;
  unsigned acc_identity_bits_ = 0;
  size_t   acc_elem_bytes_ = 0;
  bool     acc_valid_ = false;
  size_t   bits_words_ = 0;
  bool     bits_valid_ = false;

 private:
  struct FromArgs {                           // knob <- vm[name]
    const po::variables_map& vm;
    template <typename Field>
    void operator()(const char* name, Field& field) const {
      field = vm[name].template as<Field>();
    }
  };
  struct ByName {                             // one knob <-> a double
    const std::string& name;
    double value;
    bool   reading;
    bool   found;
    void operator()(const char*, std::string&) {}
    template <typename Field>
    void operator()(const char* knob_name, Field& field) {
      if (name != knob_name) return;
      found = true;
      if (reading) value = static_cast<double>(field);
      else         field = static_cast<Field>(value);
    }
  };
};

}  // namespace backend
}  // namespace graphblas

#endif  // GRAPHBLAS_BACKEND_CUDA_DESCRIPTOR_HPP_
